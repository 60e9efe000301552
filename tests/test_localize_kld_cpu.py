"""CPU-side checks of the localiser's KLD-sampling (adaptive population, slamrs_gpu_set_kld): the KLD oracle's bound
against its closed form and the chi-square quantile it approximates, its bin function against a numpy restatement at
the edges, its M-draw fold against a numpy restatement of the reference's loop, its step against the fixed-size
localiser and recovery oracles, the Kld dataclass, the argument checks on a NULL handle and the -sys declarations."""
import ctypes as C
import math
import os
import re

import numpy as np
import pytest
from scipy.stats import chi2, norm

from oracle import kld_oracle as KO
from oracle import loc_oracle as LO
from oracle import recovery_oracle as RO
from slamrs_b200 import GridMapSlamConfig, Kld, _lib
from slamrs_b200.simulator import reference_scene, scene_map

from common import SEED, make_scans

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TWO_PI = float.fromhex("0x1.921fb54442d18p+2")


def _bound_py(k, n_min, n_max, err, z):
    if k <= 1:
        return n_min
    b = 2.0 / (9.0 * (k - 1))
    x = 1.0 - b + math.sqrt(b) * z
    n = ((k - 1) / (2.0 * err)) * x * x * x
    if not n < n_max:
        return n_max
    return max(n_min, math.ceil(n))


def test_bound_equals_the_closed_form():
    for err, z in ((0.01, 2.326), (0.05, 1.645), (0.2, 0.0), (1.0, 3.0), (1e-4, 2.326)):
        for k in list(range(0, 300)) + [1000, 4097, 65536, 1 << 20, (1 << 28) + 1]:
            for n_min, n_max in ((1, (1 << 31) - 1), (256, 5000), (7, 7)):
                assert KO.kld_bound(k, n_min, n_max, err, z) == _bound_py(k, n_min, n_max, err, z), (err, z, k, n_min, n_max)
    assert KO.kld_bound(0, 300, 500, 0.01, 2.326) == KO.kld_bound(1, 300, 500, 0.01, 2.326) == 300   # not n_max
    assert KO.kld_bound(10, 1, 1 << 30, 0.01, 2.326) == 1085


def test_bound_approximates_the_chi_square_quantile():
    """Wilson-Hilferty: with z = the (1 - delta) normal quantile, the bound is chi2.ppf(1 - delta, k - 1) / (2 err)
    within 1 % for every k >= 2 at delta = 0.01."""
    delta, err = 0.01, 0.01
    z = float(norm.ppf(1.0 - delta))
    for k in list(range(2, 200)) + [500, 1000, 5000, 20000]:
        want = chi2.ppf(1.0 - delta, k - 1) / (2.0 * err)
        got = KO.kld_bound(k, 1, 1 << 40, err, z)
        assert abs(got - want) <= 0.01 * want + 1.0, (k, got, want)


def _as_usize(v):
    v = np.float32(v)
    if not v == v or v <= 0.0:
        return 0
    if v >= np.float32(2.0 ** 64):
        return 2 ** 64 - 1
    return int(v)


def _bin_numpy(x, y, theta, pos, res, gw, gh, bc, tb):
    nbx, nby = -(-gw // bc), -(-gh // bc)
    with np.errstate(invalid="ignore", over="ignore"):
        gx = (np.float32(x) - np.float32(pos[0])) / np.float32(res)
        gy = (np.float32(y) - np.float32(pos[1])) / np.float32(res)
    if gx < 0.0 or gy < 0.0 or _as_usize(gx) >= gw or _as_usize(gy) >= gh:
        return nbx * nby * tb
    th = float(np.float32(theta))
    t = math.fmod(th, TWO_PI) if math.isfinite(th) else float("nan")
    if t < 0.0:
        t += TWO_PI
    h = min(tb - 1, int((t * tb) / TWO_PI)) if 0.0 <= t < TWO_PI else 0
    return ((_as_usize(gy) // bc) * nbx + _as_usize(gx) // bc) * tb + h


@pytest.mark.parametrize("gw,bc,tb", [(200, 25, 36), (200, 1, 1), (64, 7, 3600), (101, 10, 5)])
def test_bin_equals_numpy_restatement_at_the_edges(gw, bc, tb):
    pos, res = (-2.0, -1.5), 0.02
    f32 = np.float32
    xs = [pos[0] + c * res for c in (0, bc - 1, bc, 2 * bc, gw - 1, gw)]
    xs += [float(np.nextafter(f32(v), f32(-np.inf))) for v in xs] + [float(np.nextafter(f32(v), f32(np.inf))) for v in xs]
    xs += [pos[0] - 1e-3, -1e30, 1e30, float("nan"), float("inf"), float("-inf")]
    thetas = [0.0, -0.0, math.pi, -math.pi, TWO_PI, -TWO_PI, float(np.nextafter(f32(TWO_PI), f32(0))), 1e-30, -1e-30,
              float(np.float32(-1e-8)), 100.0, -100.0, 3.0e38, float("inf"), float("-inf"), float("nan")]
    thetas += [(j + 0.5) * TWO_PI / tb for j in (0, tb // 2, tb - 1)] + [j * TWO_PI / tb for j in (1, tb - 1)]
    rng = np.random.default_rng(7)
    ys = xs[::3] + [pos[1] + 0.5 * res]
    seen = set()
    for x in xs:
        for y in ys:
            for t in thetas[:: max(1, len(thetas) // 6)] if y != ys[-1] else thetas:
                want = _bin_numpy(x, y + (pos[1] - pos[0]), t, pos, res, gw, gw, bc, tb)
                got = KO.kld_bin(x, y + (pos[1] - pos[0]), t, pos, res, gw, gw, bc, tb)
                assert got == want, (x, y, t, got, want)
                seen.add(got)
    off = (-(-gw // bc)) ** 2 * tb
    assert off in seen and len(seen) > 10
    for _ in range(2000):   # random poses, a fifth of them off the grid
        x, y = rng.uniform(pos[0] - 0.5, pos[0] + gw * res * 1.2, 2)
        t = rng.uniform(-20.0, 20.0)
        assert KO.kld_bin(x, y, t, pos, res, gw, gw, bc, tb) == _bin_numpy(x, y, t, pos, res, gw, gw, bc, tb)


def test_count_is_the_number_of_distinct_bins():
    pos, res, gw = (-2.0, -2.0), 0.02, 200
    rng = np.random.default_rng(3)
    xyt = np.column_stack([rng.uniform(-2.5, 2.5, 5000), rng.uniform(-2.5, 2.5, 5000),
                           rng.uniform(-7.0, 7.0, 5000)]).astype(np.float32)
    for bc, tb in ((25, 36), (1, 1), (5, 360)):
        bins = {_bin_numpy(*p, pos, res, gw, gw, bc, tb) for p in xyt.tolist()}
        assert KO.kld_count(xyt, pos, res, gw, gw, bc, tb) == len(bins)
    assert KO.kld_count(np.tile(xyt[:1], (100, 1)), pos, res, gw, gw, 25, 36) == 1


def _fold_numpy(raw, m, u01):
    """particle.rs:78-101 with m wherever N counts draws, on the sequential normalisation."""
    n = len(raw)
    s = 0.0
    for w in raw.tolist():
        s += w
    normw = [w / s for w in raw.tolist()]
    r = u01 * 1.0 / float(m)
    c, i, idx, clamped = normw[0], 0, [], False
    for mm in range(1, m + 1):
        u = r + (float(mm) - 1.0) * 1.0 / float(m)
        while u > c:
            if i + 1 >= n:
                clamped = True
                break
            i += 1
            c += normw[i]
        idx.append(i)
    return np.array(normw), np.array(idx, np.uint64), clamped


@pytest.mark.parametrize("n", [1, 2, 3, 17, 256, 4099])
def test_m_draw_fold_equals_numpy_restatement(n):
    rng = np.random.default_rng(n)
    raw = rng.exponential(1.0, n) ** 4
    if n > 3:
        raw[rng.integers(0, n, n // 3)] = 0.0
    for m in sorted({1, 2, max(1, n // 3), n, n + 1, 3 * n + 5, 1000}):
        for u01 in (0.0, 0.37, 1.0 - 2 ** -53):
            norm_o, idx_o, mp, cl = KO.resample_fold_m(raw, m, u01)
            norm_p, idx_p, cl_p = _fold_numpy(raw, m, u01)
            assert np.array_equal(norm_o.view(np.uint64), norm_p.view(np.uint64))
            assert np.array_equal(idx_o, idx_p), (m, u01)
            assert bool(cl) == cl_p and idx_o.size == m and np.all(np.diff(idx_o.astype(np.int64)) >= 0)
            assert mp == max(range(n), key=lambda p: (norm_p[p], p))
            if m == n:
                f = KO.resample_fold(raw, u01)
                assert np.array_equal(f[1], idx_o) and f[2] == mp and f[3] == cl


def _room(cfg, g):
    prob = scene_map(reference_scene(1.0), cfg)
    prob[(prob == 0.5) & (np.arange(g * g) % 4 != 0)] = 0.2
    return prob


@pytest.mark.parametrize("recovery", [False, True])
def test_oracle_at_a_fixed_population_equals_the_fixed_size_oracles(oracle, recovery):
    """KLD-sampling with n_min = n_max = C, and KLD-sampling off, step for step bitwise equal to loc_oracle.c (or
    recovery_oracle.c) on a cloud scattered at step 2."""
    n, g, res, pos = 384, 200, 0.02, (-2.0, -2.0)
    cfg = GridMapSlamConfig(position=pos, width=4.0, height=4.0, resolution=res, n_particles=n)
    prob = _room(cfg, g)
    ref = (RO.OracleRecoveryLocalizer if recovery else LO.OracleLocalizer)(pos, res, g, g, n, prob, 1, 0.1, 0.05, 0.5)
    fixed = KO.OracleKldLocalizer(pos, res, g, g, n, prob, 1, 0.1, 0.05, 0.5)
    off = KO.OracleKldLocalizer(pos, res, g, g, n, prob, 1, 0.1, 0.05, 0.5)
    fixed.set_kld((n, n, 0.01, 2.326, 25, 36))
    if recovery:
        for o in (ref, fixed, off):
            o.set_recovery(0.05, 0.5, SEED)
    for step, (obs, odo) in enumerate(make_scans(1.0, 90, 1.0, 6)):
        if step == 2:
            scatter = oracle.uniform_poses(SEED + 1, 0, n, (-1.8, -1.8, 1.8, 1.8))
            for o in (ref, fixed, off):
                o.set_poses(scatter)
        z = oracle.motion_normals(SEED, step, 0, n)
        u = oracle.resample_uniform(SEED, step)
        ang = obs.angle.astype(np.float32).astype(np.float64)
        dist = obs.distance.astype(np.float32).astype(np.float64)
        args = (ang, dist, obs.valid.astype(np.uint8), np.float32(odo.distance_left), np.float32(odo.distance_right),
                np.float32(odo.wheel_distance), z, u)
        for o in (ref, fixed, off):
            assert o.update(*args) == 0
        for o in (fixed, off):
            assert np.array_equal(o.poses().view(np.uint32), ref.poses().view(np.uint32)), step
            assert np.array_equal(o.indices(), ref.indices()) and o.max_particle == ref.max_particle
            for a, b in zip(o.weights(), ref.weights()):
                assert np.array_equal(a.view(np.uint64), b.view(np.uint64))
            assert np.array_equal(o.estimated_pose().view(np.uint32), ref.estimated_pose().view(np.uint32))
            if recovery:
                assert o.recovery_state() == ref.recovery_state()
        assert off.kld_state() == (0, 0, 0)
        assert fixed.kld_state()[0] == fixed.kld_state()[2] == n and fixed.kld_state()[1] >= 1


def test_oracle_population_follows_the_bins(oracle):
    """A cloud scattered over the room grows the population; the same cloud collapsed onto one pose shrinks it to
    n_min; the estimate is the new particle at max_particle * M / N_t; indices stay below N_t."""
    cap, g, res, pos = 4096, 200, 0.02, (-2.0, -2.0)
    cfg = GridMapSlamConfig(position=pos, width=4.0, height=4.0, resolution=res, n_particles=cap)
    prob = _room(cfg, g)
    o = KO.OracleKldLocalizer(pos, res, g, g, cap, prob, 1, 0.1, 0.05, 0.5)
    kld = (100, cap, 0.05, 2.326, 10, 12)
    o.set_kld(kld)
    o.set_poses(np.tile(np.float32([0.1, 0.2, 0.3]), (cap, 1)))
    scans = make_scans(1.0, 90, 1.0, 5)
    pops = []
    for step, (obs, odo) in enumerate(scans):
        if step == 2:
            o.set_poses(oracle.uniform_poses(SEED + 2, 0, o.population, (-1.8, -1.8, 1.8, 1.8)))
        n_t = o.population
        start = o.poses()
        k = KO.kld_count(start, pos, res, g, g, kld[4], kld[5])
        z = oracle.motion_normals(SEED, step, 0, n_t)
        u = oracle.resample_uniform(SEED, step)
        assert o.update(obs.angle.astype(np.float32).astype(np.float64), obs.distance.astype(np.float32).astype(np.float64),
                        obs.valid.astype(np.uint8), np.float32(odo.distance_left), np.float32(odo.distance_right),
                        np.float32(odo.wheel_distance), z, u) == 0
        m = KO.kld_bound(k, kld[0], kld[1], kld[2], kld[3])
        assert o.kld_state() == (n_t, k, m) and o.population == m
        idx = o.indices()
        assert idx.size == m and int(idx.max()) < n_t and o.weights()[0].size == n_t
        assert np.array_equal(o.estimated_pose().view(np.uint32), o.poses()[o.max_particle * m // n_t].view(np.uint32))
        pops.append(m)
    assert pops[0] == 100 and pops[2] > 1000, pops
    o.set_kld(None)
    n_t = o.population
    obs, odo = scans[0]
    o.update(obs.angle, obs.distance, obs.valid.astype(np.uint8), np.float32(odo.distance_left),
             np.float32(odo.distance_right), np.float32(odo.wheel_distance), oracle.motion_normals(SEED, 9, 0, n_t), 0.5)
    assert o.population == cap and o.kld_state() == (0, 0, 0) and o.weights()[0].size == n_t
    o.close()


def test_kld_dataclass_and_struct():
    assert C.sizeof(_lib.Kld) == 40
    k = Kld()
    assert (k.n_min, k.n_max, k.err, k.z, k.bin_xy, k.theta_bins) == (256, None, 0.01, 2.326, 0.5, 36)
    s = k.to_struct(4096, 0.02)
    assert (s.struct_size, s.n_min, s.n_max, s.err, s.z, s.bin_cells, s.theta_bins) == (40, 256, 4096, 0.01, 2.326, 25, 36)
    assert Kld(bin_xy=0.001).bin_cells(0.05) == 1 and Kld(bin_xy=0.5).bin_cells(0.05) == 10
    assert Kld(n_max=1000).to_struct(4096, 0.05).n_max == 1000


def test_kld_entry_points_reject_a_null_handle():
    L = _lib.load()
    s = Kld().to_struct(4096, 0.02)
    assert L.slamrs_gpu_set_kld(None, C.byref(s)) == _lib.E_INVALID_ARG
    assert L.slamrs_gpu_set_kld(None, None) == _lib.E_INVALID_ARG
    out = np.zeros(3, np.uint64)
    assert L.slamrs_gpu_get_kld_state(None, out.ctypes.data) == _lib.E_INVALID_ARG
    n = C.c_uint64(7)
    assert L.slamrs_gpu_get_population(None, C.byref(n)) == _lib.E_INVALID_ARG and n.value == 7


def _c_fields(struct, text):
    body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (struct, struct), text, flags=re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    return [re.findall(r"(\w+)\s*(?:\[[^\]]*\])?$", d.strip())[0] for d in body.split(";") if d.strip()]


def test_sys_crate_declares_kld():
    header = open(os.path.join(ROOT, "include", "slamrs_gpu.h")).read()
    rust = open(os.path.join(ROOT, "rust", "slam-gpu-sys", "src", "lib.rs")).read()
    fields = _c_fields("slamrs_gpu_kld", header)
    assert fields == ["struct_size", "n_min", "n_max", "pad", "err", "z", "bin_cells", "theta_bins"]
    assert [n for n, _ in _lib.Kld._fields_] == fields
    body = re.search(r"pub struct slamrs_gpu_kld \{(.*?)\}", rust, flags=re.S).group(1)
    assert re.findall(r"pub (\w+):", body) == fields
    for name in ("slamrs_gpu_set_kld", "slamrs_gpu_get_kld_state", "slamrs_gpu_get_population"):
        c = re.search(r"int %s\((.*?)\);" % name, header, flags=re.S).group(1)
        r = re.search(r"pub fn %s\((.*?)\)" % name, rust, flags=re.S).group(1)
        assert len([a for a in r.split(",") if a.strip()]) == len(c.split(",")), name
        assert name in _lib.EXPORTS
