"""CPU-side checks of the localiser: the oracle's exact distance transform against scipy, its term tables against the
formulas in numpy, its step against a short independent numpy restatement, the argument checks of
slamrs_gpu_create_localizer (all before the device query) and the -sys crate's declarations."""
import ctypes as C
import math
import os
import re

import numpy as np
import pytest
import scipy.ndimage as ndi

from oracle import loc_oracle as LO
from oracle import numpy_restatement as NP
from slamrs_b200 import GridMapSlamConfig, SensorModel, _lib
from slamrs_b200.simulator import reference_scene, scene_map

from common import SEED, gpu_present, make_scans

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _scipy_d2(obstacles):
    return np.rint(ndi.distance_transform_edt(~obstacles) ** 2).astype(np.int64).reshape(-1)


@pytest.mark.parametrize("n,density,seed", [(16, 0.1, 1), (64, 0.02, 2), (200, 0.005, 3), (257, 0.01, 4), (257, 0.0005, 5)])
def test_oracle_distance_transform_equals_scipy_on_random_maps(oracle, n, density, seed):
    rng = np.random.default_rng(seed)
    prob = np.where(rng.random(n * n) < density, rng.uniform(0.51, 1.0, n * n), rng.uniform(0.0, 0.5, n * n))
    obstacles = (prob > 0.5).reshape(n, n)
    assert obstacles.any()
    d2, k = LO.distance2(prob, n, n, 0.5)
    assert k == int(obstacles.sum())
    assert np.array_equal(d2, _scipy_d2(obstacles))


def test_oracle_distance_transform_corner_cells_and_full_maps(oracle):
    n = 200
    for r, c in [(0, 0), (0, n - 1), (n - 1, 0), (n - 1, n - 1)]:
        prob = np.full((n, n), 0.5)
        prob[r, c] = 0.9
        d2, k = LO.distance2(prob, n, n, 0.5)
        assert k == 1 and np.array_equal(d2, _scipy_d2(prob > 0.5))
    full = np.full(n * n, 1.0)
    d2, k = LO.distance2(full, n, n, 0.5)
    assert k == n * n and not d2.any()
    # the threshold is strict: p == occupied_above is not an obstacle
    prob = np.full(n * n, 0.7)
    prob[12345] = 0.70000001
    d2, _ = LO.distance2(prob, n, n, 0.7)
    assert np.array_equal(d2, _scipy_d2((prob > 0.7).reshape(n, n)))


def test_scene_map_distance_transform(oracle):
    cfg = GridMapSlamConfig(position=(-12.8, -12.8), width=25.6, height=25.6, resolution=0.05, n_particles=1)
    prob = scene_map(reference_scene(5.0), cfg)
    assert set(np.unique(prob)) == {0.5, 0.9}
    d2, _ = LO.distance2(prob, 512, 512, 0.5)
    assert np.array_equal(d2, _scipy_d2((prob > 0.5).reshape(512, 512)))


def _field_terms_numpy(d2, res, sigma, z_rand):
    zr = np.float64(np.float32(z_rand)); zh = 1.0 - zr
    rr = np.float64(np.float32(res)) * np.float64(np.float32(res))
    ss = np.float64(np.float32(sigma)) * np.float64(np.float32(sigma))
    # exp and log elementwise from the platform libm (numpy's vector exp/log may differ from it by an ulp)
    arg = ((-0.5 * d2.astype(np.float64)) * rr) / ss
    return np.array([math.log(zh * math.exp(a) + zr) for a in arg])


@pytest.mark.parametrize("sigma,z_rand,occ", [(0.1, 0.05, 0.5), (0.25, 0.2, 0.65), (0.03, 0.5, 0.9)])
def test_oracle_field_terms_match_the_formula(oracle, sigma, z_rand, occ):
    n, res = 96, 0.05
    rng = np.random.default_rng(11)
    prob = np.where(rng.random(n * n) < 0.01, 0.95, rng.uniform(0.0, 0.6, n * n))
    ol = LO.OracleLocalizer((-2.4, -2.4), res, n, n, 1, prob, 1, sigma, z_rand, occ)
    d2, _ = LO.distance2(prob, n, n, np.float64(np.float32(occ)))
    want = _field_terms_numpy(d2, res, sigma, z_rand)
    got = ol.terms()
    assert np.max(np.abs(got - want) / np.maximum(np.abs(want), 1e-300)) <= 1e-15   # (0 at obstacles: log(z_hit + z_rand))
    assert ol.outside == math.log(np.float64(np.float32(z_rand)))
    ol.close()


def test_oracle_terms_without_obstacles_and_beam_endpoint(oracle):
    n = 40
    prob = np.random.default_rng(3).uniform(0.0, 0.5, n * n)
    prob[:7] = 0.5
    ol = LO.OracleLocalizer((-1.0, -1.0), 0.05, n, n, 1, prob, 1, 0.1, 0.05, 0.5)
    assert np.all(ol.terms() == math.log(np.float64(np.float32(0.05))))
    ol.close()
    ob = LO.OracleLocalizer((-1.0, -1.0), 0.05, n, n, 1, prob, 0)
    want = np.where(prob == 0.5, 0.0, np.log(0.9 * prob + (1.0 - 0.9) * 1.0 / 1.0))
    assert np.array_equal(ob.terms(), want) and ob.outside == 0.0
    ob.close()


def _numpy_loc_step(poses, terms, outside, pos, res, g, ang, dist, valid, dl, dr, wheel, z, u01):
    """The localisation step restated from the prose of SURVEY.md Appendix A (A.3-A.5, A.8) with a shared map."""
    F = np.float32
    mean_c = float(F((F(dl) + F(dr)) / F(2.0)))
    mean_t = float(F((F(dr) - F(dl)) / F(wheel)))
    std_c = (0.01 + abs(mean_c) * 0.05) / 2.0
    std_t = 5.0 * (math.pi / 180.0) + 0.1 * abs(mean_t)
    n = len(poses)
    new, raw = [], []
    for p in range(n):
        x, y, th = (F(v) for v in poses[p])
        cd = F(mean_c + std_c * z[2 * p])
        nth = F(th + F(mean_t + std_t * z[2 * p + 1]))
        nx, ny = F(x + F(NP.cosf(nth) * cd)), F(y + F(NP.sinf(nth) * cd))
        lp = 0.0
        for a, d, v in zip(ang, dist, valid):
            if not v:
                continue
            aa = F(nth + F(a))
            ex, ey = F(nx + F(NP.cosf(aa) * F(d))), F(ny + F(NP.sinf(aa) * F(d)))
            gx, gy = F(F(ex - F(pos[0])) / F(res)), F(F(ey - F(pos[1])) / F(res))
            if gx < 0 or gy < 0 or NP.rust_as_usize(gx) >= g or NP.rust_as_usize(gy) >= g:
                lp += outside
            else:
                lp += terms[NP.rust_as_usize(gy) * g + NP.rust_as_usize(gx)]
        dx, dy = F(x - nx), F(y - ny)
        moved = float(F(np.sqrt(F(F(dx * dx) + F(dy * dy)))))
        lm = math.log(NP.normal_pdf(moved, mean_c, std_c)) + math.log(NP.normal_pdf(NP.angle_diff(float(th), float(nth)), mean_t, std_t))
        raw.append(math.exp(lp + lm))
        new.append((nx, ny, nth))
    total = 0.0
    for w in raw:
        total += w
    norm = [w / total for w in raw]
    best = max(range(n), key=lambda i: (norm[i], i))
    r, c, i, idx = u01 * 1.0 / n, norm[0], 0, []
    for m in range(1, n + 1):
        uu = r + (m - 1.0) * 1.0 / n
        while uu > c and i + 1 < n:
            i += 1
            c += norm[i]
        idx.append(i)
    poses_next = np.array([new[k] for k in idx], np.float32)
    return np.array(raw), np.array(norm), np.array(idx), best, poses_next


@pytest.mark.parametrize("kind", [0, 1])
def test_oracle_step_equals_numpy_restatement(oracle, kind):
    n, g, res, pos = 64, 64, 0.05, (-1.6, -1.6)
    cfg = GridMapSlamConfig(position=pos, width=g * res, height=g * res, resolution=res, n_particles=n)
    prob = scene_map(reference_scene(1.2), cfg)
    ol = LO.OracleLocalizer(pos, res, g, g, n, prob, kind, 0.1, 0.05, 0.5)
    poses = oracle.uniform_poses(SEED, 0, n, (-1.0, -1.0, 1.0, 1.0))
    ol.set_poses(poses)
    terms = ol.terms()
    for step, (obs, odo) in enumerate(make_scans(1.2, 90, 1.5, 3)):
        z = oracle.motion_normals(SEED, step, 0, n)
        u = oracle.resample_uniform(SEED, step)
        ang = obs.angle.astype(np.float32).astype(np.float64)
        dist = obs.distance.astype(np.float32).astype(np.float64)
        dl, dr, wb = np.float32(odo.distance_left), np.float32(odo.distance_right), np.float32(odo.wheel_distance)
        raw, norm, idx, best, nxt = _numpy_loc_step(poses, terms, ol.outside, pos, res, g, ang, dist, obs.valid, dl, dr, wb, z, u)
        assert ol.update(ang, dist, obs.valid.astype(np.uint8), dl, dr, wb, z, u) == 0
        w_o, raw_o = ol.weights()
        assert np.max(np.abs(raw_o - raw) / np.maximum(raw, 1e-300)) < 1e-12, step
        assert np.max(np.abs(w_o - norm) / np.maximum(norm, 1e-300)) < 1e-12, step
        assert np.array_equal(ol.indices().astype(np.int64), idx), step
        assert ol.max_particle == best
        poses = ol.poses()
        assert np.array_equal(poses.view(np.uint32), nxt.view(np.uint32)), step
    ol.close()


def _cfg(**kw):
    c = _lib.Config()
    c.struct_size = C.sizeof(_lib.Config); c.abi_version = _lib.ABI_VERSION
    c.pos_x = c.pos_y = -1.0; c.resolution = 0.05; c.grid_w = c.grid_h = 40; c.n_particles = 64; c.world_size = 1
    for k, v in kw.items():
        setattr(c, k, v)
    return c


def _model(**kw):
    m = SensorModel.likelihood_field().to_struct()
    for k, v in kw.items():
        setattr(m, k, v)
    return m


@pytest.mark.parametrize("what,cfg_kw,model_kw,cell,msg", [
    ("world_size", dict(world_size=2), {}, None, b"world_size"),
    ("flags", dict(flags=1), {}, None, b"flags"),
    ("slot_cells", dict(slot_cells=256), {}, None, b"slot_cells"),
    ("spare_slots", dict(spare_slots=4), {}, None, b"spare_slots"),
    ("non_square", dict(grid_h=20), {}, None, b"grid_w"),
    ("struct_size", dict(struct_size=12), {}, None, b"slamrs_gpu_config"),
    ("model_struct_size", {}, dict(struct_size=8), None, b"slamrs_gpu_sensor_model"),
    ("kind", {}, dict(kind=2), None, b"kind"),
    ("sigma", {}, dict(sigma=0.0), None, b"sigma"),
    ("sigma_nan", {}, dict(sigma=float("nan")), None, b"sigma"),
    ("z_rand_0", {}, dict(z_rand=0.0), None, b"z_rand"),
    ("z_rand_1", {}, dict(z_rand=1.0), None, b"z_rand"),
    ("occupied_low", {}, dict(occupied_above=0.49), None, b"occupied_above"),
    ("occupied_1", {}, dict(occupied_above=1.0), None, b"occupied_above"),
    ("cell_nan", {}, {}, float("nan"), b"map_probability"),
    ("cell_negative", {}, {}, -0.01, b"map_probability"),
    ("cell_above_one", {}, {}, 1.5, b"map_probability"),
])
def test_create_localizer_argument_checks(what, cfg_kw, model_kw, cell, msg):
    L = _lib.load()
    h = C.c_void_p()
    cfg, m = _cfg(**cfg_kw), _model(**model_kw)
    prob = np.full(40 * 40, 0.5)
    if cell is not None:
        prob[777] = cell
    assert L.slamrs_gpu_create_localizer(C.byref(cfg), C.byref(m), prob.ctypes.data, C.byref(h)) == _lib.E_INVALID_ARG
    assert msg in L.slamrs_gpu_last_error(None)
    assert not h.value


def test_create_localizer_null_arguments_and_beam_model_skips_field_checks():
    L = _lib.load()
    h = C.c_void_p()
    cfg, m = _cfg(), _model()
    prob = np.full(40 * 40, 0.5)
    assert L.slamrs_gpu_create_localizer(None, C.byref(m), prob.ctypes.data, C.byref(h)) == _lib.E_INVALID_ARG
    assert L.slamrs_gpu_create_localizer(C.byref(cfg), None, prob.ctypes.data, C.byref(h)) == _lib.E_INVALID_ARG
    assert b"sensor model" in L.slamrs_gpu_last_error(None)
    assert L.slamrs_gpu_create_localizer(C.byref(cfg), C.byref(m), None, C.byref(h)) == _lib.E_INVALID_ARG
    assert b"map_probability" in L.slamrs_gpu_last_error(None)
    assert L.slamrs_gpu_create_localizer(C.byref(cfg), C.byref(m), prob.ctypes.data, None) == _lib.E_INVALID_ARG
    assert L.slamrs_gpu_get_sensor_terms(None, prob.ctypes.data) == _lib.E_INVALID_ARG
    # the beam-endpoint model has no parameters: out-of-range field parameters are not an error there
    beam = _model(kind=_lib.SENSOR_BEAM_ENDPOINT, sigma=0.0, z_rand=2.0, occupied_above=0.0)
    rc = L.slamrs_gpu_create_localizer(C.byref(cfg), C.byref(beam), prob.ctypes.data, C.byref(h))
    if not gpu_present():
        assert rc == _lib.E_NO_DEVICE
    else:
        assert rc == _lib.OK
        L.slamrs_gpu_destroy(h)


@pytest.mark.skipif(gpu_present(), reason="GPU present")
def test_valid_arguments_without_a_gpu_give_no_device():
    L = _lib.load()
    h = C.c_void_p()
    cfg, m = _cfg(), _model()
    prob = np.full(40 * 40, 0.5)
    assert L.slamrs_gpu_create_localizer(C.byref(cfg), C.byref(m), prob.ctypes.data, C.byref(h)) == _lib.E_NO_DEVICE
    assert b"no CPU fallback" in L.slamrs_gpu_last_error(None)


def _c_fields(struct, text):
    body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (struct, struct), text, flags=re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    return [re.findall(r"(\w+)\s*(?:\[[^\]]*\])?$", d.strip())[0] for d in body.split(";") if d.strip()]


def test_sys_crate_declares_the_localizer():
    header = open(os.path.join(ROOT, "include", "slamrs_gpu.h")).read()
    rust = open(os.path.join(ROOT, "rust", "slam-gpu-sys", "src", "lib.rs")).read()
    fields = _c_fields("slamrs_gpu_sensor_model", header)
    assert fields == ["struct_size", "kind", "sigma", "z_rand", "occupied_above"]
    body = re.search(r"pub struct slamrs_gpu_sensor_model \{(.*?)\}", rust, flags=re.S).group(1)
    assert re.findall(r"pub (\w+):", body) == fields
    for name, value in [("SLAMRS_SENSOR_BEAM_ENDPOINT", 0), ("SLAMRS_SENSOR_LIKELIHOOD_FIELD", 1)]:
        assert re.search(rf"{name}\s*=\s*{value}\b", header) and re.search(rf"pub const {name}: u32 = {value};", rust)
    for name in ("slamrs_gpu_create_localizer", "slamrs_gpu_get_sensor_terms"):
        c = re.search(r"int %s\((.*?)\);" % name, header, flags=re.S).group(1)
        r = re.search(r"pub fn %s\((.*?)\)" % name, rust, flags=re.S).group(1)
        assert len([a for a in r.split(",") if a.strip()]) == len(c.split(",")), name
    assert C.sizeof(_lib.SensorModel) == 20
