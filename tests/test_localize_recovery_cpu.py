"""CPU-side checks of the localiser's recovery (augmented MCL, slamrs_gpu_set_recovery): the recovery oracle's
free-cell list, its recovery draw against a numpy restatement from philox / u53, its state update on hand-made sums,
one oracle step with injections, and the -sys crate's declarations."""
import ctypes as C
import math
import os
import re

import numpy as np
import pytest

from oracle import recovery_oracle as RO
from slamrs_b200 import GridMapSlamConfig, Recovery, _lib
from slamrs_b200.simulator import reference_scene, scene_map

from common import SEED, make_scans

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _u53(hi, lo):
    return float(((int(hi) << 32) | int(lo)) >> 11) * 2.0 ** -53


def _draw_numpy(O, seed, step, m, p, free, grid_h, pos, res):
    """The recovery draw restated from the stream's Philox words (None: not replaced)."""
    key = [seed & 0xFFFFFFFF, seed >> 32]
    ctr = lambda d: [m & 0xFFFFFFFF, step & 0xFFFFFFFF, step >> 32, d]   # noqa: E731
    a = O.philox(ctr(4), key)
    if not _u53(a[0], a[1]) < p:
        return None
    n_free = len(free)
    cell = int(free[min(n_free - 1, int(_u53(a[2], a[3]) * float(n_free)))])
    b, c = O.philox(ctr(5), key), O.philox(ctr(6), key)
    col, row = float(cell % grid_h), float(cell // grid_h)
    px, py, r = float(np.float32(pos[0])), float(np.float32(pos[1])), float(np.float32(res))
    return np.array([px + (col + _u53(b[0], b[1])) * r, py + (row + _u53(b[2], b[3])) * r,
                     -math.pi + _u53(c[0], c[1]) * (2.0 * math.pi)], np.float32)


def _free_map(n, seed):
    rng = np.random.default_rng(seed)
    return np.choose(rng.integers(0, 3, n * n), [np.full(n * n, 0.5), rng.uniform(0.0, 0.5, n * n),
                                                  rng.uniform(0.5, 1.0, n * n)])


@pytest.mark.parametrize("n,seed", [(16, 1), (64, 2), (129, 3)])
def test_oracle_free_cells_are_the_cells_below_one_half(n, seed):
    prob = _free_map(n, seed)
    prob[:5] = [0.5, np.nextafter(0.5, 0.0), 0.0, 1.0, np.nextafter(0.5, 1.0)]
    ol = RO.OracleRecoveryLocalizer((-1.0, -1.0), 0.05, n, n, 1, prob, 1)
    assert np.array_equal(ol.free_cells().astype(np.int64), np.flatnonzero(prob < 0.5))
    ol.close()
    cfg = GridMapSlamConfig(position=(-2.0, -2.0), width=4.0, height=4.0, resolution=0.02, n_particles=1)
    ol = RO.OracleRecoveryLocalizer(cfg.position, cfg.resolution, 200, 200, 1, scene_map(reference_scene(1.0), cfg), 1)
    assert ol.free_cells().size == 0   # walls and unknown space only
    ol.close()


@pytest.mark.parametrize("step", [0, 1, 7, (1 << 32) + 5])
def test_recovery_draw_equals_numpy_restatement(oracle, step):
    prob = _free_map(48, 4)
    free = np.flatnonzero(prob < 0.5).astype(np.uint32)
    pos, res = (-1.3, 0.7), 0.05
    for p in (0.0, 0.3, 1.0):
        inject, poses = RO.recovery_draws(SEED, step, 100, 300, p, free, 48, pos, res)
        for k in range(300):
            want = _draw_numpy(oracle, SEED, step, 100 + k, p, free, 48, pos, res)
            assert inject[k] == (want is not None), (p, k)
            if want is not None:
                assert np.array_equal(poses[k].view(np.uint32), want.view(np.uint32)), (p, k)
        assert (not inject.any()) if p == 0.0 else inject.any()
        if p == 1.0:
            assert inject.all()


def test_recovery_slot_clamps_to_the_last_entry():
    top = (2 ** 53 - 1) * 2.0 ** -53   # the largest u53 value
    for n in (1, 2, 3, 7, 1000, 12345, 2 ** 20, 2 ** 31 - 1, 2 ** 31, 2 ** 32 - 1):
        assert RO.recovery_slot(top, n) == n - 1, n
        assert RO.recovery_slot(0.0, n) == 0
        assert RO.recovery_slot(1.0, n) == n - 1, n   # the product reaches n_free: clamped
        assert RO.recovery_slot(0.5, n) == min(n - 1, int(0.5 * n))


def _update_py(raw_sum, n, a_slow, a_fast, ws, wf):
    if not math.isfinite(raw_sum):
        return ws, wf, 0.0
    avg = raw_sum / n
    ws = avg if ws == 0.0 else ws + a_slow * (avg - ws)
    wf = avg if wf == 0.0 else wf + a_fast * (avg - wf)
    if not ws > 0.0:
        return ws, wf, 0.0
    p = 1.0 - wf / ws
    return ws, wf, p if p > 0.0 else 0.0


@pytest.mark.parametrize("raw_sum,n,ws,wf", [
    (3.0, 3, 0.0, 0.0),            # first step: both averages seeded with w_avg, p = 0
    (1e-3, 1000, 0.0, 2e-6),       # w_slow == 0 seeds only w_slow
    (1e-3, 1000, 2e-6, 0.0),
    (0.0, 64, 1e-5, 2e-5),         # a zero sum: both decay, w_fast faster -> p > 0
    (0.0, 64, 0.0, 0.0),           # all zero: w_slow stays 0 -> p = 0
    (7.0, 4096, 1e-3, 5e-4),
    (7.0, 4096, 5e-4, 1e-3),       # w_fast above w_slow -> p = 0
    (float("inf"), 16, 1e-3, 5e-4),
    (float("nan"), 16, 1e-3, 5e-4),
    (5e-324, 3, 1e-300, 1e-310),
])
def test_recovery_state_update_on_hand_made_sums(raw_sum, n, ws, wf):
    for a_slow, a_fast in ((0.001, 0.1), (0.05, 0.5), (0.2, 1.0)):
        got = RO.recovery_update(raw_sum, n, a_slow, a_fast, ws, wf)
        want = _update_py(raw_sum, n, a_slow, a_fast, ws, wf)
        assert np.array_equal(np.array(got).view(np.uint64), np.array(want).view(np.uint64)), (got, want)
    if not math.isfinite(raw_sum):
        assert RO.recovery_update(raw_sum, n, 0.05, 0.5, ws, wf) == (ws, wf, 0.0)
    if ws == wf == 0.0:
        assert RO.recovery_update(raw_sum, n, 0.05, 0.5, ws, wf)[2] == 0.0


def test_oracle_step_injects_into_free_cells_after_recording_the_estimate(oracle):
    """A scattered cloud on a room map with free space: the oracle's injected poses are the stream's draws, lie in
    free cells, and the estimate is the resampled pose of max_particle."""
    n, g, res, pos = 512, 64, 0.05, (-1.6, -1.6)
    cfg = GridMapSlamConfig(position=pos, width=g * res, height=g * res, resolution=res, n_particles=n)
    prob = scene_map(reference_scene(1.2), cfg)
    prob[(prob == 0.5) & (np.arange(g * g) % 3 != 0)] = 0.2
    ol = RO.OracleRecoveryLocalizer(pos, res, g, g, n, prob, 1, 0.1, 0.05, 0.5)
    free = ol.free_cells()
    ol.set_recovery(0.05, 0.5, SEED)
    scans = make_scans(1.2, 90, 1.5, 4)
    ol.set_poses(np.zeros((n, 3), np.float32))
    injected = []
    for step, (obs, odo) in enumerate(scans):
        if step == 2:
            ol.set_poses(oracle.uniform_poses(SEED, 0, n, (-1.5, -1.5, 1.5, 1.5)))
        z = oracle.motion_normals(SEED, step, 0, n)
        u = oracle.resample_uniform(SEED, step)
        ang = obs.angle.astype(np.float32).astype(np.float64)
        dist = obs.distance.astype(np.float32).astype(np.float64)
        before = ol.recovery_state()
        assert ol.update(ang, dist, obs.valid.astype(np.uint8), np.float32(odo.distance_left),
                         np.float32(odo.distance_right), np.float32(odo.wheel_distance), z, u) == 0
        st = ol.recovery_state()
        _, raw = ol.weights()
        s = 0.0
        for w in raw:
            s += w
        ws, wf, p = _update_py(s, n, 0.05, 0.5, before["w_slow"], before["w_fast"])
        assert (st["w_slow"], st["w_fast"], st["p_inject"]) == (ws, wf, p), step
        inject, draws = RO.recovery_draws(SEED, step, 0, n, p, free, g, pos, res)
        assert st["injected"] == int(inject.sum())
        poses = ol.poses()
        assert np.array_equal(poses[inject].view(np.uint32), draws[inject].view(np.uint32))
        cells = (np.floor((poses[inject, 1] - np.float32(pos[1])) / np.float32(res)).astype(np.int64) * g +
                 np.floor((poses[inject, 0] - np.float32(pos[0])) / np.float32(res)).astype(np.int64))
        assert np.all(prob[cells] < 0.5)
        mp = ol.max_particle
        est = ol.estimated_pose()
        assert np.array_equal(est.view(np.uint32), poses[mp].view(np.uint32)) != bool(inject[mp])
        injected.append(st["injected"])
    assert injected[0] == 0 and max(injected) > 0, injected
    ol.set_recovery(0.0, 0.0, SEED)
    assert ol.recovery_state() == {"w_slow": 0.0, "w_fast": 0.0, "p_inject": 0.0, "injected": 0}
    ol.close()


def test_recovery_struct_and_null_handle():
    assert C.sizeof(_lib.Recovery) == 24
    r = Recovery().to_struct()
    assert (r.struct_size, r.alpha_slow, r.alpha_fast) == (24, 0.001, 0.1)
    L = _lib.load()
    assert L.slamrs_gpu_set_recovery(None, C.byref(r)) == _lib.E_INVALID_ARG
    out = np.zeros(3)
    assert L.slamrs_gpu_get_recovery_state(None, out.ctypes.data, None) == _lib.E_INVALID_ARG


def _c_fields(struct, text):
    body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (struct, struct), text, flags=re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    return [re.findall(r"(\w+)\s*(?:\[[^\]]*\])?$", d.strip())[0] for d in body.split(";") if d.strip()]


def test_sys_crate_declares_recovery():
    header = open(os.path.join(ROOT, "include", "slamrs_gpu.h")).read()
    rust = open(os.path.join(ROOT, "rust", "slam-gpu-sys", "src", "lib.rs")).read()
    fields = _c_fields("slamrs_gpu_recovery", header)
    assert fields == ["struct_size", "pad", "alpha_slow", "alpha_fast"]
    body = re.search(r"pub struct slamrs_gpu_recovery \{(.*?)\}", rust, flags=re.S).group(1)
    assert re.findall(r"pub (\w+):", body) == fields
    for name in ("slamrs_gpu_set_recovery", "slamrs_gpu_get_recovery_state"):
        c = re.search(r"int %s\((.*?)\);" % name, header, flags=re.S).group(1)
        r = re.search(r"pub fn %s\((.*?)\)" % name, rust, flags=re.S).group(1)
        assert len([a for a in r.split(",") if a.strip()]) == len(c.split(",")), name
