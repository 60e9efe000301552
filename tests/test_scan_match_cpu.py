"""Scan-matching pose refinement on the CPU: an independent numpy restatement of the score S and of the hill climb
against the C oracle, on hand-built grids and on grids from oracle steps; convergence on a hand-drawn room; the
argument checks that need no device."""
from __future__ import annotations

import ctypes as C

import numpy as np
import pytest

from oracle import oracle as O
from oracle.scan_match_oracle import ScanMatchOracle
from slamrs_b200 import GridMapSlamConfig, ScanMatcher, _lib
from slamrs_b200.simulator import rect_segments, reference_scene, scan, scene_map

from common import make_scans, oracle_step

f32 = np.float32
L_FREE, L_OCC = -0.8472978603872036, 2.1972245773362196   # the device's binary64 constants (slam_device.cuh)


# ---------------------------------------------------------------------------------------------- numpy restatement
def f32_as_usize(v):
    v = np.asarray(v, np.float32)
    out = np.zeros(v.shape, np.float64)
    ok = np.isfinite(v) & (v > 0)
    out[ok] = np.floor(v[ok].astype(np.float64))
    out[np.isposinf(v)] = 2.0 ** 64
    return out


class Restated:
    """S(pose) and the climb, written from the definition in DESIGN.md."""

    def __init__(self, cfg: GridMapSlamConfig, n_free, n_occ, radius, step_xy, step_theta, levels, max_moves):
        self.px, self.py, self.res = f32(cfg.position[0]), f32(cfg.position[1]), f32(cfg.resolution)
        self.gw, self.gh = n_free.shape[1], n_free.shape[0]
        nf = n_free.astype(np.float64); no = n_occ.astype(np.float64)
        self.occ = (nf * L_FREE + no * L_OCC) > 0.0          # [row, column]
        self.r = radius
        self.step_xy, self.step_theta, self.levels, self.max_moves = f32(step_xy), f32(step_theta), levels, max_moves

    def beam_scores(self, pose, angle, dist):
        x, y, t = (f32(v) for v in pose)
        a = (t + angle.astype(np.float32)).astype(np.float32)
        s, c = O.libm_sincosf(a)
        d = dist.astype(np.float32)
        ex = (x + (c * d).astype(np.float32)).astype(np.float32)
        ey = (y + (s * d).astype(np.float32)).astype(np.float32)
        with np.errstate(invalid="ignore"):
            gx = ((ex - self.px).astype(np.float32) / self.res).astype(np.float32)
            gy = ((ey - self.py).astype(np.float32) / self.res).astype(np.float32)
            ok = ~((gx < 0) | (gy < 0) | (f32_as_usize(gx) >= self.gw) | (f32_as_usize(gy) >= self.gh))
        cx = np.where(ok, f32_as_usize(gx), 0).astype(np.int64)
        cy = np.where(ok, f32_as_usize(gy), 0).astype(np.int64)
        best = np.zeros(angle.size, np.int64)
        r = self.r
        for dy in range(-r, r + 1):
            for dx in range(-r, r + 1):
                xx, yy = cx + dx, cy + dy
                inside = ok & (xx >= 0) & (yy >= 0) & (xx < self.gw) & (yy < self.gh)
                hit = np.zeros(angle.size, bool)
                hit[inside] = self.occ[yy[inside], xx[inside]]
                best = np.where(hit, np.maximum(best, (r + 1) ** 2 - (dx * dx + dy * dy)), best)
        return best

    def score(self, pose, angle, dist, valid):
        v = valid.astype(bool)
        return int(self.beam_scores(pose, angle[v], dist[v]).sum())

    def climb(self, pose, angle, dist, valid):
        """(pose, moves, scored, log) with one log entry per round: (level, six scores, chosen index or None)."""
        p = [f32(v) for v in pose]
        best = self.score(p, angle, dist, valid)
        moves, scored, log = 0, 1, []
        for level in range(self.levels):
            dxy = f32(self.step_xy * f32(2.0 ** -level)); dth = f32(self.step_theta * f32(2.0 ** -level))
            while moves < self.max_moves:
                x, y, t = p
                cands = [[f32(x + dxy), y, t], [f32(x - dxy), y, t], [x, f32(y + dxy), t], [x, f32(y - dxy), t],
                         [x, y, f32(t + dth)], [x, y, f32(t - dth)]]
                sc = [self.score(c, angle, dist, valid) for c in cands]
                scored += 6
                k = int(np.argmax(sc))                     # the first of the largest
                if sc[k] <= best:
                    log.append((level, sc, None))
                    break
                log.append((level, sc, k))
                best, p, moves = sc[k], cands[k], moves + 1
        return np.array(p, np.float32), moves, scored, log


def oracle_slam(cfg: GridMapSlamConfig, track_counts=True):
    return ScanMatchOracle(cfg.position, cfg.width, cfg.height, cfg.resolution, cfg.n_particles, track_counts)


def small_cfg(n=2, res=0.02, side=4.0):
    return GridMapSlamConfig(position=(-side / 2, -side / 2), width=side, height=side, resolution=res, n_particles=n)


def _oracle_with(cfg, n_free, n_occ, **m):
    osl = oracle_slam(cfg)
    for p in range(osl.n):
        osl.set_counts(p, n_free.reshape(-1), n_occ.reshape(-1))
    osl.set_scan_match(**m)
    return osl


def _bits(a):
    return np.asarray(a, np.float32).view(np.uint32)


def _room_counts(cfg, segments):
    prob = scene_map(segments, cfg)
    gw = int(round(np.sqrt(prob.size)))
    n_occ = np.where(prob > 0.5, 3, 0).astype(np.uint16).reshape(gw, gw)
    n_free = np.where(prob > 0.5, 0, 1).astype(np.uint16).reshape(gw, gw)
    return n_free, n_occ


# ---------------------------------------------------------------------------------------------- S against the oracle
@pytest.mark.parametrize("radius", [0, 1, 2])
def test_score_matches_oracle_on_hand_built_grid(radius):
    cfg = small_cfg()
    rng = np.random.default_rng(radius)
    gw = O.grid_cells(cfg.width, cfg.resolution)
    n_free = rng.integers(0, 6, (gw, gw)).astype(np.uint16)
    n_occ = np.where(rng.random((gw, gw)) < 0.15, rng.integers(0, 4, (gw, gw)), 0).astype(np.uint16)
    # counter pairs on both sides of the sign change of the log-odds (2.197 no vs 0.847 nf: 5 free > 2 occupied)
    n_free[:4, :4] = 5; n_occ[:4, :4] = 2
    n_free[:4, 4:8] = 2; n_occ[:4, 4:8] = 1
    n_free[0, 0], n_occ[0, 0] = 65535, 65535
    osl = _oracle_with(cfg, n_free, n_occ, radius=radius)
    ref = Restated(cfg, n_free, n_occ, radius, 0.1, 0.05, 4, 32)
    obs = scan(reference_scene(1.0), (0.1, -0.2, 0.3), 180, 2.0)
    for _ in range(20):
        pose = (rng.uniform(-2.2, 2.2), rng.uniform(-2.2, 2.2), rng.uniform(-4, 4))
        pose = tuple(float(f32(v)) for v in pose)
        assert osl.match_score(0, obs.angle, obs.distance, obs.valid, pose) == ref.score(pose, obs.angle, obs.distance,
                                                                                          obs.valid)
    osl.close()


def test_score_borders_and_non_finite_endpoints():
    """Endpoints on the border cells (neighbours outside the grid), off the grid, and NaN / +-inf distances on valid
    beams (NaN lands on cell (0, 0) through `as usize`; +-inf leaves the grid)."""
    cfg = small_cfg()
    gw = O.grid_cells(cfg.width, cfg.resolution)
    n_free = np.zeros((gw, gw), np.uint16); n_occ = np.zeros((gw, gw), np.uint16)
    n_occ[0, :] = 1; n_occ[-1, :] = 1; n_occ[:, 0] = 1; n_occ[:, -1] = 1
    osl = _oracle_with(cfg, n_free, n_occ, radius=2)
    ref = Restated(cfg, n_free, n_occ, 2, 0.1, 0.05, 4, 32)
    angle = np.array([0.0, np.pi / 2, np.pi, -np.pi / 2, 0.3, 0.1, 0.2, 0.4, 0.0], np.float64)
    dist = np.array([1.99, 1.99, 1.995, 1.97, np.nan, np.inf, -np.inf, 5.0, 2.03], np.float64)
    valid = np.ones(angle.size, np.uint8)
    per = ref.beam_scores((0.0, 0.0, 0.0), angle, dist)
    assert per[0] > 0 and per[4] > 0            # a border cell; the NaN beam on cell (0, 0)
    assert per[5] == 0 and per[6] == 0 and per[7] == 0 and per[8] == 0   # off the grid
    for pose in [(0.0, 0.0, 0.0), (0.005, -0.013, 0.002), (0.03, 0.01, -0.01)]:
        assert osl.match_score(0, angle, dist, valid, pose) == ref.score(pose, angle, dist, valid)
    valid[:] = 0
    assert osl.match_score(0, angle, dist, valid, (0.0, 0.0, 0.0)) == 0
    osl.close()


# ---------------------------------------------------------------------------------------------- the climb
def _climb_both(cfg, n_free, n_occ, obs, pose, **m):
    osl = _oracle_with(cfg, n_free, n_occ, **m)
    ref = Restated(cfg, n_free, n_occ, m["radius"], m["step_xy"], m["step_theta"], m["levels"], m["max_moves"])
    got, moves, scored = osl.match_climb(0, obs.angle, obs.distance, obs.valid, pose)
    want, wm, ws, log = ref.climb(pose, obs.angle, obs.distance, obs.valid)
    osl.close()
    assert np.array_equal(_bits(got), _bits(want)), (got, want)
    assert (moves, scored) == (wm, ws)
    return got, moves, scored, log


@pytest.mark.parametrize("radius", [0, 1, 2])
def test_climb_matches_oracle_in_a_room(radius):
    cfg = small_cfg(res=0.02)
    segs = reference_scene(1.0)
    n_free, n_occ = _room_counts(cfg, segs)
    true = (f32(0.1), f32(-0.2), f32(0.3))
    obs = scan(segs, true, 360, 2.0)
    start = (f32(0.16), f32(-0.25), f32(0.33))
    m = dict(radius=radius, step_xy=0.1, step_theta=0.05, levels=4, max_moves=32)
    got, moves, scored, log = _climb_both(cfg, n_free, n_occ, obs, start, **m)
    assert moves > 0
    assert {lv for lv, _, k in log if k is not None} - {0}, "moves happened only at the first level"
    # every accepted move strictly improved, and each level ended on a round with no improvement (or the cap)
    last = None
    for lv, sc, k in log:
        if k is not None:
            assert sc[k] == max(sc) and sc.index(max(sc)) == k
            assert last is None or sc[k] > last
            last = sc[k]


def test_climb_first_candidate_wins_ties():
    """A single valid beam pointing along +x onto a wall cell that both (x+d, y) and (x, y+d) reach with the same
    score: the climb takes (x+d, y), the first of the tied candidates."""
    cfg = small_cfg(res=0.1, side=2.0)
    gw = O.grid_cells(cfg.width, cfg.resolution)
    n_free = np.zeros((gw, gw), np.uint16); n_occ = np.zeros((gw, gw), np.uint16)
    # the endpoint from (0.05, 0.05) at 0.5 m along +x lies in cell (15, 10); occupied: (16, 11) and its row/column
    n_occ[11, 16] = 1
    obs = type("Obs", (), {})()
    obs.angle = np.array([0.0]); obs.distance = np.array([0.5]); obs.valid = np.array([1], np.uint8)
    start = (f32(0.05), f32(0.05), f32(0.0))
    got, moves, scored, log = _climb_both(cfg, n_free, n_occ, obs, start, radius=1, step_xy=0.1, step_theta=0.001,
                                          levels=1, max_moves=8)
    lv, sc, k = log[0]
    assert sc[0] == sc[2] == max(sc) and k == 0, log
    assert moves >= 1 and got[0] > start[0]


def test_climb_stops_at_max_moves_and_on_no_improvement():
    cfg = small_cfg(res=0.02)
    segs = reference_scene(1.0)
    n_free, n_occ = _room_counts(cfg, segs)
    obs = scan(segs, (0.1, -0.2, 0.3), 360, 2.0)
    start = (f32(0.25), f32(-0.05), f32(0.4))
    got, moves, scored, _ = _climb_both(cfg, n_free, n_occ, obs, start, radius=1, step_xy=0.02, step_theta=0.01,
                                        levels=3, max_moves=2)
    assert moves == 2 and scored == 1 + 6 * 2          # the cap ends every later level at once
    # an empty grid scores 0 everywhere: no candidate is strictly better, one round per level
    empty = np.zeros_like(n_free)
    got, moves, scored, _ = _climb_both(cfg, empty, empty, obs, start, radius=1, step_xy=0.1, step_theta=0.05,
                                        levels=3, max_moves=32)
    assert moves == 0 and scored == 1 + 6 * 3 and np.array_equal(_bits(got), _bits(start))


def test_climb_on_grids_from_oracle_steps():
    cfg = small_cfg(n=4)
    scans = make_scans(1.0, 360, 1.0, 6)
    osl = oracle_slam(cfg)
    for step, (obs, odo) in enumerate(scans[:5]):
        assert oracle_step(O, osl, obs, odo, step)[0] == 0
    nf, no = osl.counts(0)
    gw = osl.gw
    m = dict(radius=1, step_xy=0.1, step_theta=0.05, levels=4, max_moves=32)
    osl.set_scan_match(**m)
    ref = Restated(cfg, nf.reshape(gw, gw), no.reshape(gw, gw), 1, 0.1, 0.05, 4, 32)
    obs = scans[5][0]
    ang = obs.angle.astype(np.float32).astype(np.float64); dist = obs.distance.astype(np.float32).astype(np.float64)
    pose0 = osl.poses()[0]
    rng = np.random.default_rng(5)
    total_moves = 0
    for k in range(6):
        pose = (pose0 + rng.normal(0, [0.05, 0.05, 0.05])).astype(np.float32)
        got, moves, scored = osl.match_climb(0, ang, dist, obs.valid, pose)
        want, wm, ws, _ = ref.climb(pose, ang, dist, obs.valid)
        assert np.array_equal(_bits(got), _bits(want)) and (moves, scored) == (wm, ws)
        total_moves += moves
    assert total_moves > 0
    osl.close()


def test_oracle_update_with_matcher_refines_and_reports():
    """so_update with the matcher: the stats add up, and with it off the update is the reference's bit for bit."""
    cfg = small_cfg(n=8)
    scans = make_scans(1.0, 360, 1.0, 6)
    a, b = oracle_slam(cfg), oracle_slam(cfg)
    b.set_scan_match(radius=1, step_xy=0.1, step_theta=0.05, levels=4, max_moves=32)
    moved = 0
    for step, (obs, odo) in enumerate(scans):
        if step < 2:
            b.set_scan_match(levels=0)
        elif step == 2:
            b.set_scan_match(radius=1, step_xy=0.1, step_theta=0.05, levels=4, max_moves=32)
        oracle_step(O, a, obs, odo, step); oracle_step(O, b, obs, odo, step)
        st = b.scan_match_stats()
        if step < 2:
            assert st == (0, 0, 0, 0)
            assert np.array_equal(_bits(a.poses()), _bits(b.poses()))
            assert np.array_equal(a.weights()[1], b.weights()[1])
        else:
            assert st[2] >= cfg.n_particles * 7 and st[1] >= st[0] and st[3] <= st[0]
            moved += st[0]
    assert moved > 0
    a.close(); b.close()


# ---------------------------------------------------------------------------------------------- convergence
def test_climb_converges_in_a_hand_drawn_room():
    cfg = small_cfg(res=0.01, side=3.0)
    segs = np.array(rect_segments(-1.2, -1.0, 2.4, 2.0) + rect_segments(-0.3, 0.2, 0.4, 0.3), np.float32)
    n_free, n_occ = _room_counts(cfg, segs)
    levels, step_xy, step_theta = 4, 0.08, 0.08
    fine_xy, fine_th = step_xy / 2 ** (levels - 1), step_theta / 2 ** (levels - 1)
    for true, off in [((0.1, -0.2, 0.3), (0.04, -0.03, 0.03)), ((-0.5, 0.4, -1.0), (-0.03, -0.04, -0.02)),
                      ((0.6, -0.5, 2.0), (0.05, 0.02, 0.04))]:
        true = tuple(f32(v) for v in true)
        obs = scan(segs, true, 360, 4.0)
        start = tuple(f32(t + o) for t, o in zip(true, off))
        got, moves, _, _ = _climb_both(cfg, n_free, n_occ, obs, start, radius=1, step_xy=step_xy,
                                       step_theta=step_theta, levels=levels, max_moves=64)
        assert moves > 0
        assert abs(float(got[0]) - float(true[0])) <= fine_xy + 1e-6, (got, true)
        assert abs(float(got[1]) - float(true[1])) <= fine_xy + 1e-6, (got, true)
        assert abs(float(got[2]) - float(true[2])) <= fine_th + 1e-6, (got, true)


# ---------------------------------------------------------------------------------------------- argument checks
def test_scan_matcher_struct_and_oracle_argument_checks():
    assert C.sizeof(_lib.ScanMatch) == 24
    m = ScanMatcher().to_struct()
    assert m.struct_size == 24 and m.radius == 1 and m.levels == 4 and m.max_moves == 32
    cfg = small_cfg()
    osl = oracle_slam(cfg)
    for bad in [dict(radius=3), dict(step_xy=0.0), dict(step_xy=float("inf")), dict(step_theta=-0.1),
                dict(step_theta=float("nan")), dict(levels=9), dict(max_moves=0), dict(max_moves=1025)]:
        with pytest.raises(ValueError):
            osl.set_scan_match(**bad)
    osl.set_scan_match(levels=0)
    osl.close()
    no_counts = oracle_slam(cfg, track_counts=False)
    with pytest.raises(ValueError):
        no_counts.set_scan_match()
    no_counts.set_scan_match(levels=0)       # off needs no counters
    no_counts.close()


def test_set_scan_match_rejects_a_null_handle():
    L = _lib.load()
    m = ScanMatcher().to_struct()
    assert L.slamrs_gpu_set_scan_match(None, C.byref(m)) == _lib.E_INVALID_ARG
    out = np.zeros(4, np.uint64)
    assert L.slamrs_gpu_get_scan_match_stats(None, out.ctypes.data_as(C.c_void_p)) == _lib.E_INVALID_ARG
