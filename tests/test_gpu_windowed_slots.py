"""Windowed grid slots (slot_cells, DESIGN.md section 2) in lockstep with the CPU oracle, at the places where a torus
window goes wrong: seams, aliased cells, tenancy changes, copy fan-outs, modes not otherwise combined with windowed
slots, and the extent limits.

A windowed slot holds a P x P torus of the logical grid: cell (x, y) lives at (y & (P-1), x & (P-1)), then tiled. A
reader must refuse every cell outside the informed extent, because the physical cell there belongs to another logical
cell; a copy must clear the destination's old tenant; the ray kernels must prove that an extent still fits before they
write. A mistake in any of these shows up only as a wrong cell somewhere else on the torus, so every case here asserts
the geometry it is named for (from gpu.extents) as well as the oracle's results. Grids are 1024^2 at 2 cm with P = 256
unless a case says otherwise: seams at logical 256, 512 and 768."""
from __future__ import annotations

import dataclasses

import numpy as np
import pytest

from slamrs_b200 import GpuPlacement, GridMapSlam, GridMapSlamConfig, Observation, Odometry, ScanMatcher, _lib
from oracle.scan_match_oracle import ScanMatchOracle

from common import SEED, compare_step, install_cells, make_scans, oracle_step

pytestmark = pytest.mark.gpu

P = 256
RES = 0.02
WIDTH = {1024: 20.48, 776: 15.51, 1001: 20.01}   # logical side in cells -> width in metres at 2 cm
STILL = Odometry(0.0, 0.0, 0.1)                  # with zero draws the sampled pose is the start pose
COPY_MODES = pytest.mark.parametrize("copy_flags", [0, _lib.FLAG_EAGER_COPY, _lib.FLAG_FULL_GRID_COPY],
                                     ids=["deferred", "eager", "whole-slot"])


def config(n, side=1024):
    w = WIDTH[side]
    return GridMapSlamConfig(position=(-w / 2, -w / 2), width=w, height=w, resolution=RES, n_particles=n)


def cell_pose(cfg, cx, cy, theta=0.0):
    """World pose at the centre of logical cell (cx, cy)."""
    return [cfg.position[0] + (cx + 0.5) * RES, cfg.position[1] + (cy + 0.5) * RES, theta]


def straddles(box, k, axis):
    x0, y0, x1, y1 = box
    lo, hi = (x0, x1) if axis == 0 else (y0, y1)
    return lo < k * P < hi


def f32_scan(obs: Observation):
    """The scan as both sides use it (the reference casts angle and distance to f32 at use)."""
    return (obs.angle.astype(np.float32).astype(np.float64), obs.distance.astype(np.float32).astype(np.float64),
            obs.valid.astype(np.uint8))


class Lockstep:
    """One device handle and one oracle (ScanMatchOracle: set_counts for hand-built grids; without a matcher set it
    is the plain oracle) stepped on the same scans. step() takes the oracle's shared-stream draws, or the caller's
    (z, u) in RNG_CALLER mode, and compares the step with compare_step."""

    def __init__(self, O, cfg, flags=0, slot_cells=P, rng_mode=_lib.RNG_SHARED_STREAM, tau=0.0):
        self.O, self.cfg, self.rng_mode = O, cfg, rng_mode
        self.gpu = GridMapSlam(cfg, GpuPlacement(seed=SEED, rng_mode=rng_mode, flags=flags, slot_cells=slot_cells,
                                                 resample_threshold=tau))
        self.osl = ScanMatchOracle(cfg.position, cfg.width, cfg.height, cfg.resolution, cfg.n_particles, True)
        if tau:
            self.osl.set_adaptive_resampling(tau)
        self.n = cfg.n_particles
        self.step_no = 0

    def close(self):
        self.gpu.close()
        self.osl.close()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def set_poses(self, xyt):
        xyt = np.asarray(xyt, np.float32).reshape(self.n, 3)
        self.gpu.set_poses(xyt)
        self.osl.set_poses(xyt)

    def set_matcher(self, m):
        self.gpu.set_scan_matcher(m)
        self.osl.set_scan_match(**dataclasses.asdict(m))

    def update(self, obs, odo, z=None, u=None):
        """One step on both sides, without comparing. Returns the device's error (None on success)."""
        if self.rng_mode == _lib.RNG_CALLER and z is not None:
            a, d, v = f32_scan(obs)
            rc = self.osl.update(a, d, v, np.float32(odo.distance_left), np.float32(odo.distance_right),
                                 np.float32(odo.wheel_distance), np.ascontiguousarray(z, np.float64), float(u))
        else:
            rc, z, u = oracle_step(self.O, self.osl, obs, odo, self.step_no)
        assert rc == 0
        self.step_no += 1
        try:
            if self.rng_mode == _lib.RNG_CALLER:
                self.gpu.update(obs, odo, z_draws=z, resample_u=u)
            else:
                self.gpu.update(obs, odo)
        except _lib.SlamrsGpuError as e:
            return e
        return None

    def step(self, obs, odo, z=None, u=None, particles=None, check_map=True):
        err = self.update(obs, odo, z, u)
        assert err is None, err
        return compare_step(self.gpu, self.osl, particles, check_map=check_map)

    def indices(self):
        return self.gpu.resample_indices().astype(np.int64)


# ------------------------------------------------------------------------------------------------ seams
def _seam_starts():
    """(cx, cy, kx, ky): start cells on k*P - 1, k*P and k*P + 1 in x, in y and in both (k = 1, 2, 3); 0 = no seam on
    that axis (the other coordinate sits half-way between two seams)."""
    out = []
    for k in (1, 2, 3):
        for d in (-1, 0, 1):
            c = k * P + d
            out += [(c, 640, k, 0), (640, c, 0, k), (c, c, k, k)]
    return out


@COPY_MODES
@pytest.mark.parametrize("kernel", [0, _lib.FLAG_GENERIC_RAY_KERNEL], ids=["packed", "generic"])
def test_seams(oracle, kernel, copy_flags):
    """27 particles start on the seams (x, y, and the corner where both axes wrap); 6 scans of a 1 m lidar, so the
    extents keep growing across the seam after they first straddle it. Every particle's box must straddle its
    lineage's seam after every step."""
    starts = _seam_starts()
    cfg = config(len(starts))
    rng = np.random.default_rng(11)
    poses = [cell_pose(cfg, cx, cy, float(rng.uniform(-np.pi, np.pi))) for cx, cy, _, _ in starts]
    seam = np.array([(kx, ky) for _, _, kx, ky in starts])
    with Lockstep(oracle, cfg, flags=kernel | copy_flags) as ls:
        ls.set_poses(poses)
        for obs, odo in make_scans(1.0, 360, 1.0, 6):
            ls.step(obs, odo)
            seam = seam[ls.indices()]
            for p in range(cfg.n_particles):
                box = ls.gpu.extents(p)[0]
                kx, ky = seam[p]
                assert (kx == 0 or straddles(box, kx, 0)) and (ky == 0 or straddles(box, ky, 1)), (p, box, kx, ky)
        assert np.any(seam[:, 0] * seam[:, 1] > 0), "no corner particle left"


# ------------------------------------------------------------------------------------------------ aliased reads
def _endpoint_cell(O, cfg, pose, angle, dist):
    """The cell a beam's endpoint falls in, with the f32 operations of beam_endpoint and world_to_grid."""
    a = np.float32(np.float32(pose[2]) + np.float32(angle))
    s, c = O.libm_sincosf(np.array([a], np.float32))
    ex = np.float32(np.float32(pose[0]) + np.float32(c[0] * np.float32(dist)))
    ey = np.float32(np.float32(pose[1]) + np.float32(s[0] * np.float32(dist)))
    gx = np.float32(np.float32(ex - np.float32(cfg.position[0])) / np.float32(RES))
    gy = np.float32(np.float32(ey - np.float32(cfg.position[1])) / np.float32(RES))
    return int(np.floor(gx)), int(np.floor(gy))


def _beam_to(O, cfg, pose, cell):
    """(angle, distance) in f32 of a beam from `pose` whose endpoint lands in `cell`."""
    tx, ty = cfg.position[0] + (cell[0] + 0.5) * RES, cfg.position[1] + (cell[1] + 0.5) * RES
    ang = np.float32(np.arctan2(ty - float(pose[1]), tx - float(pose[0])) - float(pose[2]))
    dist = np.float32(np.hypot(tx - float(pose[0]), ty - float(pose[1])))
    assert _endpoint_cell(O, cfg, pose, ang, dist) == tuple(cell), (pose, cell)
    return float(ang), float(dist)


PUSH = 30.0   # centre-distance draw of a particle that must not survive: weight * exp(-450), far from underflow


def _sampled_pose(O, start, z1):
    return O.odometry_sample(O.odometry_new(0.0, 0.0, 0.1), start, z1, 0.0)


@COPY_MODES
def test_aliased_endpoints_read_the_prior(oracle, copy_flags):
    """Particles 0-3 each hold a hand-built grid of free cells q; the scan's endpoints from their poses land on
    q + (+-P, 0), (0, +-P) and (+-P, +-P): outside the extent, on the physical cell of q. The likelihood must read
    them as the prior. A ghost read adds log(0.9 * p + 0.1) ~ -2.2 to a log weight of which the oracle has 0, so
    weights within 1e-9 catch it. Particles 0-3 are pushed 30 sigma out (they do not survive and are never
    integrated; a ray to an aliased cell could not fit the window); particles 4-7 hold empty grids and survive,
    and two more scans run on their clones in the old tenants' slots."""
    cfg = config(8)
    O = oracle
    cells_a, beams, targets = [], [], []
    starts = []
    for q_i, (sx, sy) in enumerate([(1, 1), (-1, 1), (1, -1), (-1, -1)]):
        centre = (300 if sx > 0 else 700, 300 if sy > 0 else 700)
        start = np.array(cell_pose(cfg, *centre), np.float32)
        starts.append(start)
        pose = _sampled_pose(O, start, PUSH)
        pc = (int(np.floor((pose[0] - cfg.position[0]) / RES)), int(np.floor((pose[1] - cfg.position[1]) / RES)))
        img = np.zeros((1024, 1024), np.uint32)
        tq = []
        for (ox, oy), (ux, uy) in [((sx * P, 0), (sx * 60, 0)), ((0, sy * P), (0, sy * 60)),
                                    ((sx * P, sy * P), (sx * 42, sy * 42))]:
            a = (pc[0] + ux, pc[1] + uy)
            q = (a[0] - ox, a[1] - oy)
            img[q[1], q[0]] = 5                      # five free hits: p = 0.015
            beams.append(_beam_to(O, cfg, pose, a))
            tq.append((a, q))
        cells_a.append(img)
        targets.append(tq)
    for cx, cy in [(150, 900), (400, 850), (880, 160), (900, 420)]:
        starts.append(np.array(cell_pose(cfg, cx, cy), np.float32))
    ang = np.array([b[0] for b in beams]); dist = np.array([b[1] for b in beams])
    obs = Observation(0, angle=ang, distance=dist, valid=np.ones(ang.size, bool))
    with Lockstep(O, cfg, flags=copy_flags, rng_mode=_lib.RNG_CALLER) as ls:
        for p in range(4):
            install_cells(ls.gpu, ls.osl, p, cells_a[p])
        ls.set_poses(np.array(starts))
        for p in range(4):
            box = ls.gpu.extents(p)[0]
            for a, q in targets[p]:
                inside = lambda c: box[0] <= c[0] < box[2] and box[1] <= c[1] < box[3]   # noqa: E731
                assert inside(q) and not inside(a) and (a[0] - q[0]) % P == 0 and (a[1] - q[1]) % P == 0, (p, box, a, q)
        z = np.zeros(16); z[0:8:2] = PUSH
        ls.step(obs, STILL, z, 0.5)
        raw = ls.gpu.weights()[1]
        assert np.all(raw[:4] > 0) and np.all(raw[:4] < 1e-150 * raw[4:].min()), raw
        assert set(ls.indices().tolist()) <= {4, 5, 6, 7}
        rng = np.random.default_rng(3)
        for obs2, odo2 in make_scans(1.0, 360, 1.0, 2):
            ls.step(obs2, odo2, rng.standard_normal(16) * 0.5, float(rng.random()))


def test_aliased_endpoints_scan_matcher(oracle):
    """The scan matcher at radius 2 around endpoints just outside an extent that is exactly P wide with both edges on
    seams (x in [256, 512)): occupied cells at x = 511 (inside, one cell from the endpoint) and at x = 256, whose
    physical cell the endpoint column 512 shares. Neighbourhoods cross the extent's edge; a ghost read would score the
    endpoint cell itself. The same in y. Poses and the matcher statistics must equal the oracle's."""
    cfg = config(4)
    O = oracle
    img_x = np.zeros((1024, 1024), np.uint32)
    img_x[600:606, 256] = 3 << 16
    img_x[600:606, 511] = 3 << 16
    img_y = img_x.T.copy()
    starts = [np.array(cell_pose(cfg, 560, 590), np.float32), np.array(cell_pose(cfg, 590, 560), np.float32),
              np.array(cell_pose(cfg, 150, 150), np.float32), np.array(cell_pose(cfg, 850, 850), np.float32)]
    beams = []
    for p, img in ((0, img_x), (1, img_y)):
        pose = _sampled_pose(O, starts[p], PUSH)
        for j in range(600, 606):
            beams.append(_beam_to(O, cfg, pose, (512, j) if p == 0 else (j, 512)))
    ang = np.array([b[0] for b in beams]); dist = np.array([b[1] for b in beams])
    obs = Observation(0, angle=ang, distance=dist, valid=np.ones(ang.size, bool))
    m = ScanMatcher(radius=2, step_xy=0.04, step_theta=0.02, levels=3, max_moves=16)
    with Lockstep(O, cfg, rng_mode=_lib.RNG_CALLER) as ls:
        install_cells(ls.gpu, ls.osl, 0, img_x)
        install_cells(ls.gpu, ls.osl, 1, img_y)
        assert ls.gpu.extents(0)[0] == (256, 600, 512, 606) and ls.gpu.extents(1)[0] == (600, 256, 608, 512)
        ls.set_poses(np.array(starts))
        ls.set_matcher(m)
        z = np.zeros(8); z[0:4:2] = PUSH
        ls.step(obs, STILL, z, 0.5)
        s = ls.gpu.scan_match_stats()
        assert (s["moved"], s["moves"], s["scored"], s["capped"]) == ls.osl.scan_match_stats()
        assert s["scored"] > 0


@pytest.mark.parametrize("fmt", [_lib.MAP_F64, _lib.MAP_F32, _lib.MAP_U8], ids=["f64", "f32", "u8"])
def test_aliased_cells_in_exported_windows(oracle, fmt):
    """estimated_likelihood_window over windows that hold a cell and its aliases: the aliases read exactly 0.5
    (u8: 128) and every window equals the oracle's dense map."""
    cfg = config(1)
    rng = np.random.default_rng(8)
    img = np.zeros((1024, 1024), np.uint32)
    img[300:420, 200:440] = (rng.integers(0, 6, (120, 240)) | (rng.integers(0, 4, (120, 240)) << 16)).astype(np.uint32)
    img[300, 200] = 7
    img[419, 439] = 1 << 16
    with Lockstep(oracle, cfg, rng_mode=_lib.RNG_CALLER) as ls:
        install_cells(ls.gpu, ls.osl, 0, img)
        box = ls.gpu.extents(0)[0]
        assert box == (200, 300, 440, 420)
        ls.set_poses([cell_pose(cfg, 320, 360)])     # inside the box: the empty scan's square (reach 6) fits
        ls.step(Observation(0, angle=[], distance=[], valid=[]), STILL, np.zeros(2), 0.5)
        ref = ls.osl.estimated_likelihood().reshape(1024, 1024)
        conv = {_lib.MAP_F64: lambda a: a, _lib.MAP_F32: lambda a: a.astype(np.float32),
                _lib.MAP_U8: lambda a: np.rint(a * 255.0).astype(np.uint8)}[fmt]
        prior = conv(np.array([0.5]))[0]
        hits = 0
        for win in [(0, 0, 1024, 1024), (190, 290, 470, 570), (150, 40, 460, 430), (456, 556, 700, 700)]:
            x0, y0, x1, y1 = win
            got = ls.gpu.estimated_likelihood_window(window=win, fmt=fmt)[1]
            assert np.array_equal(got, conv(ref[y0:y1, x0:x1])), win
            for cx, cy in [(200, 300), (439, 419)]:
                assert ref[cy, cx] != 0.5
                for dx, dy in [(P, 0), (0, P), (P, P), (-P, 0), (0, -P), (-P, -P), (P, -P), (-P, P)]:
                    x, y = cx + dx, cy + dy
                    if x0 <= x < x1 and y0 <= y < y1 and 0 <= x < 1024 and 0 <= y < 1024:
                        assert got[y - y0, x - x0] == prior, (win, x, y)
                        hits += 1
        assert hits >= 6, hits


# ------------------------------------------------------------------------------------------------ tenancy changes
@COPY_MODES
def test_tenancy_change_clears_the_old_tenant(oracle, copy_flags):
    """Particles 0-3 hold grid G1 (logical [264, 384)^2, physical [8, 128)^2); particles 4-7 grid G2 (logical
    x [536, 560), y [280, 300): physical [24, 48) x [24, 44), inside G1's footprint). Only 4-7 survive the first step,
    so their clones take G1's slots. The survivors stand in G2's area and their extents grow over the physical cells
    that G1 informed, where stale cells would surface inside the clones' extents."""
    cfg = config(8)
    rng = np.random.default_rng(12)
    g1 = np.zeros((1024, 1024), np.uint32)
    g1[264:384, 264:384] = (rng.integers(1, 6, (120, 120)) | (rng.integers(0, 3, (120, 120)) << 16)).astype(np.uint32)
    g2 = np.zeros((1024, 1024), np.uint32)
    g2[280:300, 536:560] = rng.integers(1, 4, (20, 24)).astype(np.uint32) << 16
    scans = make_scans(1.0, 360, 1.0, 6)
    with Lockstep(oracle, cfg, flags=copy_flags, rng_mode=_lib.RNG_CALLER) as ls:
        for p in range(8):
            install_cells(ls.gpu, ls.osl, p, g1 if p < 4 else g2)
        ls.set_poses([cell_pose(cfg, 300 + 20 * (p % 4), 320, 0.5 * p) if p < 4 else
                      cell_pose(cfg, 545 + 3 * p, 290, 0.7 * p) for p in range(8)])
        z = rng.standard_normal(16) * 0.3
        z[0:8:2] = 38.0
        ls.step(*scans[0], z, 0.5)
        idx = ls.indices()
        assert set(idx.tolist()) <= {4, 5, 6, 7}, idx
        covered = False
        for obs, odo in scans[1:]:
            ls.step(obs, odo, rng.standard_normal(16) * 0.5, float(rng.random()))
            for p in range(8):
                x0, y0, x1, y1 = ls.gpu.extents(p)[0]
                # some cell of the extent is physically one that G1 informed, and G2 did not
                xs = np.arange(x0, x1) % P
                ys = np.arange(y0, y1) % P
                if np.any((xs >= 8) & (xs < 128) & ((xs < 24) | (xs >= 48))) and np.any((ys >= 8) & (ys < 128)):
                    covered = True
        assert covered, "no clone's extent grew over the old tenant's cells"


# ------------------------------------------------------------------------------------------------ fan-out
@pytest.mark.parametrize("copy_flags", [0, _lib.FLAG_EAGER_COPY], ids=["deferred", "eager"])
@pytest.mark.parametrize("n,survivors", [(17, (8,)), (33, (8,)), (48, (8,)), (40, (3, 30))],
                         ids=["17-one", "33-one", "48-one", "40-two"])
def test_fan_out_past_sixteen_on_a_ring(oracle, n, survivors, copy_flags):
    """Particles start on the seam corner (512, 512); in step 1 only `survivors` keep sane draws, so one source has
    more than COPY_FAN = 16 clones, all on a ring. In step 2 every particle has zero draws and the clones of one
    source identical weights, so (u = 0.5) every clone survives and the deferred mode copies them all from one root.
    Step 3 is an ordinary step."""
    cfg = config(n)
    rng = np.random.default_rng(n)
    scans = make_scans(1.0, 360, 1.0, 4)
    with Lockstep(oracle, cfg, flags=copy_flags, rng_mode=_lib.RNG_CALLER) as ls:
        ls.set_poses([cell_pose(cfg, 510 + p % 5, 510 + p % 3, float(rng.uniform(-np.pi, np.pi))) for p in range(n)])
        ls.step(*scans[0], rng.standard_normal(2 * n) * 0.5, 0.5)
        z = np.zeros(2 * n); z[0::2] = 38.0
        for s in survivors:
            z[2 * s] = 0.0
        ls.step(*scans[1], z, 0.5)
        idx = ls.indices()
        src, counts = np.unique(idx, return_counts=True)
        assert set(src.tolist()) <= set(survivors) and counts.max() > 16, (src, counts)
        for s in src:
            box = ls.gpu.extents(int(np.nonzero(idx == s)[0][0]))[0]
            assert straddles(box, 2, 0) and straddles(box, 2, 1), box
        st = ls.gpu.stats()
        if copy_flags & _lib.FLAG_EAGER_COPY:
            assert st["grids_copied"] == n - len(src), st
        ls.step(*scans[2], np.zeros(2 * n), 0.5)
        st2 = ls.gpu.stats()
        if not copy_flags & _lib.FLAG_EAGER_COPY and len(src) == 1:
            # every clone survived: all but one per root are copied from it now
            assert st2["distinct_sources"] == n, st2
            assert st2["grids_copied"] == n - len(src), st2
        ls.step(*scans[3], rng.standard_normal(2 * n) * 0.5, float(rng.random()))


# ------------------------------------------------------------------------------------------------ modes
MODE_CASES = {
    "eager-copy": dict(flags=_lib.FLAG_EAGER_COPY),
    "update-all": dict(flags=_lib.FLAG_UPDATE_ALL_PARTICLES),
    "adaptive": dict(tau=0.5),
    "rng-caller": dict(rng_mode=_lib.RNG_CALLER),
    "4096-beams": dict(beams=4096),
    "side-776": dict(side=776),
    "side-1001": dict(side=1001),
}


@pytest.mark.parametrize("case", list(MODE_CASES))
def test_modes_with_windowed_slots(oracle, case):
    """Modes that no other windowed test combines with windowed slots. Particles start on seams; scattered headings.
    776 = 3 * 256 + 8 leaves a partial last ring; 1001 is not a multiple of 8, so extent copies are off and windowed
    slots take whole-slot copies."""
    kw = MODE_CASES[case]
    side = kw.get("side", 1024)
    n = 20
    cfg = config(n, side)
    rng = np.random.default_rng(len(case))
    seams = [P, 2 * P, 3 * P] if side >= 3 * P + 8 else [P, 2 * P]
    poses = []
    for p in range(n):
        k = seams[p % len(seams)] + (p % 3) - 1
        cx, cy = (k, k) if p % 2 else (k, 640 if k != 2 * P else 384)
        cy = min(cy, side - 60)
        poses.append(cell_pose(cfg, cx, cy, float(rng.uniform(-np.pi, np.pi))))
    scans = make_scans(1.0, kw.get("beams", 360), 1.0, 6)
    if kw.get("beams"):
        assert len(scans[0][0]) > 2047      # more beams than the packed window takes: the generic kernel
    resampled = []
    copied = 0
    with Lockstep(oracle, cfg, flags=kw.get("flags", 0), rng_mode=kw.get("rng_mode", _lib.RNG_SHARED_STREAM),
                  tau=kw.get("tau", 0.0)) as ls:
        ls.set_poses(poses)
        for obs, odo in scans:
            ls.step(obs, odo, particles=range(0, n, 3))
            resampled.append(ls.osl.resampled())
            st = ls.gpu.stats()
            assert st["window_overflow"] == 0
            if side == 1001 and st["grids_copied"]:
                # whole slots: every copy moves the slot's bytes
                assert st["copy_bytes"] >= st["grids_copied"] * st["bytes_per_grid"] == st["grids_copied"] * P * P * 4, st
                copied += st["grids_copied"]
        if kw.get("tau"):
            assert not all(resampled), resampled       # a step that carried its weights forward
        else:
            assert all(resampled)
        if side == 1001:
            assert copied > 0
        crossing = sum(any(straddles(ls.gpu.extents(p)[0], k // P, a) for k in seams for a in (0, 1)) for p in range(n))
        assert crossing > 0


# ------------------------------------------------------------------------------------------------ extent limits
def test_set_cells_extent_limits():
    """An image whose 8-aligned box is exactly P wide and P high round-trips, also where it wraps the torus; a box
    P + 8 wide -- also one made so only by the 8-alignment of x0 -- or P + 1 high is E_WINDOW."""
    cfg = config(2)
    with GridMapSlam(cfg, GpuPlacement(slot_cells=P)) as g:
        def img(xs, ys):
            a = np.zeros((1024, 1024), np.uint32)
            for x in xs:
                for y in ys:
                    a[y, x] = 0x10002
            return a
        for x0, y0 in [(8, 0), (128, 384), (768, 768), (504, 500)]:
            a = img([x0, x0 + P - 1], [y0, y0 + P - 1])
            g.set_cells(1, a)
            assert g.extents(1)[0] == (x0, y0, x0 + P, y0 + P)
            assert np.array_equal(g.cells(1).reshape(1024, 1024), a)
        for xs, ys in [([8, 8 + P], [0]),                 # P + 1 columns: box P + 8
                       ([12, 12 + P - 1], [0]),           # P columns, but x0 aligns down to 8: box P + 8
                       ([8], [100, 100 + P])]:            # P + 1 rows
            with pytest.raises(_lib.SlamrsGpuError) as e:
                g.set_cells(0, img(xs, ys))
            assert e.value.code == _lib.E_WINDOW


@pytest.mark.parametrize("flags", [0, _lib.FLAG_UPDATE_ALL_PARTICLES], ids=["survivors", "update-all"])
def test_overflowing_step(oracle, flags):
    """Particles 0-3 hold a 200-cell-wide image far from where all eight stand: their extent plus the scan's square
    cannot fit P, particles 4-7 (empty grids) fit. Overflow is detected after resampling, so indices, poses and
    weights equal the oracle's; the grids that did not overflow equal the oracle's, each overflowing grid equals its
    source's grid before the step, and stats counts the overflowing grids."""
    cfg = config(8)
    rng = np.random.default_rng(4)
    wide = np.zeros((1024, 1024), np.uint32)
    wide[480:520, 100:300] = rng.integers(1, 5, (40, 200)).astype(np.uint32)
    (obs, _), = make_scans(1.0, 360, 1.0, 1)
    with Lockstep(oracle, cfg, flags=flags, rng_mode=_lib.RNG_CALLER) as ls:
        for p in range(4):
            install_cells(ls.gpu, ls.osl, p, wide)
        ls.set_poses([cell_pose(cfg, 600, 500)] * 8)
        before = [ls.gpu.cells(p).copy() for p in range(8)]
        err = ls.update(obs, STILL, np.zeros(16), 0.5)
        assert err is not None and err.code == _lib.E_WINDOW
        idx = ls.indices()
        assert np.array_equal(idx, ls.osl.indices().astype(np.int64))
        assert np.array_equal(ls.gpu.poses().view(np.uint32), ls.osl.poses().view(np.uint32))
        w, raw = ls.gpu.weights()
        w_ref, raw_ref = ls.osl.weights()
        assert np.max(np.abs(raw - raw_ref) / np.abs(raw_ref)) < 1e-9
        assert np.max(np.abs(w - w_ref) / np.abs(w_ref)) < 1e-9
        over = [p for p in range(8) if idx[p] < 4]
        assert len(set(idx[over].tolist())) == ls.gpu.stats()["window_overflow"] == 4, (idx, ls.gpu.stats())
        for p in range(8):
            if idx[p] < 4:
                assert np.array_equal(ls.gpu.cells(p), before[idx[p]]), p
            else:
                nf, no = ls.osl.counts(p)
                gf, go = ls.gpu.counts(p)
                assert np.array_equal(nf, gf) and np.array_equal(no, go), p


# ------------------------------------------------------------------------------------------------ the refusal rule
def window_would_overflow(P_, gw, gh, box, cx, cy, distances):
    """kernels_ray.cu window_would_overflow with the host's reach: reach = ceil(max |distance| / res) + 6 over every
    beam of the scan, valid or not (slamrs_gpu_upload_scan); the square of side 2 reach + 1 around the start cell,
    x widened to multiples of 8 and clipped to the grid, united with the informed box, must fit P x P."""
    maxd = np.float32(0.0)
    for d in np.abs(np.asarray(distances, np.float32)):
        if not np.isfinite(d):
            maxd = np.float32(np.inf)
            break
        maxd = max(maxd, d)
    cells = np.ceil(np.float32(maxd / np.float32(RES)))
    reach = (int(cells) if cells < 4096 else 4096) + 6
    x0 = max(0, cx - reach) & ~7
    x1 = min(gw, (min(gw, cx + reach + 1) + 7) & ~7)
    y0, y1 = max(0, cy - reach), min(gh, cy + reach + 1)
    if box[2] > box[0] and box[3] > box[1]:
        x0, x1, y0, y1 = min(x0, box[0]), max(x1, box[2]), min(y0, box[1]), max(y1, box[3])
    return x1 - x0 > P_ or y1 - y0 > P_


def test_refusal_rule(oracle):
    """The window proof on both sides of its boundary, pinned against the restatement above. Twelve particles with
    empty grids stand on start cells whose square is exactly P (reach 127 with x aligned), one cell over through the
    8-alignment of x, and at the grid border; the scan's longest beam decides the reach for all of them, and it
    counts when it is invalid too. Zero draws and u = 0.5: every particle survives and is integrated."""
    starts = [(511, 500), (513, 500), (504, 504), (519, 300), (100, 127), (127, 900), (1000, 1000), (3, 3),
              (639, 639), (641, 640), (383, 200), (385, 700)]
    n = len(starts)
    cfg = config(n)
    (obs, _), = make_scans(1.0, 360, 1.0, 1)
    rng = np.random.default_rng(5)
    # the longest f32 distance that is 121 cells at 2 cm after ceil (reach 127), and the next f32 (122 cells, reach 128)
    def cells(d):
        return int(np.ceil(np.float32(np.float32(d) / np.float32(RES))))
    d121 = np.float32(121 * RES)
    while cells(d121) > 121:
        d121 = np.nextafter(d121, np.float32(0))
    while cells(np.nextafter(d121, np.float32(10))) <= 121:
        d121 = np.nextafter(d121, np.float32(10))
    d122 = np.nextafter(d121, np.float32(10))
    assert cells(d121) == 121 and cells(d122) == 122
    cases = []
    for longest, valid in [(d121, True), (d122, True), (d122, False), (d121, False)]:
        d = obs.distance.astype(np.float32).copy()
        v = obs.valid.copy()
        d[0] = longest
        v[0] = valid
        cases.append(Observation(0, angle=obs.angle, distance=d.astype(np.float64), valid=v))
    for scan in cases:
        verdict = [window_would_overflow(P, 1024, 1024, (0, 0, 0, 0), cx, cy, scan.distance) for cx, cy in starts]
        assert any(verdict) and (scan.distance[0] > d121 or not all(verdict)), verdict
        with Lockstep(oracle, cfg, rng_mode=_lib.RNG_CALLER) as ls:
            ls.set_poses([cell_pose(cfg, cx, cy, float(rng.uniform(-np.pi, np.pi))) for cx, cy in starts])
            err = ls.update(scan, STILL, np.zeros(2 * n), 0.5)
            assert np.array_equal(ls.indices(), np.arange(n))
            assert ls.gpu.stats()["window_overflow"] == sum(verdict), (verdict, ls.gpu.stats())
            assert (err is not None) == any(verdict)
            if err is not None:
                assert err.code == _lib.E_WINDOW
            for p in range(n):
                gf, go = ls.gpu.counts(p)
                if verdict[p]:
                    assert not gf.any() and not go.any(), p
                else:
                    nf, no = ls.osl.counts(p)
                    assert np.array_equal(nf, gf) and np.array_equal(no, go), p
    # a scan without beams still has reach 6: a particle standing 72 cells beyond its 240-cell box is refused
    img = np.zeros((1024, 1024), np.uint32)
    img[300:420, 200:440] = 1
    assert window_would_overflow(P, 1024, 1024, (200, 300, 440, 420), 512, 360, [])
    assert not window_would_overflow(P, 1024, 1024, (200, 300, 440, 420), 320, 360, [])
    with Lockstep(oracle, config(1), rng_mode=_lib.RNG_CALLER) as ls:
        install_cells(ls.gpu, ls.osl, 0, img)
        ls.set_poses([cell_pose(ls.cfg, 512, 360)])
        err = ls.update(Observation(0, angle=[], distance=[], valid=[]), STILL, np.zeros(2), 0.5)
        assert err is not None and err.code == _lib.E_WINDOW and ls.gpu.stats()["window_overflow"] == 1
        assert np.array_equal(ls.gpu.cells(0).reshape(1024, 1024), img)
    # the boundary itself: a square of exactly P fits, one cell more does not, an invalid beam counts as a valid one
    assert not window_would_overflow(P, 1024, 1024, (0, 0, 0, 0), 511, 500, [d121])
    assert window_would_overflow(P, 1024, 1024, (0, 0, 0, 0), 513, 500, [d121])
    assert window_would_overflow(P, 1024, 1024, (0, 0, 0, 0), 511, 500, [d122])
    assert window_would_overflow(P, 1024, 1024, (0, 0, 0, 0), 511, 500, [0.5, np.inf])
