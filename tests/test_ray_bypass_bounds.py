"""CPU checks (no GPU) of the bound behind the fused ray update's parking lists (kernels_ray.cu, RAY_OCC_PER_RAY_MAX):
one valid ray emits at most 7 occupied cells (the proof is in kernels_ray.cu), so a work item parks at most 7 hits
per ray of its half. A lattice of start offsets, headings and short measured distances, walked with the reference's
iterator and sensor model, finds at most 5, and finds 5: the 4 per ray the lists were once sized from is too few.
The capacities are read from the kernel source."""
import os
import re

import numpy as np

from oracle import oracle as O

F = np.float32
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RAY_SRC = os.path.join(ROOT, "slamrs_b200", "csrc", "kernels_ray.cu")
PROVEN_PER_RAY = 7        # kernels_ray.cu: 5 cells meeting the line within 1.71 cells before the endpoint, + 2 after
LATTICE_MAX = 5           # what the searches below find
GRID = 512
START = 200               # start cell: every lattice ray stays inside the grid


def _kernel_constants():
    """Every `constexpr uint32_t NAME = EXPR;` of kernels_ray.cu, evaluated in order."""
    vals = {}
    for name, expr in re.findall(r"constexpr\s+uint32_t\s+(\w+)\s*=\s*([^;]+);", open(RAY_SRC).read()):
        expr = re.sub(r"\b(\d+)u\b", r"\1", expr)
        vals[name] = int(eval(expr, {"__builtins__": {}}, dict(vals)))   # noqa: S307 (the project's own source)
    return vals


def _occupied_per_ray(sx, sy, gx, gy, md, max_steps):
    """Occupied cells each ray emits: the reference's GridRayIterator (oracle ray_walk, 2 additional steps) and
    inverse sensor model (tolerance 2), restated in f32 numpy over many rays at once. Walks of more than
    `max_steps` cells are not allowed (the caller keeps distances short)."""
    dxa, dya = np.abs(gx - sx), np.abs(gy - sy)
    fx0, fy0 = np.floor(sx), np.floor(sy)
    x, y = fx0.astype(np.int64), fy0.astype(np.int64)
    one = F(1.0)
    inf = F(np.inf)
    with np.errstate(invalid="ignore", over="ignore"):
        xp = gx > sx
        x_inc = np.where(dxa == 0, 0, np.where(xp, 1, -1))
        n = 3 + np.where(dxa == 0, 0, np.where(xp, np.floor(gx).astype(np.int64) - x, x - np.floor(gx).astype(np.int64)))
        err = np.where(dxa == 0, inf, np.where(xp, ((fx0 + one) - sx) * dya, (sx - fx0) * dya)).astype(F)
        yp = gy > sy
        y_inc = np.where(dya == 0, 0, np.where(yp, 1, -1))
        n = n + np.where(dya == 0, 0, np.where(yp, np.floor(gy).astype(np.int64) - y, y - np.floor(gy).astype(np.int64)))
        err = np.where(dya == 0, err - inf, np.where(yp, err - ((fy0 + one) - sy) * dxa, err - (sy - fy0) * dxa)).astype(F)
    assert n.max() <= max_steps, int(n.max())
    lo, hi = (md - one).astype(F), (md + one).astype(F)
    count = np.zeros(sx.shape, np.int64)
    for k in range(int(n.max())):
        live = k < n
        dxx = (sx - (x.astype(F) + F(0.5))).astype(F)
        dyy = (sy - (y.astype(F) + F(0.5))).astype(F)
        d = np.sqrt((dxx * dxx + dyy * dyy).astype(F)).astype(F)
        count += live & ~(d < lo) & ~(d > hi)
        step_y = err > 0
        y = np.where(step_y, y + y_inc, y)
        x = np.where(step_y, x, x + x_inc)
        err = np.where(step_y, err - dxa, err + dya).astype(F)
    return count


def _oracle_occupied(sx, sy, gx, gy, md):
    n = 0
    for cx, cy in O.ray_cells(float(sx), float(sy), float(gx), float(gy), GRID, GRID):
        dx = F(sx - F(F(cx) + F(0.5)))
        dy = F(sy - F(F(cy) + F(0.5)))
        d = np.sqrt(F(F(dx * dx) + F(dy * dy)), dtype=F)
        n += O.inverse_sensor_model(float(d), float(md), True) == 2
    return n


def _rays(sx, sy, ang, md):
    """Endpoints in cell units the way the step computes them: start + f32(direction x distance)."""
    c, s = np.cos(ang).astype(F), np.sin(ang).astype(F)
    return (sx + (c * md).astype(F)).astype(F), (sy + (s * md).astype(F)).astype(F)


def _headings():
    """Every quarter degree, and around each axis and diagonal the nearest f32 headings on both sides."""
    base = np.arange(1440) * (2 * np.pi / 1440)
    near = []
    for k in range(8):
        a = k * np.pi / 4
        near += [a + e for e in (-1e-3, -1e-5, -1e-7, 1e-7, 1e-5, 1e-3)]
    return np.concatenate([base, np.array(near)])


def test_restatement_matches_the_oracle_walk():
    rng = np.random.default_rng(11)
    k = 3000
    sx = (START + rng.random(k)).astype(F)
    sy = (START + rng.random(k)).astype(F)
    ang = rng.uniform(-np.pi, np.pi, k)
    ang[:200] = rng.choice([0.0, np.pi / 2, np.pi, -np.pi / 2, np.pi / 4, -3 * np.pi / 4], 200)
    md = rng.uniform(0.0, 4.0, k).astype(F)
    gx, gy = _rays(sx, sy, ang, md)
    got = _occupied_per_ray(sx, sy, gx, gy, md, 16)
    want = np.array([_oracle_occupied(*v) for v in zip(sx, sy, gx, gy, md)])
    assert np.array_equal(got, want)
    assert want.max() >= 4


def test_the_recorded_ray_emits_five_occupied_cells():
    sx, sy, ang, md = F(200.8050537), F(200.9636688), 0.9457754, F(1.4466372)
    gx, gy = _rays(np.array([sx]), np.array([sy]), np.array([ang]), np.array([md]))
    assert _oracle_occupied(sx, sy, gx[0], gy[0], md) == 5


def test_short_rays_on_a_lattice():
    """Start offsets in 1/16 cell steps, 1,488 headings, distances 0.25 to 3.5 cells in 1/16 steps: 17.7 M rays."""
    off = np.arange(16, dtype=np.float64) / 16
    ang = _headings()
    dist = np.arange(4, 57) / 16
    best, worst_ray = 0, None
    for ox in off:
        oy, a, d = (v.reshape(-1) for v in np.meshgrid(off, ang, dist, indexing="ij"))
        sx = np.full(oy.shape, START + ox, F)
        sy = (START + oy).astype(F)
        md = d.astype(F)
        gx, gy = _rays(sx, sy, a, md)
        c = _occupied_per_ray(sx, sy, gx, gy, md, 16)
        i = int(np.argmax(c))
        if c[i] > best:
            best, worst_ray = int(c[i]), (float(sx[i]), float(sy[i]), float(a[i]), float(md[i]))
    assert best <= PROVEN_PER_RAY, worst_ray
    assert best == LATTICE_MAX, (best, worst_ray)
    sx, sy, a, md = (np.array([v], t) for v, t in zip(worst_ray, (F, F, np.float64, F)))
    gx, gy = _rays(sx, sy, a, md)
    assert _oracle_occupied(sx[0], sy[0], gx[0], gy[0], md[0]) == best   # (the restatement agrees on that ray)


def test_fine_start_offsets_near_the_worst_case():
    """1/64 cell start offsets at the distances and headings where five occupied cells occur."""
    off = np.arange(64, dtype=np.float64) / 64
    ang = np.arange(-40, 41) * (np.pi / 2 / 80) + np.pi / 4
    ang = np.concatenate([ang + q * np.pi / 2 for q in range(4)])
    dist = np.arange(16, 41) / 16
    best = 0
    for ox in off:
        oy, a, d = (v.reshape(-1) for v in np.meshgrid(off, ang, dist, indexing="ij"))
        sx = np.full(oy.shape, START + ox, F)
        sy = (START + oy).astype(F)
        md = d.astype(F)
        gx, gy = _rays(sx, sy, a, md)
        best = max(best, int(_occupied_per_ray(sx, sy, gx, gy, md, 16).max()))
    assert best <= LATTICE_MAX <= PROVEN_PER_RAY


def test_longer_rays_sampled():
    """Distances 3 to 150 cells (a 6 m lidar at 4 cm cells) through the oracle's own walk."""
    rng = np.random.default_rng(5)
    best = 0
    for _ in range(1500):
        sx, sy = F(START + rng.random()), F(START + rng.random())
        md = F(rng.uniform(3.0, 150.0))
        gx, gy = _rays(np.array([sx]), np.array([sy]), np.array([rng.uniform(-np.pi, np.pi)]), np.array([md]))
        best = max(best, _oracle_occupied(sx, sy, gx[0], gy[0], md))
    assert best <= PROVEN_PER_RAY


def test_parking_capacities_cover_the_bound():
    c = _kernel_constants()
    beams = c["RAY_PACKED_MAX_BEAMS"]
    assert beams == 2047
    assert c["RAY_OCC_PER_RAY_MAX"] >= PROVEN_PER_RAY
    # one work item: every ray of its half (<= all beams) parks at most the bound; a zero-length ray parks 3
    assert c["RAY_SPILL_CAP"] >= max(PROVEN_PER_RAY, 3) * beams
    # the lower half's start-row hits travel as 16-bit counts per cell: at most the bound times the lower half's rays
    src = open(RAY_SRC).read()
    struct = re.search(r"struct alignas\(16\) HalfXchg \{(.*?)\};", src, re.S).group(1)
    assert re.search(r"uint4 occ\[HALF_XCHG_GROUPS\];.*16 bits", struct)
    assert PROVEN_PER_RAY * beams <= 0xFFFF
    assert "HALF_XCHG_HITS" not in src   # (the fixed 60-entry list it replaces)


def test_zero_length_rays_park_three():
    """A ray whose endpoint is its start point emits the start cell 1 + 2 times (the bound's zero-length case)."""
    sx, sy = F(200.25), F(200.75)
    assert len(O.ray_cells(float(sx), float(sy), float(sx), float(sy), GRID, GRID)) == 3
