"""CPU checks of two rules the round-2 kernels rely on (no GPU):

* k_resample_indices decides from the FIRST selector of a source alone whether a new particle of another rank
  selects it (that rank pulls the grid; the item is listed first and the ray update signals its completion):
  either the first selector belongs to another rank, or the run of selectors crosses the end of the owner's
  range (kernels_resample.cu, `remote`).
* ray_walk_packed skips the free test for the first K cells of a walk: the cell reached after k steps of the
  reference's ray iterator (ray.rs:83-110) satisfies acc <= (k + 0.5)^2 + 0.25, whatever the direction."""
import numpy as np
import pytest

from oracle import oracle as O


def _remote_by_first_selector(idx, first, n_local):
    """The kernel's rule, for every source of rank [first, first + n_local) that some new particle selects."""
    n = len(idx)
    end = first + n_local
    out = {}
    for m in range(n):
        src = int(idx[m])
        if not (first <= src < end):
            continue
        if m > 0 and idx[m - 1] == src:
            continue                                  # not the first selector
        remote = not (first <= m < end)
        if not remote and end < n:
            remote = int(idx[end]) == src             # the run reaches past the end of this rank's range
        out[src] = remote
    return out


@pytest.mark.parametrize("world", [2, 3, 4, 8])
def test_first_selector_knows_whether_another_rank_selects_the_source(world):
    rng = np.random.default_rng(7 + world)
    for trial in range(200):
        n_local = int(rng.integers(1, 40))
        n = n_local * world
        # systematic resampling yields a non-decreasing index vector; weights of very different shapes
        w = rng.random(n) ** int(rng.integers(1, 12))
        if trial % 5 == 0:
            w[rng.integers(0, n)] += 50.0             # one dominant particle: a run across several ranks
        cum = np.cumsum(w / w.sum())
        u = (rng.random() + np.arange(n)) / n
        idx = np.minimum(np.searchsorted(cum, u, side="left"), n - 1)
        assert np.all(np.diff(idx) >= 0)
        for r in range(world):
            first = r * n_local
            got = _remote_by_first_selector(idx, first, n_local)
            for src in range(first, first + n_local):
                sel = np.nonzero(idx == src)[0]
                if len(sel) == 0:
                    assert src not in got
                    continue
                want = bool(np.any((sel < first) | (sel >= first + n_local)))
                assert got[src] == want, (trial, r, src)


def test_cells_reached_after_k_steps_are_within_the_manhattan_bound():
    """acc of the k-th visited cell (f32, as apply_measurement computes it, map.rs:98-100) <= (k + 0.5)^2 + 0.25."""
    rng = np.random.default_rng(3)
    F = np.float32
    w = h = 600
    for _ in range(400):
        sx, sy = F(300 + rng.random()), F(300 + rng.random())
        ang = rng.uniform(-np.pi, np.pi)
        if rng.random() < 0.2:
            ang = rng.choice([0.0, np.pi / 2, np.pi, -np.pi / 2, np.pi / 4]) + rng.choice([0.0, 1e-7, -1e-7])
        length = rng.uniform(0.0, 250.0)
        x1, y1 = F(sx + F(length * np.cos(ang))), F(sy + F(length * np.sin(ang)))
        cells = O.ray_cells(float(sx), float(sy), float(x1), float(y1), w, h)
        for k, (cx, cy) in enumerate(cells):
            dx = F(sx - F(F(cx) + F(0.5)))
            dy = F(sy - F(F(cy) + F(0.5)))
            acc = F(F(dx * dx) + F(dy * dy))
            assert float(acc) <= (k + 0.5) ** 2 + 0.25 + 1e-3 * (k + 1), (k, cx, cy, float(acc))
            # and the Manhattan distance to the start cell is exactly k
            assert abs(int(cx) - 300) + abs(int(cy) - 300) == k
