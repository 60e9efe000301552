"""CPU-side checks of the localiser's pose clusters (slamrs_gpu_pose_clusters): the cluster oracle's components against
scipy.ndimage.label on the dense bin occupancy (3 x 3 x 3, labels merged across the heading seam), its bins against
so_kld_bin, its moments against a numpy restatement, the Clustering dataclass, the argument checks on a NULL handle and
the -sys declarations."""
import ctypes as C
import math
import os
import re

import numpy as np
import pytest
import scipy.ndimage as ndi

from oracle import cluster_oracle as CO
from oracle import kld_oracle as KO
from slamrs_b200 import Clustering, _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
POS, RES = (-2.0, -1.0), 0.02


def _scipy_labels(xyt, gw, bc, tb):
    """Per pose: the smallest bin id of its component of the dense occupancy under scipy's 3 x 3 x 3 labelling, with
    the components that touch across the heading seam (heading bins tb - 1 and 0) merged; None when excluded."""
    nb = -(-gw // bc)
    off = nb * nb * tb
    bins = []
    for x, y, t in np.asarray(xyt, np.float32).tolist():
        b = KO.kld_bin(x, y, t, POS, RES, gw, gw, bc, tb) if all(map(math.isfinite, (x, y, t))) else off
        bins.append(None if b == off else b)
    occ = np.zeros((nb, nb, tb), bool)
    for b in bins:
        if b is not None:
            occ[(b // tb) // nb, (b // tb) % nb, b % tb] = True
    lab, n = ndi.label(occ, structure=np.ones((3, 3, 3), bool))
    parent = list(range(n + 1))

    def find(a):
        while parent[a] != a:
            a = parent[a]
        return a
    if tb >= 3:   # (tb <= 2: headings 0 and tb - 1 are already neighbours)
        for by, bx in zip(*np.nonzero(occ[:, :, 0])):
            for dy in (-1, 0, 1):
                for dx in (-1, 0, 1):
                    y2, x2 = by + dy, bx + dx
                    if 0 <= y2 < nb and 0 <= x2 < nb and occ[y2, x2, tb - 1]:
                        a, c = find(lab[by, bx, 0]), find(lab[y2, x2, tb - 1])
                        parent[max(a, c)] = min(a, c)
    smallest = {}
    for by, bx, h in zip(*np.nonzero(occ)):
        r = find(lab[by, bx, h])
        smallest[r] = min(smallest.get(r, 1 << 62), int((by * nb + bx) * tb + h))
    out = []
    for b in bins:
        out.append(None if b is None else smallest[find(lab[(b // tb) // nb, (b // tb) % nb, b % tb])])
    return out, n


def _check_against_scipy(xyt, gw, bc, tb):
    labels, n_excl, n_bins, n_clusters, ranked = CO.clusters(xyt, POS, RES, gw, gw, bc, tb)
    want, _ = _scipy_labels(xyt, gw, bc, tb)
    got = [None if v == CO.EXCLUDED else int(v) for v in labels.tolist()]
    assert got == want
    assert n_excl == sum(v is None for v in want)
    assert n_clusters == len({v for v in want if v is not None}) == len(ranked)
    counts = {}
    for v in want:
        if v is not None:
            counts[v] = counts.get(v, 0) + 1
    assert ranked == sorted(counts.items(), key=lambda lc: (-lc[1], lc[0]))
    return n_bins, n_clusters


@pytest.mark.parametrize("gw,bc,tb", [(200, 25, 36), (200, 10, 1), (200, 10, 2), (101, 7, 5), (64, 1, 3600)])
def test_labels_equal_scipy_on_random_clouds(gw, bc, tb):
    rng = np.random.default_rng(gw * 31 + tb)
    for n, spread in ((300, 0.3), (2000, 1.0), (4000, 3.0)):
        centres = rng.uniform(POS[0], POS[0] + gw * RES, (5, 2))
        xy = centres[rng.integers(0, 5, n)] + rng.normal(0.0, spread, (n, 2))
        xyt = np.column_stack([xy[:, 0], xy[:, 1] + (POS[1] - POS[0]), rng.uniform(-7.0, 7.0, n)]).astype(np.float32)
        xyt[rng.integers(0, n, 10), rng.integers(0, 3, 10)] = np.float32("nan")
        _check_against_scipy(xyt, gw, bc, tb)


def _at(col, row, h, bc, tb):
    """A pose in the middle of bin column `col`, bin row `row`, heading bin h."""
    return [POS[0] + (col + 0.5) * bc * RES, POS[1] + (row + 0.5) * bc * RES, (h + 0.5) * 2.0 * math.pi / tb]


def test_hand_made_clouds():
    gw, bc, tb = 200, 10, 36
    # a diagonal chain across bin corners (bx, by and h all step by 1): one cluster
    chain = np.array([_at(i, i, i, bc, tb) for i in range(8)], np.float32)
    assert _check_against_scipy(chain, gw, bc, tb) == (8, 1)
    # the same chain with one bin skipped: two clusters
    gap = np.array([_at(i, i, i, bc, tb) for i in range(8) if i != 4], np.float32)
    assert _check_against_scipy(gap, gw, bc, tb) == (7, 2)
    # a blob at theta = +-pi and one at theta = 0 across the seam of heading bins 0 / tb - 1
    pi = float(np.float32(math.pi))
    blob = np.array([[0.0, 0.0, pi], [0.0, 0.0, -pi], [0.05, 0.0, 3.1], [0.05, 0.0, -3.1], [1.0, 1.0, 0.01],
                     [1.0, 1.0, -0.01]], np.float32)
    labels, _, n_bins, n_clusters, _ = CO.clusters(blob, POS, RES, gw, gw, bc, tb)
    assert n_clusters == 2 and n_bins == 4 and labels[4] == labels[5] and labels[0] == labels[1] == labels[3]
    _check_against_scipy(blob, gw, bc, tb)
    for tbs in (1, 2):   # every heading in one or two bins
        rng = np.random.default_rng(tbs)
        xyt = np.column_stack([rng.uniform(-1.0, 1.0, 500), rng.uniform(-0.5, 0.5, 500), rng.uniform(-4.0, 4.0, 500)])
        _check_against_scipy(xyt.astype(np.float32), gw, bc, tbs)
    # excluded poses: non-finite components and off the grid
    ex = np.array([[np.nan, 0, 0], [0, np.inf, 0], [0, 0, -np.inf], [-5.0, 0, 0], [0, 100.0, 0], [0, 0, 0]], np.float32)
    labels, n_excl, n_bins, n_clusters, ranked = CO.clusters(ex, POS, RES, gw, gw, bc, tb)
    assert n_excl == 5 and n_bins == 1 and n_clusters == 1 and ranked[0][1] == 1
    assert (labels[:5] == np.uint64(CO.EXCLUDED)).all()


def test_bins_are_so_kld_bin():
    rng = np.random.default_rng(11)
    gw, bc, tb = 200, 7, 13
    xyt = np.column_stack([rng.uniform(-2.5, 2.5, 3000), rng.uniform(-1.5, 3.5, 3000), rng.uniform(-9.0, 9.0, 3000)])
    xyt = xyt.astype(np.float32)
    labels, n_excl, n_bins, _, _ = CO.clusters(xyt, POS, RES, gw, gw, bc, tb)
    off = (-(-gw // bc)) ** 2 * tb
    bins = [KO.kld_bin(x, y, t, POS, RES, gw, gw, bc, tb) for x, y, t in xyt.tolist()]
    assert [CO.kld_bin(x, y, t, POS, RES, gw, gw, bc, tb) for x, y, t in xyt[:200].tolist()] == bins[:200]
    assert n_excl == sum(b == off for b in bins)
    assert n_bins == len({b for b in bins if b != off})
    assert all((lab == np.uint64(CO.EXCLUDED)) == (b == off) for lab, b in zip(labels, bins))
    assert all(lab == np.uint64(CO.EXCLUDED) or int(lab) <= b for lab, b in zip(labels, bins))   # the smallest bin


def test_moments_equal_numpy_restatement():
    rng = np.random.default_rng(4)
    gw, bc, tb, k = 200, 25, 36, 5
    n = 5000
    xy = rng.normal(0.0, 0.4, (n, 2)) + np.array([0.0, 1.0])   # (the grid: x in [-2, 2), y in [-1, 3))
    t = np.where(rng.random(n) < 0.5, rng.normal(math.pi, 0.2, n), rng.normal(0.5, 0.3, n))
    xyt = np.column_stack([xy, t]).astype(np.float32)
    xyt[:7, 0] = 50.0   # off the grid
    stats, out, _ = CO.expected(xyt, POS, RES, gw, gw, bc, tb, k)
    labels = CO.clusters(xyt, POS, RES, gw, gw, bc, tb)[0]
    sets = [("overall", labels != np.uint64(CO.EXCLUDED), stats["overall"])]
    sets += [(j, labels == np.uint64(rec["label"]), rec) for j, rec in enumerate(out)]
    assert stats["n_excluded"] == 7 and len(out) == min(k, stats["n_clusters"])
    for name, sel, rec in sets:
        a = xyt[sel].astype(np.float64)
        m = a.shape[0]
        mx, my = a[:, 0].mean(), a[:, 1].mean()
        S, Cc = np.sin(a[:, 2]).sum(), np.cos(a[:, 2]).sum()
        dx, dy = a[:, 0] - mx, a[:, 1] - my
        want = [m, m / n, mx, my, math.atan2(S, Cc), (dx * dx).mean(), (dx * dy).mean(), (dy * dy).mean(),
                -2.0 * math.log(math.hypot(S, Cc) / m)]
        got = [rec["count"], rec["weight"], *rec["mean"], rec["cov_xx"], rec["cov_xy"], rec["cov_yy"], rec["var_theta"]]
        assert np.allclose(got, want, rtol=1e-12, atol=1e-12), (name, got, want)


def test_clustering_dataclass_and_structs():
    assert (C.sizeof(_lib.Clustering), C.sizeof(_lib.PoseCluster), C.sizeof(_lib.PoseStats)) == (16, 80, 112)
    c = Clustering()
    assert (c.bin_xy, c.theta_bins, c.max_clusters) == (0.5, 36, 16)
    s = c.to_struct(0.05)
    assert (s.struct_size, s.bin_cells, s.theta_bins, s.max_clusters) == (16, 10, 36, 16)
    assert Clustering(bin_xy=0.001).bin_cells(0.05) == 1


def test_pose_clusters_rejects_a_null_handle():
    L = _lib.load()
    c = Clustering().to_struct(0.05)
    st = _lib.PoseStats()
    arr = (_lib.PoseCluster * 16)()
    assert L.slamrs_gpu_pose_clusters(None, C.byref(c), C.byref(st), arr) == _lib.E_INVALID_ARG
    assert L.slamrs_gpu_pose_clusters(None, None, None, None) == _lib.E_INVALID_ARG


def _c_fields(struct, text):
    body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (struct, struct), text, flags=re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = []
    for d in body.split(";"):
        if d.strip():
            names += [re.findall(r"(\w+)\s*(?:\[[^\]]*\])?$", v.strip())[0] for v in d.split(",")]
    return names


def test_sys_crate_declares_pose_clusters():
    header = open(os.path.join(ROOT, "include", "slamrs_gpu.h")).read()
    rust = open(os.path.join(ROOT, "rust", "slam-gpu-sys", "src", "lib.rs")).read()
    for struct, ct in (("slamrs_gpu_clustering", _lib.Clustering), ("slamrs_gpu_pose_cluster", _lib.PoseCluster),
                       ("slamrs_gpu_pose_stats", _lib.PoseStats)):
        fields = _c_fields(struct, header)
        assert [n for n, _ in ct._fields_] == fields, struct
        body = re.search(r"pub struct %s \{(.*?)\}" % struct, rust, flags=re.S).group(1)
        assert re.findall(r"pub (\w+):", body) == fields, struct
    name = "slamrs_gpu_pose_clusters"
    c = re.search(r"int %s\((.*?)\);" % name, header, flags=re.S).group(1)
    c = re.sub(r"/\*.*?\*/", "", c, flags=re.S)
    r = re.search(r"pub fn %s\((.*?)\)" % name, rust, flags=re.S).group(1)
    assert len([a for a in r.split(",") if a.strip()]) == len(c.split(",")) == 4
    assert name in _lib.EXPORTS
