"""TEST INFRASTRUCTURE ONLY -- ctypes binding of the pose-cluster oracle (oracle/libcluster_oracle.so) and the moments
of slamrs_gpu_pose_clusters from its labels, with correctly rounded sums (math.fsum).

cluster_oracle.c takes its bins from kld_oracle.c's so_kld_bin; kld_oracle.c links the localiser, recovery and SLAM
oracles, so the six files are compiled into a library of their own, with the flags of oracle/Makefile. Only tests/ and
tools/ import this module; the product package never does.
"""
from __future__ import annotations

import ctypes as C
import math
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libcluster_oracle.so")
_SOURCES = ("cluster_oracle.c", "kld_oracle.c", "recovery_oracle.c", "loc_oracle.c", "slam_oracle.c", "shared_stream.c")
_HEADERS = ("cluster_oracle.h", "kld_oracle.h", "recovery_oracle.h", "loc_oracle.h", "slam_oracle.h", "shared_stream.h")
# oracle/Makefile's CFLAGS: no contraction, no fast math
_CFLAGS = ["-O3", "-fno-fast-math", "-ffp-contract=off", "-fPIC", "-Wall", "-Wextra", "-Wno-unused-parameter", "-fopenmp"]
EXCLUDED = (1 << 64) - 1


def build(force: bool = False) -> str:
    """Compile libcluster_oracle.so with gcc if it is missing or older than its sources."""
    deps = [os.path.join(_HERE, f) for f in _SOURCES + _HEADERS + ("cluster_oracle.py",)]
    if force or not os.path.exists(_LIB_PATH) or any(os.path.getmtime(d) > os.path.getmtime(_LIB_PATH) for d in deps):
        tmp = _LIB_PATH + ".%d.tmp" % os.getpid()
        subprocess.run(["gcc"] + _CFLAGS + ["-shared", "-o", tmp] + [os.path.join(_HERE, s) for s in _SOURCES] + ["-lm"],
                       check=True, cwd=_HERE)
        os.replace(tmp, _LIB_PATH)
    return _LIB_PATH


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    build()
    L = C.CDLL(_LIB_PATH)
    f, u32, u64, vp = C.c_float, C.c_uint32, C.c_uint64, C.c_void_p
    L.so_pose_clusters.restype = C.c_int
    L.so_pose_clusters.argtypes = [vp, u64, f, f, f, u64, u64, u32, u32, vp, vp, vp, vp]
    L.so_kld_bin.restype = u64
    L.so_kld_bin.argtypes = [f, f, f, f, f, f, u64, u64, u32, u32]
    _lib = L
    return L


def _p(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


def clusters(xyt, position, resolution, grid_w, grid_h, bin_cells, theta_bins):
    """(labels[n] (EXCLUDED for an excluded pose), n_excluded, n_bins, n_clusters, [(label, count)] ranked by count
    descending, then label ascending) of the poses xyt[n, 3] (so_pose_clusters); position and resolution as f32."""
    a = np.ascontiguousarray(xyt, np.float32).reshape(-1, 3)
    n = a.shape[0]
    labels = np.zeros(max(n, 1), np.uint64); out3 = np.zeros(3, np.uint64)
    rl = np.zeros(max(n, 1), np.uint64); rc = np.zeros(max(n, 1), np.uint64)
    rc_ = lib().so_pose_clusters(_p(a), n, float(np.float32(position[0])), float(np.float32(position[1])),
                                 float(np.float32(resolution)), grid_w, grid_h, bin_cells, theta_bins, _p(labels), _p(out3),
                                 _p(rl), _p(rc))
    if rc_ != 0:
        raise MemoryError("oracle allocation failed")
    k = int(out3[2])
    return (labels[:n], int(out3[0]), int(out3[1]), k, [(int(rl[j]), int(rc[j])) for j in range(k)])


def kld_bin(x, y, theta, position, resolution, grid_w, grid_h, bin_cells, theta_bins) -> int:
    return int(lib().so_kld_bin(float(np.float32(x)), float(np.float32(y)), float(np.float32(theta)),
                                float(np.float32(position[0])), float(np.float32(position[1])), float(np.float32(resolution)),
                                grid_w, grid_h, bin_cells, theta_bins))


def moments(xyt, n_poses):
    """The record of one set of poses (rows of xyt[m, 3], f32) out of n_poses: count, weight = count / n_poses, mean
    (x, y, atan2(S, C)), the centred covariances and var_theta = -2 ln(sqrt(S^2 + C^2) / count), each sum correctly
    rounded (fsum) over the f64 terms. Also returns the sums' magnitudes the tests derive their bounds from."""
    a = np.asarray(xyt, np.float32).reshape(-1, 3).astype(np.float64)
    m = a.shape[0]
    zero = {"count": 0, "weight": 0.0, "mean": (0.0, 0.0, 0.0), "cov_xx": 0.0, "cov_xy": 0.0, "cov_yy": 0.0,
            "var_theta": 0.0}
    if m == 0:
        return zero, None
    xs, ys, ts = a[:, 0].tolist(), a[:, 1].tolist(), a[:, 2].tolist()
    sn = [math.sin(t) for t in ts]
    cs = [math.cos(t) for t in ts]
    mx, my = math.fsum(xs) / m, math.fsum(ys) / m
    S, Cc = math.fsum(sn), math.fsum(cs)
    dx = [x - mx for x in xs]
    dy = [y - my for y in ys]
    xx = [d * d for d in dx]
    xy = [u * v for u, v in zip(dx, dy)]
    yy = [d * d for d in dy]
    r = math.sqrt(S * S + Cc * Cc) / m
    rec = {"count": m, "weight": m / n_poses, "mean": (mx, my, math.atan2(S, Cc)), "cov_xx": math.fsum(xx) / m,
           "cov_xy": math.fsum(xy) / m, "cov_yy": math.fsum(yy) / m, "var_theta": -2.0 * math.log(r) if r > 0 else math.inf}
    mags = {"x": math.fsum(abs(v) for v in xs), "y": math.fsum(abs(v) for v in ys), "s": math.fsum(abs(v) for v in sn),
            "c": math.fsum(abs(v) for v in cs), "xx": math.fsum(xx), "xy": math.fsum(abs(v) for v in xy),
            "yy": math.fsum(yy), "dx": math.fsum(abs(v) for v in dx), "dy": math.fsum(abs(v) for v in dy), "S": S, "C": Cc}
    return rec, mags


def expected(xyt, position, resolution, grid_w, grid_h, bin_cells, theta_bins, k):
    """What slamrs_gpu_pose_clusters returns for the poses xyt: (stats, clusters[:min(k, n_clusters)], mags) with the
    integer outputs from so_pose_clusters and the moments from `moments`; mags[j] (j = 'overall' or an index) are the
    magnitudes for the bounds."""
    a = np.ascontiguousarray(xyt, np.float32).reshape(-1, 3)
    n = a.shape[0]
    labels, n_excl, n_bins, n_clusters, ranked = clusters(a, position, resolution, grid_w, grid_h, bin_cells, theta_bins)
    keep = labels != np.uint64(EXCLUDED)
    overall, mo = moments(a[keep], n)
    stats = {"n_poses": n, "n_excluded": n_excl, "n_bins": n_bins, "n_clusters": n_clusters, "overall": overall}
    out, mags = [], {"overall": mo}
    for j, (label, count) in enumerate(ranked[:k]):
        rec, mg = moments(a[labels == np.uint64(label)], n)
        assert rec["count"] == count
        rec["label"] = label
        out.append(rec)
        mags[j] = mg
    return stats, out, mags
