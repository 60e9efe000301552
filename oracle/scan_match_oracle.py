"""TEST INFRASTRUCTURE ONLY -- ctypes binding of the scan-matching oracle (oracle/libscan_match_oracle.so).

scan_match_oracle.c adds scan-matching pose refinement to the SLAM oracle (slam_oracle.c, which it includes) without
changing it; it is compiled into a library of its own, with the flags of oracle/Makefile. `ScanMatchOracle` is an
`OracleSlam` whose update() refines every sampled pose while a matcher is set. Only tests/ import this module; the
product package never does.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

from . import oracle as _oracle

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libscan_match_oracle.so")
_SOURCES = ("scan_match_oracle.c", "shared_stream.c")
_DEPS = _SOURCES + ("slam_oracle.c", "slam_oracle.h", "shared_stream.h", "scan_match_oracle.py")
# oracle/Makefile's CFLAGS: no contraction, no fast math (rustc never contracts a*b+c)
_CFLAGS = ["-O3", "-fno-fast-math", "-ffp-contract=off", "-fPIC", "-Wall", "-Wextra", "-Wno-unused-parameter", "-fopenmp"]


def build(force: bool = False) -> str:
    """Compile libscan_match_oracle.so with gcc if it is missing or older than its sources."""
    deps = [os.path.join(_HERE, f) for f in _DEPS]
    if force or not os.path.exists(_LIB_PATH) or any(os.path.getmtime(d) > os.path.getmtime(_LIB_PATH) for d in deps):
        tmp = _LIB_PATH + ".%d.tmp" % os.getpid()
        subprocess.run(["gcc"] + _CFLAGS + ["-shared", "-o", tmp] + [os.path.join(_HERE, s) for s in _SOURCES] + ["-lm"],
                       check=True, cwd=_HERE)
        os.replace(tmp, _LIB_PATH)
    return _LIB_PATH


class Params(C.Structure):
    """sm_params: the fields of slamrs_gpu_scan_match after struct_size."""
    _fields_ = [("radius", C.c_uint32), ("step_xy", C.c_float), ("step_theta", C.c_float), ("levels", C.c_uint32),
                ("max_moves", C.c_uint32)]


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    build()
    L = C.CDLL(_LIB_PATH)
    d, f, u64, vp = C.c_double, C.c_float, C.c_uint64, C.c_void_p
    P = C.POINTER(Params)
    L.sm_update.restype = C.c_int; L.sm_update.argtypes = [vp, vp, vp, vp, u64, f, f, f, vp, d, P, vp, vp]
    L.sm_match_score.restype = C.c_int64; L.sm_match_score.argtypes = [vp, u64, vp, vp, vp, u64, _oracle._Pose, P]
    L.sm_match_climb.restype = C.c_int
    L.sm_match_climb.argtypes = [vp, u64, vp, vp, vp, u64, _oracle._Pose, P, C.POINTER(_oracle._Pose), vp]
    L.sm_set_counts.restype = C.c_int; L.sm_set_counts.argtypes = [vp, u64, vp, vp]
    L.sm_check.restype = C.c_int; L.sm_check.argtypes = [vp, P]
    _lib = L
    return L


def _p(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


class ScanMatchOracle(_oracle.OracleSlam):
    """OracleSlam with scan-matching pose refinement (off until set_scan_match is called with settings)."""

    def __init__(self, *args, **kwargs):
        super().__init__(*args, **kwargs)
        self._params = None
        self._moves = np.zeros(self.n, np.uint32)
        self._scored = np.zeros(self.n, np.uint32)
        self._last = None   # the settings of the last update, None when it ran without the matcher

    def set_scan_match(self, radius=1, step_xy=0.1, step_theta=0.05, levels=4, max_moves=32):
        """Settings for the following updates; levels=0 turns the matcher off (the default)."""
        if levels == 0:
            self._params = None
            return
        p = Params(radius, step_xy, step_theta, levels, max_moves)
        if not lib().sm_check(self._h, C.byref(p)):
            raise ValueError("scan match settings out of range, or the oracle keeps no hit counters")
        self._params = p

    def update(self, angle, dist, valid, dl, dr, wheel, z, u01) -> int:
        if self._params is None:
            self._last = None
            return super().update(angle, dist, valid, dl, dr, wheel, z, u01)
        angle = np.ascontiguousarray(angle, np.float64); dist = np.ascontiguousarray(dist, np.float64)
        valid = np.ascontiguousarray(valid, np.uint8); z = np.ascontiguousarray(z, np.float64)
        assert z.size == 2 * self.n and angle.size == dist.size == valid.size
        rc = lib().sm_update(self._h, _p(angle), _p(dist), _p(valid), angle.size, dl, dr, wheel, _p(z), u01,
                             C.byref(self._params), _p(self._moves), _p(self._scored))
        if rc == -2:
            raise ValueError("scan match settings out of range, or the oracle keeps no hit counters")
        self._last = self._params
        return rc

    def scan_match_stats(self):
        """(particles that moved, total moves, poses scored, particles stopped at max_moves) of the last update."""
        if self._last is None:
            return (0, 0, 0, 0)
        m = self._moves.astype(np.int64)
        return (int(np.sum(m > 0)), int(m.sum()), int(self._scored.astype(np.int64).sum()),
                int(np.sum(m == self._last.max_moves)))

    @staticmethod
    def _scan(angle, dist, valid):
        return (np.ascontiguousarray(angle, np.float64), np.ascontiguousarray(dist, np.float64),
                np.ascontiguousarray(valid, np.uint8))

    def match_score(self, particle, angle, dist, valid, pose) -> int:
        """S(pose) on the particle's current grid with the set radius."""
        a, d, v = self._scan(angle, dist, valid)
        r = lib().sm_match_score(self._h, particle, _p(a), _p(d), _p(v), a.size,
                                 _oracle._Pose(*[float(x) for x in pose]), C.byref(self._params))
        assert r >= 0
        return int(r)

    def match_climb(self, particle, angle, dist, valid, pose):
        """(refined pose as f32[3], moves, poses scored) from `pose` on the particle's grid."""
        a, d, v = self._scan(angle, dist, valid)
        ms = np.zeros(2, np.uint32); out = _oracle._Pose()
        rc = lib().sm_match_climb(self._h, particle, _p(a), _p(d), _p(v), a.size, _oracle._Pose(*[float(x) for x in pose]),
                                  C.byref(self._params), C.byref(out), _p(ms))
        assert rc == 0
        return np.array([out.x, out.y, out.theta], np.float32), int(ms[0]), int(ms[1])

    def set_counts(self, particle, n_free, n_occ):
        """Hand-built grid: the particle's hit counters (flat, index row * grid_h + column) and matching log-odds."""
        a = np.ascontiguousarray(n_free, np.uint16).reshape(-1); b = np.ascontiguousarray(n_occ, np.uint16).reshape(-1)
        assert a.size == b.size == self.gw * self.gh
        assert lib().sm_set_counts(self._h, particle, _p(a), _p(b)) == 0
