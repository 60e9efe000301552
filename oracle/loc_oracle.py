"""TEST INFRASTRUCTURE ONLY -- ctypes binding of the localiser's CPU oracle (oracle/libloc_oracle.so).

loc_oracle.c uses the SLAM oracle's motion model and resampling fold (slam_oracle.c, shared_stream.c); the three
files are compiled into a library of their own, with the flags of oracle/Makefile. Only tests/ and
tools/bench_localize.py's CPU reference point import this module; the product package never does.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libloc_oracle.so")
_SOURCES = ("loc_oracle.c", "slam_oracle.c", "shared_stream.c")
_HEADERS = ("loc_oracle.h", "slam_oracle.h", "shared_stream.h")
# oracle/Makefile's CFLAGS: no contraction, no fast math (rustc never contracts a*b+c)
_CFLAGS = ["-O3", "-fno-fast-math", "-ffp-contract=off", "-fPIC", "-Wall", "-Wextra", "-Wno-unused-parameter", "-fopenmp"]


def build(force: bool = False) -> str:
    """Compile libloc_oracle.so with gcc if it is missing or older than its sources."""
    deps = [os.path.join(_HERE, f) for f in _SOURCES + _HEADERS + ("loc_oracle.py",)]
    if force or not os.path.exists(_LIB_PATH) or any(os.path.getmtime(d) > os.path.getmtime(_LIB_PATH) for d in deps):
        tmp = _LIB_PATH + ".%d.tmp" % os.getpid()
        subprocess.run(["gcc"] + _CFLAGS + ["-shared", "-o", tmp] + [os.path.join(_HERE, s) for s in _SOURCES] + ["-lm"],
                       check=True, cwd=_HERE)
        os.replace(tmp, _LIB_PATH)
    return _LIB_PATH


class _Pose(C.Structure):
    _fields_ = [("x", C.c_float), ("y", C.c_float), ("theta", C.c_float)]


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    build()
    L = C.CDLL(_LIB_PATH)
    d, f, u64, i64, vp = C.c_double, C.c_float, C.c_uint64, C.c_int64, C.c_void_p
    L.so_loc_distance2.restype = i64; L.so_loc_distance2.argtypes = [vp, u64, u64, d, vp]
    L.so_loc_create.restype = vp; L.so_loc_create.argtypes = [f, f, f, u64, u64, u64, C.c_int, f, f, f, vp]
    L.so_loc_destroy.restype = None; L.so_loc_destroy.argtypes = [vp]
    L.so_loc_terms.restype = None; L.so_loc_terms.argtypes = [vp, vp]
    L.so_loc_outside.restype = d; L.so_loc_outside.argtypes = [vp]
    L.so_loc_set_adaptive_resampling.restype = None; L.so_loc_set_adaptive_resampling.argtypes = [vp, d]
    L.so_loc_resampled.restype = C.c_int; L.so_loc_resampled.argtypes = [vp]
    L.so_loc_set_weight_override.restype = None; L.so_loc_set_weight_override.argtypes = [vp, vp]
    L.so_loc_get_own_raw.restype = None; L.so_loc_get_own_raw.argtypes = [vp, vp]
    L.so_loc_update.restype = C.c_int; L.so_loc_update.argtypes = [vp, vp, vp, vp, u64, f, f, f, vp, d]
    L.so_loc_get_poses.restype = None; L.so_loc_get_poses.argtypes = [vp, vp]
    L.so_loc_set_poses.restype = None; L.so_loc_set_poses.argtypes = [vp, vp]
    L.so_loc_get_weights.restype = None; L.so_loc_get_weights.argtypes = [vp, vp, vp]
    L.so_loc_get_indices.restype = None; L.so_loc_get_indices.argtypes = [vp, vp]
    L.so_loc_max_particle.restype = u64; L.so_loc_max_particle.argtypes = [vp]
    L.so_loc_estimated_pose.restype = _Pose; L.so_loc_estimated_pose.argtypes = [vp]
    L.so_loc_effective_particles.restype = d; L.so_loc_effective_particles.argtypes = [vp]
    _lib = L
    return L


def _p(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


def distance2(prob, grid_w: int, grid_h: int, occupied_above: float):
    """Exact squared distance in cells to the nearest cell with p > occupied_above, exhaustive search (loc_oracle.c);
    (d2 as int64, -1 everywhere without obstacles; number of obstacle cells)."""
    m = np.ascontiguousarray(prob, np.float64).reshape(-1)
    assert m.size == grid_w * grid_h
    out = np.zeros(m.size, np.int64)
    k = lib().so_loc_distance2(_p(m), grid_w, grid_h, float(occupied_above), _p(out))
    return out, int(k)


class OracleLocalizer:
    """The localiser step (slamrs_gpu_create_localizer) restated on the CPU with externalised draws.
    kind 0 = beam endpoint, 1 = likelihood field (as slamrs_sensor_kind)."""

    def __init__(self, position, resolution, grid_w, grid_h, n_particles, prob, kind=0, sigma=0.1, z_rand=0.05,
                 occupied_above=0.5):
        m = np.ascontiguousarray(prob, np.float64).reshape(-1)
        assert m.size == grid_w * grid_h
        self._override = None
        self._h = lib().so_loc_create(position[0], position[1], resolution, grid_w, grid_h, n_particles, int(kind), sigma,
                                      z_rand, occupied_above, _p(m))
        if not self._h:
            raise MemoryError("oracle allocation failed")
        self.n, self.gw, self.gh = int(n_particles), int(grid_w), int(grid_h)

    def close(self):
        if self._h:
            lib().so_loc_destroy(self._h)
            self._h = None

    def __del__(self):
        self.close()

    def terms(self):
        o = np.zeros(self.gw * self.gh, np.float64); lib().so_loc_terms(self._h, _p(o)); return o

    @property
    def outside(self): return float(lib().so_loc_outside(self._h))

    def set_adaptive_resampling(self, tau): lib().so_loc_set_adaptive_resampling(self._h, float(tau))
    def resampled(self): return bool(lib().so_loc_resampled(self._h))

    def set_weight_override(self, raw):
        """The next update resamples on these raw weights (see so_set_weight_override in slam_oracle.c)."""
        self._override = np.ascontiguousarray(raw, np.float64).copy()
        assert self._override.size == self.n
        lib().so_loc_set_weight_override(self._h, _p(self._override))

    def own_raw_weights(self):
        out = np.zeros(self.n, np.float64); lib().so_loc_get_own_raw(self._h, _p(out)); return out

    def update(self, angle, dist, valid, dl, dr, wheel, z, u01) -> int:
        angle = np.ascontiguousarray(angle, np.float64); dist = np.ascontiguousarray(dist, np.float64)
        valid = np.ascontiguousarray(valid, np.uint8); z = np.ascontiguousarray(z, np.float64)
        assert z.size == 2 * self.n and angle.size == dist.size == valid.size
        return lib().so_loc_update(self._h, _p(angle), _p(dist), _p(valid), angle.size, dl, dr, wheel, _p(z), u01)

    def poses(self):
        out = np.zeros((self.n, 3), np.float32); lib().so_loc_get_poses(self._h, _p(out)); return out

    def set_poses(self, xyt):
        a = np.ascontiguousarray(xyt, np.float32).reshape(self.n, 3); lib().so_loc_set_poses(self._h, _p(a))

    def weights(self):
        w = np.zeros(self.n, np.float64); r = np.zeros(self.n, np.float64)
        lib().so_loc_get_weights(self._h, _p(w), _p(r)); return w, r

    def indices(self):
        i = np.zeros(self.n, np.uint64); lib().so_loc_get_indices(self._h, _p(i)); return i

    @property
    def max_particle(self): return int(lib().so_loc_max_particle(self._h))

    def estimated_pose(self):
        r = lib().so_loc_estimated_pose(self._h); return np.array([r.x, r.y, r.theta], np.float32)

    def number_of_effective_particles(self): return float(lib().so_loc_effective_particles(self._h))
