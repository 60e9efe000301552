"""TEST INFRASTRUCTURE ONLY -- ctypes binding of the localiser's KLD-sampling oracle (oracle/libkld_oracle.so).

kld_oracle.c uses the localiser oracle's term table (loc_oracle.c), the recovery oracle's state update and draw
(recovery_oracle.c) and the SLAM oracle's motion (slam_oracle.c, shared_stream.c); the five files are compiled into a
library of their own, with the flags of oracle/Makefile. Only tests/ and tools/ import this module; the product package
never does.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libkld_oracle.so")
_SOURCES = ("kld_oracle.c", "recovery_oracle.c", "loc_oracle.c", "slam_oracle.c", "shared_stream.c")
_HEADERS = ("kld_oracle.h", "recovery_oracle.h", "loc_oracle.h", "slam_oracle.h", "shared_stream.h")
# oracle/Makefile's CFLAGS: no contraction, no fast math (rustc never contracts a*b+c)
_CFLAGS = ["-O3", "-fno-fast-math", "-ffp-contract=off", "-fPIC", "-Wall", "-Wextra", "-Wno-unused-parameter", "-fopenmp"]


def build(force: bool = False) -> str:
    """Compile libkld_oracle.so with gcc if it is missing or older than its sources."""
    deps = [os.path.join(_HERE, f) for f in _SOURCES + _HEADERS + ("kld_oracle.py",)]
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
    d, f, u32, u64, vp = C.c_double, C.c_float, C.c_uint32, C.c_uint64, C.c_void_p
    L.so_kld_bin.restype = u64; L.so_kld_bin.argtypes = [f, f, f, f, f, f, u64, u64, u32, u32]
    L.so_kld_count.restype = u64; L.so_kld_count.argtypes = [vp, u64, f, f, f, u64, u64, u32, u32]
    L.so_kld_bound.restype = u64; L.so_kld_bound.argtypes = [u64, u64, u64, d, d]
    L.so_resample_fold_m.restype = C.c_int; L.so_resample_fold_m.argtypes = [vp, u64, u64, d, vp, vp, vp]
    L.so_resample_fold.restype = C.c_int; L.so_resample_fold.argtypes = [vp, u64, d, vp, vp, vp, vp]
    L.so_kld_create.restype = vp; L.so_kld_create.argtypes = [f, f, f, u64, u64, u64, C.c_int, f, f, f, vp]
    L.so_kld_destroy.restype = None; L.so_kld_destroy.argtypes = [vp]
    L.so_kld_set_kld.restype = None; L.so_kld_set_kld.argtypes = [vp, C.c_int, u64, u64, d, d, u32, u32]
    L.so_kld_set_recovery.restype = None; L.so_kld_set_recovery.argtypes = [vp, d, d, u64]
    L.so_kld_set_weight_override.restype = None; L.so_kld_set_weight_override.argtypes = [vp, vp]
    L.so_kld_update.restype = C.c_int; L.so_kld_update.argtypes = [vp, vp, vp, vp, u64, f, f, f, vp, d]
    L.so_kld_population.restype = u64; L.so_kld_population.argtypes = [vp]
    L.so_kld_state.restype = None; L.so_kld_state.argtypes = [vp, vp]
    L.so_kld_recovery_state.restype = None; L.so_kld_recovery_state.argtypes = [vp, vp, vp]
    L.so_kld_get_poses.restype = None; L.so_kld_get_poses.argtypes = [vp, vp]
    L.so_kld_set_poses.restype = None; L.so_kld_set_poses.argtypes = [vp, vp]
    L.so_kld_get_weights.restype = None; L.so_kld_get_weights.argtypes = [vp, vp, vp]
    L.so_kld_get_own_raw.restype = None; L.so_kld_get_own_raw.argtypes = [vp, vp]
    L.so_kld_get_indices.restype = None; L.so_kld_get_indices.argtypes = [vp, vp]
    L.so_kld_max_particle.restype = u64; L.so_kld_max_particle.argtypes = [vp]
    L.so_kld_estimated_pose.restype = _Pose; L.so_kld_estimated_pose.argtypes = [vp]
    _lib = L
    return L


def _p(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


def kld_bin(x, y, theta, position, resolution, grid_w, grid_h, bin_cells, theta_bins) -> int:
    """The bin of one pose (so_kld_bin); position and resolution are taken as f32, as the config holds them."""
    return int(lib().so_kld_bin(float(np.float32(x)), float(np.float32(y)), float(np.float32(theta)),
                                float(np.float32(position[0])), float(np.float32(position[1])),
                                float(np.float32(resolution)), grid_w, grid_h, bin_cells, theta_bins))


def kld_count(xyt, position, resolution, grid_w, grid_h, bin_cells, theta_bins) -> int:
    """The number of distinct bins of the poses xyt[n, 3] (so_kld_count)."""
    a = np.ascontiguousarray(xyt, np.float32).reshape(-1, 3)
    return int(lib().so_kld_count(_p(a), a.shape[0], float(np.float32(position[0])), float(np.float32(position[1])),
                                  float(np.float32(resolution)), grid_w, grid_h, bin_cells, theta_bins))


def kld_bound(k: int, n_min: int, n_max: int, err: float, z: float) -> int:
    """AMCL's bound on the particle count for k occupied bins (so_kld_bound)."""
    return int(lib().so_kld_bound(int(k), int(n_min), int(n_max), float(err), float(z)))


def resample_fold_m(raw_weights, m: int, u01: float):
    """(norm, idx[m], max_particle, clamped): m systematic draws from the weights (so_resample_fold_m)."""
    raw = np.ascontiguousarray(raw_weights, np.float64)
    norm = np.zeros(raw.size, np.float64); idx = np.zeros(max(int(m), 1), np.uint64); mp = C.c_uint64(0)
    cl = lib().so_resample_fold_m(_p(raw), raw.size, int(m), float(u01), _p(norm), _p(idx), C.byref(mp))
    return norm, idx[:int(m)], int(mp.value), int(cl)


def resample_fold(raw_weights, u01: float):
    """(norm, idx, max_particle, clamped) of slam_oracle.c's so_resample_fold."""
    raw = np.ascontiguousarray(raw_weights, np.float64)
    norm = np.zeros(raw.size, np.float64); idx = np.zeros(raw.size, np.uint64); mp = C.c_uint64(0)
    cl = lib().so_resample_fold(_p(raw), raw.size, float(u01), _p(norm), None, _p(idx), C.byref(mp))
    return norm, idx, int(mp.value), int(cl)


class OracleKldLocalizer:
    """The localiser step with a variable population (capacity n_particles), KLD-sampling and recovery.
    kind 0 = beam endpoint, 1 = likelihood field (as slamrs_sensor_kind)."""

    def __init__(self, position, resolution, grid_w, grid_h, n_particles, prob, kind=0, sigma=0.1, z_rand=0.05,
                 occupied_above=0.5):
        m = np.ascontiguousarray(prob, np.float64).reshape(-1)
        assert m.size == grid_w * grid_h
        self._override = None
        self._h = lib().so_kld_create(position[0], position[1], resolution, grid_w, grid_h, n_particles, int(kind), sigma,
                                      z_rand, occupied_above, _p(m))
        if not self._h:
            raise MemoryError("oracle allocation failed")
        self.capacity = int(n_particles)
        self._n_weighted, self._m_drawn = self.capacity, self.capacity

    def close(self):
        if self._h:
            lib().so_kld_destroy(self._h)
            self._h = None

    def __del__(self):
        self.close()

    def set_kld(self, kld=None):
        """kld: (n_min, n_max, err, z, bin_cells, theta_bins), or None (off: the next update draws the capacity)."""
        if kld is None:
            lib().so_kld_set_kld(self._h, 0, 0, 0, 0.0, 0.0, 1, 1)
            return
        lib().so_kld_set_kld(self._h, 1, int(kld[0]), int(kld[1]), float(kld[2]), float(kld[3]), int(kld[4]), int(kld[5]))

    def set_recovery(self, alpha_slow, alpha_fast, seed):
        lib().so_kld_set_recovery(self._h, float(alpha_slow), float(alpha_fast), int(seed))

    @property
    def population(self) -> int:
        return int(lib().so_kld_population(self._h))

    def kld_state(self):
        out = np.zeros(3, np.uint64); lib().so_kld_state(self._h, _p(out)); return tuple(int(v) for v in out)

    def recovery_state(self):
        st = np.zeros(3, np.float64); k = np.zeros(1, np.uint64)
        lib().so_kld_recovery_state(self._h, _p(st), _p(k))
        return {"w_slow": float(st[0]), "w_fast": float(st[1]), "p_inject": float(st[2]), "injected": int(k[0])}

    def set_weight_override(self, raw):
        """The next update resamples on these N_t raw weights (the device's)."""
        self._override = np.ascontiguousarray(raw, np.float64).copy()
        assert self._override.size == self.population
        lib().so_kld_set_weight_override(self._h, _p(self._override))

    def update(self, angle, dist, valid, dl, dr, wheel, z, u01) -> int:
        angle = np.ascontiguousarray(angle, np.float64); dist = np.ascontiguousarray(dist, np.float64)
        valid = np.ascontiguousarray(valid, np.uint8); z = np.ascontiguousarray(z, np.float64)
        assert z.size >= 2 * self.population and angle.size == dist.size == valid.size
        self._n_weighted = self.population
        rc = lib().so_kld_update(self._h, _p(angle), _p(dist), _p(valid), angle.size, dl, dr, wheel, _p(z), u01)
        self._m_drawn = self.population
        return rc

    def own_raw_weights(self):
        out = np.zeros(self._n_weighted, np.float64); lib().so_kld_get_own_raw(self._h, _p(out)); return out

    def poses(self):
        out = np.zeros((self.population, 3), np.float32); lib().so_kld_get_poses(self._h, _p(out)); return out

    def set_poses(self, xyt):
        a = np.ascontiguousarray(xyt, np.float32).reshape(self.population, 3); lib().so_kld_set_poses(self._h, _p(a))

    def weights(self):
        w = np.zeros(self._n_weighted, np.float64); r = np.zeros(self._n_weighted, np.float64)
        lib().so_kld_get_weights(self._h, _p(w), _p(r)); return w, r

    def indices(self):
        i = np.zeros(self._m_drawn, np.uint64); lib().so_kld_get_indices(self._h, _p(i)); return i

    @property
    def max_particle(self): return int(lib().so_kld_max_particle(self._h))

    def estimated_pose(self):
        r = lib().so_kld_estimated_pose(self._h); return np.array([r.x, r.y, r.theta], np.float32)
