"""TEST INFRASTRUCTURE ONLY -- ctypes binding of the localiser's recovery oracle (oracle/librecovery_oracle.so).

recovery_oracle.c wraps the localiser oracle (loc_oracle.c, which uses slam_oracle.c and shared_stream.c); the four
files are compiled into a library of their own, with the flags of oracle/Makefile. Only tests/ import this module;
the product package never does.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "librecovery_oracle.so")
_SOURCES = ("recovery_oracle.c", "loc_oracle.c", "slam_oracle.c", "shared_stream.c")
_HEADERS = ("recovery_oracle.h", "loc_oracle.h", "slam_oracle.h", "shared_stream.h")
# oracle/Makefile's CFLAGS: no contraction, no fast math (rustc never contracts a*b+c)
_CFLAGS = ["-O3", "-fno-fast-math", "-ffp-contract=off", "-fPIC", "-Wall", "-Wextra", "-Wno-unused-parameter", "-fopenmp"]


def build(force: bool = False) -> str:
    """Compile librecovery_oracle.so with gcc if it is missing or older than its sources."""
    deps = [os.path.join(_HERE, f) for f in _SOURCES + _HEADERS + ("recovery_oracle.py",)]
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
    L.ss_recovery_slot.restype = u32; L.ss_recovery_slot.argtypes = [d, u32]
    L.ss_fill_recovery_draws.restype = None
    L.ss_fill_recovery_draws.argtypes = [u64, u64, u64, u64, d, vp, u32, u64, d, d, d, vp, vp]
    L.so_recovery_update.restype = d; L.so_recovery_update.argtypes = [d, u64, d, d, vp, vp]
    L.so_rec_create.restype = vp; L.so_rec_create.argtypes = [f, f, f, u64, u64, u64, C.c_int, f, f, f, vp]
    L.so_rec_destroy.restype = None; L.so_rec_destroy.argtypes = [vp]
    L.so_rec_loc.restype = vp; L.so_rec_loc.argtypes = [vp]
    L.so_rec_free_cells.restype = u64; L.so_rec_free_cells.argtypes = [vp, vp]
    L.so_rec_set_recovery.restype = None; L.so_rec_set_recovery.argtypes = [vp, d, d, u64]
    L.so_rec_update.restype = C.c_int; L.so_rec_update.argtypes = [vp, vp, vp, vp, u64, f, f, f, vp, d]
    L.so_rec_state.restype = None; L.so_rec_state.argtypes = [vp, vp, vp]
    L.so_rec_estimated_pose.restype = _Pose; L.so_rec_estimated_pose.argtypes = [vp]
    # the wrapped localiser oracle's accessors (loc_oracle.c, compiled into this library)
    L.so_loc_set_weight_override.restype = None; L.so_loc_set_weight_override.argtypes = [vp, vp]
    L.so_loc_get_own_raw.restype = None; L.so_loc_get_own_raw.argtypes = [vp, vp]
    L.so_loc_get_poses.restype = None; L.so_loc_get_poses.argtypes = [vp, vp]
    L.so_loc_set_poses.restype = None; L.so_loc_set_poses.argtypes = [vp, vp]
    L.so_loc_get_weights.restype = None; L.so_loc_get_weights.argtypes = [vp, vp, vp]
    L.so_loc_get_indices.restype = None; L.so_loc_get_indices.argtypes = [vp, vp]
    L.so_loc_max_particle.restype = u64; L.so_loc_max_particle.argtypes = [vp]
    _lib = L
    return L


def _p(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


def recovery_slot(u_c: float, n_free: int) -> int:
    """The free-list entry that the cell uniform u_c selects: min(n_free - 1, (uint32)(u_c * n_free))."""
    return int(lib().ss_recovery_slot(float(u_c), int(n_free)))


def recovery_draws(seed: int, step: int, first: int, count: int, p: float, free_cells, grid_h: int, position, resolution):
    """The recovery draws of particles first..first+count-1 at `step` (ss_recovery_draw): (inject[count] bool,
    poses[count, 3] f32, zero where not injected). position and resolution are taken as f32, as the config holds them."""
    free = np.ascontiguousarray(free_cells, np.uint32)
    inject = np.zeros(count, np.uint8); out = np.zeros((count, 3), np.float32)
    px, py = (float(np.float32(v)) for v in position)
    lib().ss_fill_recovery_draws(seed, step, first, count, float(p), _p(free), free.size, grid_h, px, py,
                                 float(np.float32(resolution)), _p(inject), _p(out))
    return inject.astype(bool), out


def recovery_update(raw_sum: float, n: int, alpha_slow: float, alpha_fast: float, w_slow: float, w_fast: float):
    """One step of the recovery averages (so_recovery_update): (w_slow, w_fast, p)."""
    ws = np.array([w_slow], np.float64); wf = np.array([w_fast], np.float64)
    p = lib().so_recovery_update(float(raw_sum), int(n), float(alpha_slow), float(alpha_fast), _p(ws), _p(wf))
    return float(ws[0]), float(wf[0]), float(p)


class OracleRecoveryLocalizer:
    """The localiser oracle (loc_oracle.OracleLocalizer's step) with recovery behind its resampling.
    kind 0 = beam endpoint, 1 = likelihood field (as slamrs_sensor_kind)."""

    def __init__(self, position, resolution, grid_w, grid_h, n_particles, prob, kind=0, sigma=0.1, z_rand=0.05,
                 occupied_above=0.5):
        m = np.ascontiguousarray(prob, np.float64).reshape(-1)
        assert m.size == grid_w * grid_h
        self._override = None
        self._h = lib().so_rec_create(position[0], position[1], resolution, grid_w, grid_h, n_particles, int(kind), sigma,
                                      z_rand, occupied_above, _p(m))
        if not self._h:
            raise MemoryError("oracle allocation failed")
        self._loc = lib().so_rec_loc(self._h)
        self.n = int(n_particles)

    def close(self):
        if self._h:
            lib().so_rec_destroy(self._h)
            self._h = None

    def __del__(self):
        self.close()

    def free_cells(self):
        """Ascending indices (row * grid_h + column) of the map's cells with p < 0.5."""
        k = int(lib().so_rec_free_cells(self._h, None))
        out = np.zeros(max(k, 1), np.uint32); lib().so_rec_free_cells(self._h, _p(out)); return out[:k]

    def set_recovery(self, alpha_slow, alpha_fast, seed):
        """Recovery with the stream keyed by `seed` (alpha_fast = 0: off); resets the averages."""
        lib().so_rec_set_recovery(self._h, float(alpha_slow), float(alpha_fast), int(seed))

    def recovery_state(self):
        """{w_slow, w_fast, p_inject, injected} of the last update (all zero without recovery)."""
        st = np.zeros(3, np.float64); k = np.zeros(1, np.uint64)
        lib().so_rec_state(self._h, _p(st), _p(k))
        return {"w_slow": float(st[0]), "w_fast": float(st[1]), "p_inject": float(st[2]), "injected": int(k[0])}

    def set_weight_override(self, raw):
        """The next update resamples on these raw weights (see so_set_weight_override in slam_oracle.c)."""
        self._override = np.ascontiguousarray(raw, np.float64).copy()
        assert self._override.size == self.n
        lib().so_loc_set_weight_override(self._loc, _p(self._override))

    def own_raw_weights(self):
        out = np.zeros(self.n, np.float64); lib().so_loc_get_own_raw(self._loc, _p(out)); return out

    def update(self, angle, dist, valid, dl, dr, wheel, z, u01) -> int:
        angle = np.ascontiguousarray(angle, np.float64); dist = np.ascontiguousarray(dist, np.float64)
        valid = np.ascontiguousarray(valid, np.uint8); z = np.ascontiguousarray(z, np.float64)
        assert z.size == 2 * self.n and angle.size == dist.size == valid.size
        return lib().so_rec_update(self._h, _p(angle), _p(dist), _p(valid), angle.size, dl, dr, wheel, _p(z), u01)

    def poses(self):
        out = np.zeros((self.n, 3), np.float32); lib().so_loc_get_poses(self._loc, _p(out)); return out

    def set_poses(self, xyt):
        a = np.ascontiguousarray(xyt, np.float32).reshape(self.n, 3); lib().so_loc_set_poses(self._loc, _p(a))

    def weights(self):
        w = np.zeros(self.n, np.float64); r = np.zeros(self.n, np.float64)
        lib().so_loc_get_weights(self._loc, _p(w), _p(r)); return w, r

    def indices(self):
        i = np.zeros(self.n, np.uint64); lib().so_loc_get_indices(self._loc, _p(i)); return i

    @property
    def max_particle(self): return int(lib().so_loc_max_particle(self._loc))

    def estimated_pose(self):
        r = lib().so_rec_estimated_pose(self._h); return np.array([r.x, r.y, r.theta], np.float32)
