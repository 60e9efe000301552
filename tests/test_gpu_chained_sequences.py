"""The chained step sequence (one GPU, device-resident scan, fused ray update: k_plan publishes an epoch, the ray
update's last CTA acquires it and commits the step, the side stream is never joined) under everything a caller can
do between two steps: switch the scan source, cross the sort and fused-update bounds, toggle scan matching and
profiling, write grids and poses from the host, supply its own draws, read results back without a sync.

Every sequence runs on a default handle and on a SLAMRS_FLAG_SERIAL_STEPS handle (same seed, same calls), whose state
must agree bit for bit, and where the population allows against the oracle too. Which steps chained is read from the
launch counts: a chained step issues one launch fewer (no commit kernel) than the serial handle's same step, and
every test asserts the pattern of chained and serial steps it means to exercise."""
from __future__ import annotations

import dataclasses
import os
import time

import numpy as np
import pytest

from slamrs_b200 import GpuPlacement, GridMapSlam, GridMapSlamConfig, ScanMatcher, _lib
from slamrs_b200.simulator import Simulator, reference_scene
from slamrs_b200.workloads import WORKLOADS
from oracle import oracle as O
from oracle.scan_match_oracle import ScanMatchOracle

from common import SEED, WEIGHT_RTOL, at_scale_config, at_scale_scans, cloned_probes, compare_step, make_scans, oracle_step

pytestmark = pytest.mark.gpu

STEP_HISTORY = 256          # kernels.cuh: steps the device's history ring holds
DRAW_SEED = SEED ^ 0x00C0FFEE   # caller-supplied draws come from another stream than the handle's own


def small_cfg(n):
    """160^2 grid at 5 cm (tiled: the fused ray update applies) around the reference scene at scale 3."""
    return GridMapSlamConfig(position=(-4.0, -4.0), width=8.0, height=8.0, resolution=0.05, n_particles=n)


def small_sim(n_beams=180):
    return Simulator(reference_scene(3.0), n_beams=n_beams, scanner_range=3.0, wheel_base=0.1)


def _bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint8) if a.dtype.itemsize == 1 else a.view({2: np.uint16, 4: np.uint32, 8: np.uint64}[a.dtype.itemsize])


def _pose(g):
    p = g.estimated_pose()
    return np.array([p.x, p.y, p.theta], np.float32)


def _check_extent(g, full=None):
    """map_extent() (after a step: the box the step's commit left in the counters) holds every cell of the estimate's
    map that is not exactly 0.5."""
    m = (g.estimated_likelihood().data if full is None else full).reshape(g.grid_h, g.grid_w)
    x0, y0, x1, y1 = g.map_extent()
    ys, xs = np.nonzero(m != 0.5)
    if ys.size:
        assert x0 <= xs.min() and xs.max() < x1 and y0 <= ys.min() and ys.max() < y1, \
            ((x0, y0, x1, y1), (xs.min(), ys.min(), xs.max() + 1, ys.max() + 1))


class Sequence:
    """One default and one FLAG_SERIAL_STEPS handle (plus `extra` handles that must behave as the default one), all
    with the same seed, driven by the same calls; optionally the oracle in lockstep. chained[i]: step i took the
    chained sequence on the default handle."""

    def __init__(self, cfg, oracle=False, sparse=False, rng_mode=_lib.RNG_SHARED_STREAM, extra=0):
        pl = dict(seed=SEED, rng_mode=rng_mode)
        self.cfg, self.n, self.caller = cfg, cfg.n_particles, rng_mode == _lib.RNG_CALLER
        self.handles = [GridMapSlam(cfg, GpuPlacement(**pl)), GridMapSlam(cfg, GpuPlacement(flags=_lib.FLAG_SERIAL_STEPS, **pl))]
        self.handles += [GridMapSlam(cfg, GpuPlacement(**pl)) for _ in range(extra)]
        self.g, self.s = self.handles[0], self.handles[1]
        self.osl = None
        self.sparse = sparse
        if oracle:
            self.osl = ScanMatchOracle(cfg.position, cfg.width, cfg.height, cfg.resolution, cfg.n_particles, True, sparse=sparse)
            if sparse:
                self.osl.set_threads(os.cpu_count() or 1)
        self.chained = []
        self.step = 0
        self.in_flight = []   # device scans of the steps issued since the last sync

    def close(self):
        for h in self.handles:
            h.close()
        if self.osl is not None:
            self.osl.close()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # ---------------------------------------------------------------- steps
    def _draws(self):
        if not self.caller:
            return {}
        return dict(z_draws=O.motion_normals(DRAW_SEED, self.step, 0, self.n), resample_u=O.resample_uniform(DRAW_SEED, self.step))

    def _issue(self, fn):
        d = []
        for h in self.handles:
            l0 = h.launch_count
            fn(h)
            d.append(h.launch_count - l0)
        assert d[0] in (d[1], d[1] - 1) and all(x == d[0] for x in d[2:]), (self.step, d)
        self.chained.append(d[0] == d[1] - 1)

    @staticmethod
    def upload(scans):
        """Device copies (angle, distance, valid) of the scans' observations, uploaded ahead of the steps so that
        back-to-back steps are not separated by a device synchronisation."""
        import torch
        out = [tuple(torch.from_numpy(x).cuda() for x in (obs.angle.astype(np.float32), obs.distance.astype(np.float32),
                                                            obs.valid.astype(np.uint8))) for obs, _ in scans]
        torch.cuda.synchronize()
        return out

    def device(self, obs, odo, max_dist=None, check=True, dev=None):
        """set_scan_device + step_async on the scan in device memory (`dev`: from upload(), else uploaded here);
        `max_dist` None: the scan's own bound."""
        a, d, v = dev if dev is not None else self.upload([(obs, odo)])[0]
        self.in_flight.append((a, d, v))
        md = float(np.abs(obs.distance.astype(np.float32)).max(initial=0.0)) if max_dist is None else max_dist
        draws = self._draws()

        def fn(h):
            h.set_scan_device(a.data_ptr(), d.data_ptr(), v.data_ptr(), a.numel(), md)
            h.step_async(odo, **draws)
        self._issue(fn)
        self._after(obs, odo, check)

    def host(self, obs, odo, check=True):
        """The synchronous update() on a host scan."""
        draws = self._draws()
        self._issue(lambda h: h.update(obs, odo, **draws))
        self._after(obs, odo, check)

    def sim(self, segments, pose, n_beams, scanner_range, odo, check=True):
        """A scan the device simulates into the handle's own buffers (sim_scan), then step_async."""
        draws = self._draws()

        def fn(h):
            assert h.sim_scan(segments, pose, n_beams, scanner_range) > 0
            h.step_async(odo, **draws)
        self._issue(fn)
        obs = self.g.get_scan()
        other = self.s.get_scan()
        assert np.array_equal(_bits(obs.distance), _bits(other.distance)) and np.array_equal(obs.valid, other.valid)
        self._after(obs, odo, check)

    def _after(self, obs, odo, check):
        if self.osl is not None:
            self._oracle_step(obs, odo)
        self.step += 1
        if check:
            self.sync()
            self.compare()

    def sync(self):
        for h in self.handles:
            h.sync()
        self.in_flight = []

    # ---------------------------------------------------------------- oracle
    def _oracle_step(self, obs, odo):
        seed = DRAW_SEED if self.caller else SEED
        if not self.sparse:
            assert oracle_step(O, self.osl, obs, odo, self.step, seed)[0] == 0
            compare_step(self.g, self.osl)
            return
        # large populations: the oracle resamples on the device's raw weights once they have been checked against its
        # own (the device's exp/log differ from glibc's in the last bit; see lockstep_following_device_weights)
        g, osl = self.g, self.osl
        w_gpu, raw_gpu = g.weights()
        osl.set_weight_override(raw_gpu)
        assert oracle_step(O, osl, obs, odo, self.step, seed)[0] == 0
        own = osl.own_raw_weights()
        assert np.max(np.abs(own - raw_gpu) / np.maximum(np.abs(own), 1e-300)) < WEIGHT_RTOL, self.step
        w_ref, _ = osl.weights()
        assert np.array_equal(_bits(w_ref), _bits(w_gpu)), self.step
        idx_ref = osl.indices().astype(np.int64)
        assert np.array_equal(idx_ref, g.resample_indices().astype(np.int64)), self.step
        assert g.max_particle == osl.max_particle
        assert np.array_equal(_bits(osl.poses()), _bits(g.poses())), self.step
        assert np.array_equal(_bits(osl.estimated_pose()), _bits(_pose(g))), self.step
        assert np.max(np.abs(osl.estimated_likelihood() - g.estimated_likelihood().data)) < 1e-12, self.step
        for p in cloned_probes(self.n)(self.step, idx_ref):
            nf, no = osl.counts(p)
            gf, go = g.counts(p)
            assert np.array_equal(nf, gf) and np.array_equal(no, go), (self.step, p)

    # ---------------------------------------------------------------- default against serial, bit for bit
    def compare(self, particles=None, other=None):
        """Every read-out of the default handle against the serial one (or `other`); `particles` None: every
        particle's cells, read and compared one particle at a time."""
        a, b = self.g, other if other is not None else self.s
        where = self.step
        _check_extent(a)
        for x, y in zip(a.weights(), b.weights()):
            assert np.array_equal(_bits(x), _bits(y)), where
        assert np.array_equal(a.resample_indices(), b.resample_indices()), where
        assert np.array_equal(_bits(a.poses()), _bits(b.poses())), where
        assert a.max_particle == b.max_particle, where
        assert np.array_equal(_bits(_pose(a)), _bits(_pose(b))), where
        assert np.array_equal(_bits(a.estimated_likelihood().data), _bits(b.estimated_likelihood().data)), where
        assert a.stats() == b.stats(), where
        first = max(0, self.step - STEP_HISTORY)
        if self.step > first:
            assert np.array_equal(a.step_history(first, self.step - first), b.step_history(first, self.step - first)), where
        for x, y in zip(a.slots(), b.slots()):
            assert np.array_equal(x, y), where
        for p in (range(self.n) if particles is None else particles):
            assert np.array_equal(a.cells(p), b.cells(p)), (where, p)


# ------------------------------------------------------------------------------------------------ 1. launch shapes
@pytest.mark.parametrize("n", [1, 2, 3, 5])
def test_tiny_populations_tail_with_few_ctas(oracle, n):
    """n_local = 1..5: the ray update runs 2..10 CTAs, so its last CTA is found among very few."""
    with Sequence(small_cfg(n), oracle=True) as seq:
        for obs, odo in make_scans(3.0, 180, 3.0, 20):
            seq.device(obs, odo)
        assert all(seq.chained), seq.chained


@pytest.mark.parametrize("n", [600, 4096], ids=["items_just_above_ctas", "items_far_above_ctas"])
def test_work_items_above_resident_ctas_lockstep_sparse_oracle(oracle, n):
    """More work items than the 592 resident CTAs: the tail's last CTA leaves after two or more rounds."""
    stride = max(1, n // 24)
    scans = at_scale_scans(40)
    with Sequence(at_scale_config(n), oracle=True, sparse=True) as seq:
        for i, (obs, odo) in enumerate(scans):
            seq.device(obs, odo, check=False)
            seq.sync()
            seq.compare(particles=None if i == len(scans) - 1 else range(i % stride, n, stride))
        assert all(seq.chained), seq.chained


def test_configs2_chained_equals_serial_over_200_scans():
    wl = WORKLOADS["c3"]
    sim = wl.simulator()
    scans = [sim.next_scan(wl.speed_left, wl.speed_right) for _ in range(200)]
    n = wl.n_particles
    with Sequence(wl.slam_config(n)) as seq:
        dev = seq.upload(scans)
        for lo, hi in ((0, 60), (60, 130), (130, 200)):
            for (obs, odo), d in zip(scans[lo:hi], dev[lo:hi]):
                seq.device(obs, odo, check=False, dev=d)
            seq.sync()
            seq.compare(particles=None if hi == 200 else range(hi % 97, n, 97))
        assert all(seq.chained), seq.chained


# ------------------------------------------------------------------------------------------------ 2. scan sources
def test_scan_source_switches(oracle):
    """Device scans (chained) alternating with host-scan update() steps (serial), every other step and in runs of
    five, and device-simulated scans (serial)."""
    sim = small_sim()
    pattern = "DHDHDHDH" + "DDDDDHHHHH" + "DDDDDHHHHH" + "SDSDDSSD"
    with Sequence(small_cfg(32), oracle=True) as seq:
        for kind in pattern:
            obs, odo = sim.next_scan(0.08, 0.10)
            if kind == "D":
                seq.device(obs, odo)
            elif kind == "H":
                seq.host(obs, odo)
            else:
                seq.sim(sim.segments, np.array(sim.pose, np.float32), sim.n_beams, float(sim.scanner_range), odo)
        assert seq.chained == [k == "D" for k in pattern], seq.chained


def test_host_scan_update_never_chains():
    """The synchronous update() uploads a host scan, so it never takes the chained sequence (whose tail leaves no
    host counter mirror); neither does step_async behind upload_scan."""
    with Sequence(at_scale_config(600)) as seq:
        scans = at_scale_scans(6)
        for obs, odo in scans[:3]:
            seq.host(obs, odo, check=False)
        for obs, odo in scans[3:5]:
            def fn(h, obs=obs, odo=odo):
                h.upload_scan(obs)
                h.step_async(odo)
            seq._issue(fn)
            seq.step += 1
        seq.device(*scans[5])
        assert seq.chained == [False] * 5 + [True], seq.chained


# ------------------------------------------------------------------------------------------------ 3. path switches
def test_beam_count_and_max_dist_switches(oracle):
    """360 -> 2,047 (the fused bound) -> 2,048 -> 2,049 (32-bit generic kernel, serial; 2,049: no beam sort) -> 32
    (no sort) -> 33 (sorted) -> 360, then one step with max_dist = +inf (unfused update, serial) and one without."""
    beams = [360, 2047, 2048, 2049, 32, 33, 360, 360, 360]
    sim = small_sim()
    with Sequence(small_cfg(24), oracle=True) as seq:
        for i, nb in enumerate(beams):
            sim.n_beams = nb
            obs, odo = sim.next_scan(0.08, 0.10)
            assert len(obs) == nb
            seq.device(obs, odo, max_dist=float("inf") if i == 7 else None)
        assert seq.chained == [True, True, False, False, True, True, True, False, True], seq.chained


# ------------------------------------------------------------------------------------------------ 4. scan matching
def test_scan_matching_toggled_between_chained_steps(oracle):
    on = {3, 4, 7, 10, 11, 12}
    with Sequence(small_cfg(16), oracle=True) as seq:
        for step, (obs, odo) in enumerate(make_scans(3.0, 180, 3.0, 15)):
            m = ScanMatcher() if step in on else None
            for h in seq.handles:
                h.set_scan_matcher(m)
            if m is None:
                seq.osl.set_scan_match(levels=0)
            else:
                seq.osl.set_scan_match(**dataclasses.asdict(m))
            seq.device(obs, odo)
            st = seq.g.scan_match_stats()
            assert st == seq.s.scan_match_stats()
            assert tuple(st[k] for k in ("moved", "moves", "scored", "capped")) == seq.osl.scan_match_stats(), step
        assert seq.chained == [s not in on for s in range(15)], seq.chained


# ------------------------------------------------------------------------------------------------ 5. host writes
def test_host_writes_between_chained_steps(oracle):
    """set_cells (every clone made private first), set_poses and init_uniform between chained steps."""
    n = 24
    cfg = small_cfg(n)
    box = (-0.4, -0.3, 0.4, 0.3)
    with Sequence(cfg, oracle=True) as seq:
        for step, (obs, odo) in enumerate(make_scans(3.0, 180, 3.0, 20)):
            if step == 5:
                for p, src in ((n - 1, 0), (3, n // 2)):
                    img = np.roll(seq.g.cells(src).reshape(seq.g.grid_h, seq.g.grid_w), 7, axis=0).reshape(-1)
                    for h in seq.handles:
                        h.set_cells(p, img)
                    seq.osl.set_counts(p, (img & 0xFFFF).astype(np.uint16), (img >> 16).astype(np.uint16))
                assert seq.g.map_extent() == seq.s.map_extent()
            elif step == 10:
                xyt = seq.g.poses()[::-1].copy()
                xyt[:, 2] += np.float32(0.25)
                for h in seq.handles:
                    h.set_poses(xyt)
                seq.osl.set_poses(xyt)
            elif step == 15:
                for h in seq.handles:
                    h.init_uniform(box)
                seq.osl.set_poses(O.uniform_poses(SEED, 0, n, np.float32(box).astype(np.float64)))
            seq.device(obs, odo)
        assert all(seq.chained), seq.chained


# ------------------------------------------------------------------------------------------------ 6. caller draws
def test_caller_draws_in_chained_mode(oracle):
    with Sequence(small_cfg(32), oracle=True, rng_mode=_lib.RNG_CALLER) as seq:
        scans = make_scans(3.0, 180, 3.0, 16)
        for step, (obs, odo) in enumerate(scans):
            if step in (6, 7, 12):
                seq.host(obs, odo)
            else:
                seq.device(obs, odo)
        assert seq.chained == [s not in (6, 7, 12) for s in range(16)], seq.chained


# ------------------------------------------------------------------------------------------------ 7. read-outs
def _same(x, y):
    if isinstance(x, np.ndarray):
        return np.array_equal(x, y)
    if isinstance(x, (list, tuple)):
        return len(x) == len(y) and all(_same(a, b) for a, b in zip(x, y))
    return x == y


def _readouts(g, step, particles):
    """Every read-out of one handle; the order rotates with the step, so that each one is, at some step, the first
    call behind the step_async."""
    calls = [("pose", lambda: _bits(_pose(g))), ("stats", g.stats), ("weights", lambda: [_bits(w) for w in g.weights()]),
             ("n_eff", lambda: np.float64(g.number_of_effective_particles()).view(np.uint64)),
             ("map", lambda: _bits(g.estimated_likelihood().data)), ("extent", g.map_extent),
             ("history", lambda: g.step_history(step, 1))]
    calls += [(f"window{fmt}", lambda fmt=fmt: g.estimated_likelihood_window(fmt=fmt)) for fmt in (_lib.MAP_F64, _lib.MAP_F32, _lib.MAP_U8)]
    calls += [(f"extents{p}", lambda p=p: g.extents(p)) for p in particles]
    k = step % len(calls)
    out = {name: fn() for name, fn in calls[k:] + calls[:k]}
    for fmt in (_lib.MAP_F64, _lib.MAP_F32, _lib.MAP_U8):
        box, win = out[f"window{fmt}"]
        assert box == out["extent"], (step, fmt)
        out[f"window{fmt}"] = _bits(win).copy()
    return out


def test_read_outs_right_behind_chained_steps():
    """Each read-out issued straight behind a step_async, no sync() in between; the pipelined map copy is left in
    flight across the next step_async, as a caller overlapping export and step does."""
    import torch
    n = 600
    cfg = at_scale_config(n)
    particles = (0, 1, n // 2, n - 1)
    with Sequence(cfg) as seq:
        bufs = [torch.empty(seq.g.grid_w * seq.g.grid_h, dtype=torch.float64, pin_memory=True).numpy() for _ in seq.handles]
        pending = None
        scans = at_scale_scans(30)
        for (obs, odo), d in zip(scans, seq.upload(scans)):
            step = seq.step
            seq.device(obs, odo, check=False, dev=d)
            got = [_readouts(h, step, particles) for h in seq.handles]
            for k in got[0]:
                assert _same(got[0][k], got[1][k]), (step, k)
            x0, y0, x1, y1 = got[0]["extent"]
            full = got[0]["map"].view(np.float64).reshape(seq.g.grid_h, seq.g.grid_w)
            assert np.array_equal(_bits(full[y0:y1, x0:x1]), got[0][f"window{_lib.MAP_F64}"]), step
            _check_extent(seq.g, full.reshape(-1))
            if pending is not None:   # the previous step's copy, waited for only now
                for h, buf in zip(seq.handles, bufs):
                    h.map_wait()
                    assert np.array_equal(_bits(buf), pending), step
            for h, buf in zip(seq.handles, bufs):
                h.estimated_likelihood_async(buf)
            pending = got[0]["map"].copy()
        for h, buf in zip(seq.handles, bufs):
            h.map_wait()
            assert np.array_equal(_bits(buf), pending)
        seq.sync()
        seq.compare()
        assert all(seq.chained), seq.chained


# ------------------------------------------------------------------------------------------------ 8. profiling
def test_profiling_across_the_ring():
    """150 profiled steps in runs of chained (device scan) and serial (host scan) steps, so that the 64-entry ring is
    flushed with stamped and evented steps mixed; profiling is switched off for ten steps in the middle."""
    scans = at_scale_scans(160)
    runs = [("D", 20), ("H", 7), ("D", 25), ("H", 12), ("D", 11), ("off", 10), ("D", 30), ("H", 5), ("D", 40)]
    with Sequence(at_scale_config(512), extra=1) as seq:
        prof = seq.handles[2]
        prof.set_profiling(True)
        kinds = [kind for kind, count in runs for _ in range(count)]
        assert len(kinds) == len(scans)
        t0 = time.perf_counter()
        for i, ((obs, odo), kind, d) in enumerate(zip(scans, kinds, seq.upload(scans))):
            if kind != kinds[i - 1] and "off" in (kind, kinds[i - 1]):
                prof.set_profiling(kind != "off")
            if kind == "H":
                seq.host(obs, odo, check=False)
            else:
                seq.device(obs, odo, check=False, dev=d)
            if i in (63, 127):
                seq.sync()
                seq.compare(particles=range(i % 5, 512, 37), other=prof)
        seq.sync()
        wall_ms = 1e3 * (time.perf_counter() - t0)
        ph, steps = prof.phase_ms()
        assert steps == 150 == sum(k != "off" for k in kinds), steps
        assert all(0.0 <= v < wall_ms for v in ph.values()), (ph, wall_ms)
        assert ph["ray_update"] > 0.0 and ph["motion_likelihood"] > 0.0, ph
        assert seq.chained == [k != "H" for k in kinds], seq.chained
        # the ring's first two rounds each hold stamped and evented steps
        assert any(seq.chained[:64]) and not all(seq.chained[:64])
        assert any(seq.chained[64:128]) and not all(seq.chained[64:128])
        seq.compare(other=prof)
        seq.compare(particles=range(0, 512, 7))
