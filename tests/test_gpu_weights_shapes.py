"""k_weights at every launch shape, and the adaptive-resampling decision.

k_weights runs on a cluster of 1, 2, 4 or 8 CTAs with the elements in registers, or, above 65,536 particles, on
the generic kernel whose chunks are re-read from global memory (launch_weights, kernels_resample.cu). The
cross-CTA parts of its exact folds (remote records, per-CTA head tables, the argmax merge) only run at some of
these shapes, so every case here runs on device through the debug hook, is compared with the oracle's strict
left folds bit for bit, and asserts the launch the hook reports, so that it shows it reached the shape it is
named for. The last part checks the adaptive-resampling decision `N_eff < tau * N` (particle.rs:59-65, slam.rs:74
with resample_threshold > 0) against the reference's sequential fold of the squares, through the hook and in
lockstep runs of the SLAM filter and the localiser."""
import numpy as np
import pytest

from oracle import loc_oracle as LO
from slamrs_b200 import GpuPlacement, GridMapLocalizer, GridMapSlam, GridMapSlamConfig, SensorModel, _lib, grid_cells
from slamrs_b200.simulator import reference_scene, scene_map
from slamrs_b200.slam import debug_resample

from common import SEED, WEIGHT_RTOL, compare_step, make_scans, oracle_slam

pytestmark = pytest.mark.gpu

U_MAX = 1.0 - 2.0 ** -53       # largest value rand::random::<f64>() returns
FOLD_HEADS_PER_CTA = 32        # kernels_resample.cu: head records per CTA; a CTA's 33rd head overflows the table

# population -> (CTAs in the cluster, elements in registers) it is named for
SHAPES = {
    8191: (1, True), 8192: (1, True),                        # one CTA, last thread partly filled / full
    8193: (2, True),                                         # the second CTA holds one element
    16383: (2, True), 16384: (2, True), 16385: (4, True),
    32767: (4, True), 32768: (4, True), 32769: (8, True),
    65535: (8, True), 65536: (8, True),
    65537: (8, False),                                       # first generic size: chunks of 9
    73729: (8, False),                                       # chunks of 10, the last one short
    1 << 20: (8, False), (1 << 20) + 1: (8, False),
}
SHAPE_IDS = [str(n) for n in SHAPES]


def _bits(x):
    return np.asarray(x, np.float64).view(np.int64)


def _launch(n):
    """The launch k_weights uses for n particles, as the hook reports it."""
    got = debug_resample(np.ones(n), 0.0)
    assert (got["cluster"], got["regs"]) == SHAPES.get(n, (got["cluster"], got["regs"])), got
    return got


def _ctas(shape, n):
    """[first, end) of every CTA that holds an element."""
    span = shape["threads"] * shape["chunk"]
    return [(c * span, min(n, (c + 1) * span)) for c in range(shape["cluster"]) if c * span < n]


def _ref_decision(norm, tau):
    """number_of_effective_particles (particle.rs:59-65: `sum += w * w` left to right) and `N_eff < tau * N`."""
    sq = np.cumsum(norm * norm)[-1]                          # np.cumsum is a sequential fold
    n_eff = np.float64(1.0) / sq
    return n_eff, bool(n_eff < tau * norm.size)


def _check(oracle, w, u, tau=0.0, n=None, expect_no_fallback=False):
    """Device against the oracle's folds: normalised weights and running sum by bits, indices, argmax, clamp; with
    tau > 0 also N_eff by bits and the decision. Returns the hook's result."""
    ref = oracle.resample_fold(w, u)
    got = debug_resample(w, u, tau=tau)
    if n is not None:
        assert (got["cluster"], got["regs"]) == SHAPES[n], got
    assert np.array_equal(_bits(ref["norm"]), _bits(got["norm"])), \
        f"normalised weights differ first at {np.nonzero(_bits(ref['norm']) != _bits(got['norm']))[0][:4]}"
    assert np.array_equal(_bits(ref["cum"]), _bits(got["cum"])), \
        f"running sum differs first at {np.nonzero(_bits(ref['cum']) != _bits(got['cum']))[0][:4]}"
    assert ref["max_particle"] == got["max_particle"]
    if tau > 0.0:
        n_eff, resample = _ref_decision(ref["norm"], tau)
        assert got["do_resample"] == resample, (w.size, tau, float(n_eff), got["n_eff"])
        if np.isnan(n_eff):
            assert np.isnan(got["n_eff"])
        else:
            assert _bits(got["n_eff"]) == _bits(n_eff), (w.size, tau, float(n_eff), got["n_eff"])
    if tau == 0.0 or got["do_resample"]:
        assert np.array_equal(ref["idx"].astype(np.int64), got["idx"].astype(np.int64)), \
            f"indices differ first at {np.nonzero(ref['idx'].astype(np.int64) != got['idx'])[0][:4]}"
        assert bool(ref["clamped"]) == bool(got["clamped"])
    else:   # every particle stays in place
        assert np.array_equal(got["idx"], np.arange(w.size, dtype=np.uint32))
    if expect_no_fallback:
        assert got["fold_fallback"] == 0 and got["fold_rounds"] <= 3, got
    return got


# ------------------------------------------------------------------------------------------- launch shapes

@pytest.mark.parametrize("n", list(SHAPES), ids=SHAPE_IDS)
def test_launch_shapes_realistic_weights(oracle, n):
    shape = _launch(n)
    if n == 73729:
        assert shape["chunk"] == 10 and n % 10 != 0
    rng = np.random.default_rng(n)
    ctas = _ctas(shape, n)
    for u in (0.0, float(rng.random()), U_MAX):
        _check(oracle, rng.random(n), u, n=n, expect_no_fallback=True)
        _check(oracle, np.exp(rng.normal(-200.0, 10.0, n)), u, n=n, expect_no_fallback=True)
    # peaked: one weight 1.0 on the first / last element of a CTA, the rest far below it
    for first, end in (ctas[0], ctas[-1], ctas[len(ctas) // 2]):
        for at in (first, end - 1):
            w = np.exp(rng.normal(-38.0, 1.0, n))
            w[at] = 1.0
            got = _check(oracle, w, float(rng.random()), n=n, expect_no_fallback=True)
            assert got["max_particle"] == at


@pytest.mark.parametrize("n", list(SHAPES), ids=SHAPE_IDS)
def test_launch_shapes_thresholds_on_the_prefix_sums(oracle, n):
    """Equal and small-integer weights put the resampling thresholds on the running sums: every `u > c` is
    decided in the last bit."""
    rng = np.random.default_rng(n + 1)
    ints = rng.integers(0, 4, n).astype(np.float64)
    for u in (0.0, U_MAX):
        _check(oracle, np.ones(n), u, n=n, expect_no_fallback=True)
        _check(oracle, np.full(n, 3.0), u, n=n, expect_no_fallback=True)
        _check(oracle, ints, u, n=n, expect_no_fallback=True)


# ------------------------------------------------------------------------------------------- boundary structure

@pytest.mark.parametrize("n", list(SHAPES), ids=SHAPE_IDS)
def test_single_survivor_at_every_cta_edge(oracle, n):
    """One non-zero weight: every new particle is a copy of it, from the first or last element of each CTA."""
    shape = _launch(n)
    spots = sorted({i for first, end in _ctas(shape, n) for i in (first, end - 1)} | {n - 1})
    for i in spots:
        w = np.zeros(n)
        w[i] = 0.6180339887
        for u in (0.5, U_MAX):
            got = _check(oracle, w, u, n=n, expect_no_fallback=True)
            assert np.all(got["idx"] == i) and got["max_particle"] == i


@pytest.mark.parametrize("n", list(SHAPES), ids=SHAPE_IDS)
def test_tied_maxima_the_last_one_wins(oracle, n):
    """particle.rs:40-46 (max_by keeps the last maximum): ties in the first and last CTA, across adjacent chunks
    and across the boundary of two CTAs."""
    shape = _launch(n)
    ctas = _ctas(shape, n)
    L = shape["chunk"]
    rng = np.random.default_rng(n + 2)
    k = (ctas[0][1] // L) // 2                               # a chunk boundary inside the first CTA
    pairs = [(ctas[0][0] + 3, ctas[-1][1] - 2),              # first and last CTA
             (k * L - 1, k * L)]                             # last element of one chunk, first of the next
    if len(ctas) > 1:
        pairs.append((ctas[0][1] - 1, ctas[1][0]))           # across the first CTA boundary
        pairs.append((ctas[-2][1] - 1, ctas[-1][0]))         # and the last
    for a, b in pairs:
        w = rng.random(n) * 0.5
        w[a] = w[b] = 1.0
        got = _check(oracle, w, float(rng.random()), n=n, expect_no_fallback=True)
        assert got["max_particle"] == max(a, b), (a, b)


# ------------------------------------------------------------------------------------------- hostile input

@pytest.mark.parametrize("n", list(SHAPES), ids=SHAPE_IDS)
def test_hostile_input_stays_exact(oracle, n):
    """NaN, +inf and an all-zero population leave the parallel fold to its single-thread fallback; geometric
    doublings across a CTA boundary change the binade with every element. Every result is the reference's."""
    shape = _launch(n)
    ctas = _ctas(shape, n)
    rng = np.random.default_rng(n + 3)
    w = rng.random(n); w[ctas[-1][0] + (ctas[-1][1] - ctas[-1][0]) // 2] = np.nan
    got = _check(oracle, w, 0.25, n=n)
    assert got["fold_fallback"] != 0 and np.all(got["idx"] == 0)
    first, end = ctas[(len(ctas) - 1) // 2]                  # a middle CTA, and a full one
    w = rng.random(n); w[(first + end) // 2] = np.inf
    assert _check(oracle, w, 0.25, n=n)["fold_fallback"] != 0
    got = _check(oracle, np.zeros(n), 0.25, n=n)
    assert got["fold_fallback"] != 0 and np.all(got["idx"] == 0)
    # 2^-1000 .. 2^999 over 2,000 consecutive elements across a CTA boundary
    b = ctas[1][0] if len(ctas) > 1 else n // 2
    lo = min(b - 1000, n - 2000)                             # (n = 8,193: the second CTA holds one element)
    w = np.zeros(n)
    w[lo:lo + 2000] = 2.0 ** np.arange(-1000, 1000).astype(np.float64)
    got = _check(oracle, w, 0.5, n=n)
    if shape["regs"]:   # more than 32 binade-changing chunks in each CTA: the head tables overflow
        assert got["fold_fallback"] != 0, got
    else:               # long chunks (128 elements at 2^20) can keep the heads within the tables: the chain folds them
        assert got["fold_fallback"] != 0 or got["fold_heads"] > 2, got


@pytest.mark.parametrize("n", list(SHAPES), ids=SHAPE_IDS)
@pytest.mark.parametrize("tau", [0.0, 0.5])
def test_head_table_full_and_overflowing(oracle, n, tau):
    """FOLD_HEADS_PER_CTA chunks in one CTA whose fold changes binade (2^j at the start of chunk j, zeros
    elsewhere) fill the CTA's head table: the fold stays parallel. One more overflows it (a head's index in its
    CTA reaches FOLD_HEADS_PER_CTA): every fold -- the sum, the running sum and, with tau > 0, the sum of squares --
    falls back to one thread. Both sides are exact."""
    shape = _launch(n)
    ctas = _ctas(shape, n)
    first, _ = ctas[(shape["cluster"] - 1) // 2]             # a full CTA
    for m in (FOLD_HEADS_PER_CTA, FOLD_HEADS_PER_CTA + 1):
        w = np.zeros(n)
        w[first + shape["chunk"] * np.arange(m)] = 2.0 ** np.arange(m).astype(np.float64)
        got = _check(oracle, w, 0.75, tau=tau, n=n)
        if m == FOLD_HEADS_PER_CTA:
            assert got["fold_fallback"] == 0 and got["fold_heads"] == FOLD_HEADS_PER_CTA, got
        else:
            assert got["fold_fallback"] == (7 if tau > 0.0 else 3), got


# ------------------------------------------------------------------------------------------- k_resample_indices

@pytest.mark.parametrize("n", [2047, 2048, 2049, 4095, 4097, 6145])
def test_coarse_search_block_boundaries(oracle, n):
    """k_resample_indices bisects every ceil(N / 2048)-th running sum first: the block length changes at 2,049
    and 4,097 particles, and 6,145 leaves a short last block."""
    ints = np.random.default_rng(n).integers(0, 4, n).astype(np.float64)
    for u in (0.0, 2.0 ** -53, U_MAX):
        for w in (np.ones(n), np.full(n, 3.0), ints):
            _check(oracle, w, u, expect_no_fallback=True)


# ------------------------------------------------------------------------------------------- adaptive decision

def test_adaptive_decision_equal_weights(oracle):
    """Equal weights at tau = 1: N_eff is N up to rounding, so `N_eff < N` is decided by the last bit of the sum of
    squares. The device must take the reference's sequential fold, not a re-associated one."""
    for n in list(range(17, 601)) + list(SHAPES):
        for value in (1.0, np.exp(-37.25)):
            _check(oracle, np.full(n, value), 0.0, tau=1.0)


@pytest.mark.parametrize("n", [48, 100, 1000, 8200, 16384, 40000, 65536, 73728])
def test_adaptive_decision_k_equal_weights_among_zeros(oracle, n):
    """k = tau * N equal non-zero weights among zeros: N_eff = k up to rounding, against tau * N = k."""
    shape = _launch(n)
    ctas = _ctas(shape, n)
    for tau in (0.25, 0.5, 0.75):
        k = int(tau * n)
        assert k == tau * n and np.float32(tau) == tau
        b = ctas[1][0] if len(ctas) > 1 else n // 2
        start = min(max(b - k // 2, 0), n - k)
        placements = {"front": np.arange(k), "back": np.arange(n - k, n), "interleaved": (np.arange(k) * n) // k,
                      "straddling": np.arange(start, start + k)}
        for where, at in placements.items():
            assert np.unique(at).size == k, where
            for value in (1.0, 3.7e-17):
                w = np.zeros(n)
                w[at] = value
                _check(oracle, w, 0.3, tau=tau)


def test_adaptive_decision_nan_weights_never_resample(oracle):
    """NaN weights make N_eff NaN; `N_eff < tau * N` is then false on both sides: no resampling."""
    rng = np.random.default_rng(11)
    for n in (100, 8193, 65537):
        for tau in (0.5, 1.0):
            w = rng.random(n); w[n // 3] = np.nan
            got = _check(oracle, w, 0.25, tau=tau)
            assert not got["do_resample"] and np.isnan(got["n_eff"])
            got = _check(oracle, np.zeros(n), 0.25, tau=tau)
            assert not got["do_resample"] and np.isnan(got["n_eff"])


def _lockstep_equal_weights(filt, orc, scans, n, check=None):
    """Steps the device filter and the oracle with all-zero motion draws and u = 0: every particle keeps one pose and
    one grid, so the weights stay equal. The oracle resamples on the device's raw weights (set_weight_override:
    device exp/log may differ from glibc by an ulp), so N_eff must agree by bits and the decision exactly."""
    z = np.zeros(2 * n)
    decisions = []
    for step, (obs, odo) in enumerate(scans):
        filt.update(obs, odo, z_draws=z, resample_u=0.0)
        norm_g, raw_g = filt.weights()
        assert np.all(raw_g == raw_g[0]), step
        orc.set_weight_override(raw_g)
        ang = obs.angle.astype(np.float32).astype(np.float64)
        dist = obs.distance.astype(np.float32).astype(np.float64)
        assert orc.update(ang, dist, obs.valid.astype(np.uint8), np.float32(odo.distance_left),
                          np.float32(odo.distance_right), np.float32(odo.wheel_distance), z, 0.0) == 0
        own = orc.own_raw_weights()
        assert float(np.max(np.abs(raw_g - own) / np.maximum(np.abs(own), 1e-300))) < WEIGHT_RTOL, step
        n_eff_ref, n_eff_got = orc.number_of_effective_particles(), filt.number_of_effective_particles()
        assert bool(filt.stats()["resampled"]) == orc.resampled(), (step, n_eff_got, n_eff_ref)
        assert _bits(n_eff_got) == _bits(n_eff_ref), (step, n_eff_got, n_eff_ref)
        assert np.array_equal(filt.resample_indices().astype(np.int64), orc.indices().astype(np.int64)), step
        if check is not None:
            check()
        decisions.append(orc.resampled())
    return decisions


@pytest.mark.parametrize("n", [23, 25, 48, 100, 1000])
def test_adaptive_decision_end_to_end_slam(oracle, n):
    cfg = GridMapSlamConfig(position=(-2.0, -2.0), width=4.0, height=4.0, resolution=0.02, n_particles=n)
    particles = range(n) if n <= 100 else sorted(set(range(0, n, 61)) | {n - 1})
    osl = oracle_slam(oracle, cfg)
    osl.set_adaptive_resampling(1.0)
    try:
        with GridMapSlam(cfg, GpuPlacement(seed=SEED, rng_mode=_lib.RNG_CALLER, resample_threshold=1.0)) as gpu:
            _lockstep_equal_weights(gpu, osl, make_scans(1.0, 360, 1.0, 4), n,
                                    check=lambda: compare_step(gpu, osl, particles))
    finally:
        osl.close()


def test_adaptive_decision_end_to_end_localizer(oracle):
    n = 100
    cfg = GridMapSlamConfig(position=(-2.0, -2.0), width=4.0, height=4.0, resolution=0.02, n_particles=n)
    prob = scene_map(reference_scene(1.0), cfg)
    g = grid_cells(cfg.width, cfg.resolution)
    model = SensorModel()
    ol = LO.OracleLocalizer(cfg.position, cfg.resolution, g, g, n, prob, model.kind, model.sigma, model.z_rand,
                            model.occupied_above)
    ol.set_adaptive_resampling(1.0)
    try:
        with GridMapLocalizer(cfg, prob, model,
                              GpuPlacement(seed=SEED, rng_mode=_lib.RNG_CALLER, resample_threshold=1.0)) as loc:
            _lockstep_equal_weights(loc, ol, make_scans(1.0, 360, 1.0, 4), n)
            assert np.array_equal(loc.poses().view(np.uint32), ol.poses().view(np.uint32))
    finally:
        ol.close()
