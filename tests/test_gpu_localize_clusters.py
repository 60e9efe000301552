"""Pose clusters of the localiser (slamrs_gpu_pose_clusters, AMCL's cluster statistics): against the cluster oracle
(oracle/cluster_oracle.c for the integers, oracle/cluster_oracle.py for the moments) on hand-placed generations,
random clouds at 4,096 and 2^20 poses and a KLD handle whose population has shrunk; bitwise reproducibility; a handle
that calls it after every step stays bitwise equal to one that never does; the argument checks; and what cluster 0
shows in global localisation and after a kidnapping at 2^20 particles."""
import ctypes as C
import math

import numpy as np
import pytest

from oracle import cluster_oracle as CO
from slamrs_b200 import (Clustering, GpuPlacement, GridMapLocalizer, GridMapSlam, GridMapSlamConfig, Kld, Recovery,
                         SensorModel, _lib, grid_cells)
from slamrs_b200.simulator import Simulator, reference_scene, scene_map

from common import SEED, at_scale_config, make_scans
from test_gpu_localize_kld import room_map

pytestmark = pytest.mark.gpu

PRESET = GridMapSlamConfig(position=(-2.0, -2.0), width=4.0, height=4.0, resolution=0.02, n_particles=256)
FIELD = SensorModel.likelihood_field(sigma=0.1, z_rand=0.05)
U = 2.0 ** -53   # unit roundoff of f64
# ulp bounds of the f64 functions the two sides evaluate, in units of 2u = one ulp: CUDA's sin, cos and atan2 are
# within 2 ulp and its log within 1 ulp (CUDA C++ Programming Guide, double-precision mathematical functions); glibc's
# sin, cos, atan2 and log within 1 ulp
ULP_SINCOS, ULP_ATAN2, ULP_LOG = 2 + 1, 2 + 1, 1 + 1


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint64 if np.asarray(a).dtype == np.float64 else np.uint32)


def _bounds(rec, mg):
    """Tolerances of the device's moments against the oracle's correctly rounded ones for a set of m poses.
    A sum of m terms in any order is within (m - 1) u sum|t| of the exact sum, and a correctly rounded one within
    u |sum|; each division or square root adds u of its result. S and C add the ulp errors of sin and cos on each term.
    The centred second pass with the device's means instead of the exact ones differs from the exact centred sum by
    -dmx sum(dy) - dmy sum(dx) + m dmx dmy, and sum(dy) over the oracle's deviations is itself within m 2u |my| + u
    sum|dy| of 0: no first-order term remains."""
    m = rec["count"]
    mx, my, _ = rec["mean"]
    t = {}
    t["mx"] = (m * U * mg["x"]) / m + 2 * U * abs(mx)
    t["my"] = (m * U * mg["y"]) / m + 2 * U * abs(my)
    t["S"] = (m + 2 * ULP_SINCOS) * U * mg["s"]
    t["C"] = (m + 2 * ULP_SINCOS) * U * mg["c"]
    S, Cc = mg["S"], mg["C"]
    r2 = S * S + Cc * Cc
    t["mt"] = (abs(Cc) * t["S"] + abs(S) * t["C"]) / r2 + 2 * ULP_ATAN2 * U * math.pi if r2 > 0 else math.inf
    dlnr = (abs(S) * t["S"] + abs(Cc) * t["C"]) / r2 + 8 * U if r2 > 0 else math.inf
    t["var"] = 2 * dlnr + 2 * ULP_LOG * U * abs(rec["var_theta"]) + 4 * U
    sdx = m * 2 * U * abs(mx) + U * mg["dx"]
    sdy = m * 2 * U * abs(my) + U * mg["dy"]
    for key, mag, da, db, sa, sb in (("xx", mg["xx"], t["mx"], t["mx"], sdx, sdx), ("xy", mg["xy"], t["mx"], t["my"], sdy, sdx),
                                     ("yy", mg["yy"], t["my"], t["my"], sdy, sdy)):
        # m - 1 additions, and per term: the subtraction on each side and the product (3 u), on both sides
        t[key] = ((m + 6) * U * mag + da * sa + db * sb + m * da * db) / m + 4 * U * mag / m
    return t


def _angle_diff(a, b):
    return abs(math.remainder(a - b, 2.0 * math.pi))


def _check_record(got, want, mg, what):
    assert got["count"] == want["count"], what
    assert _bits(np.float64(got["weight"])) == _bits(np.float64(want["weight"])), what   # count / N, correctly rounded
    if want["count"] == 0:
        assert np.all(got["mean"] == 0) and np.all(got["cov"] == 0) and got["weight"] == 0, what
        return
    t = _bounds(want, mg)
    g = got["mean"]
    assert abs(g[0] - want["mean"][0]) <= t["mx"], (what, g, want, t)
    assert abs(g[1] - want["mean"][1]) <= t["my"], (what, g, want, t)
    assert -math.pi < g[2] <= math.pi and _angle_diff(g[2], want["mean"][2]) <= t["mt"], (what, g, want, t)
    cov = got["cov"]
    assert cov[0, 1] == cov[1, 0] and cov[0, 2] == cov[1, 2] == cov[2, 0] == cov[2, 1] == 0.0
    for key, v in (("xx", cov[0, 0]), ("xy", cov[0, 1]), ("yy", cov[1, 1])):
        assert abs(v - want["cov_" + key]) <= t[key], (what, key, v, want, t)
    assert abs(cov[2, 2] - want["var_theta"]) <= t["var"], (what, cov[2, 2], want, t)


def _against_oracle(loc, cfg, cl):
    """pose_clusters on the handle's current generation against the oracle on the same poses."""
    g = grid_cells(cfg.width, cfg.resolution)
    xyt = loc.poses()
    overall, clusters = loc.pose_clusters(cl)
    stats, want, mags = CO.expected(xyt, cfg.position, cfg.resolution, g, g, cl.bin_cells(cfg.resolution), cl.theta_bins,
                                    cl.max_clusters)
    for key in ("n_poses", "n_excluded", "n_bins", "n_clusters"):
        assert overall[key] == stats[key], (key, overall, stats)
    assert len(clusters) == len(want) == min(cl.max_clusters, stats["n_clusters"])
    assert [(c["label"], c["count"]) for c in clusters] == [(w["label"], w["count"]) for w in want]
    _check_record(overall, stats["overall"], mags["overall"], "overall")
    for j, (c, w) in enumerate(zip(clusters, want)):
        _check_record(c, w, mags[j], j)
    return overall, clusters


def _raw(loc, cl):
    """The raw output bytes of one call (stats and all K entries)."""
    c = cl.to_struct(loc.config.resolution)
    st = _lib.PoseStats()
    arr = (_lib.PoseCluster * cl.max_clusters)()
    _lib.check(loc._L.slamrs_gpu_pose_clusters(loc._h, C.byref(c), C.byref(st), arr), loc._h)
    return bytes(st) + bytes(arr)


def _blob(rng, n, x, y, t, sxy, st):
    return np.column_stack([rng.normal(x, sxy, n), rng.normal(y, sxy, n), rng.normal(t, st, n)])


def _hand_placed():
    rng = np.random.default_rng(17)
    pi = math.pi
    wrap = lambda a: np.column_stack([a[:, 0], a[:, 1], np.remainder(a[:, 2] + pi, 2 * pi) - pi])   # noqa: E731
    cases = {
        "two_blobs": np.vstack([_blob(rng, 600, 0.5, 0.5, 0.3, 0.08, 0.05), _blob(rng, 400, -1.0, -1.0, 2.0, 0.1, 0.1)]),
        "pi_blob": wrap(_blob(rng, 500, 0.2, -0.3, pi, 0.05, 0.08)),
        "corner_chain": np.array([[-2.0 + (i + 0.5) * 0.2, -2.0 + (i + 0.5) * 0.2, -pi + (i + 0.5) * 2 * pi / 36]
                                  for i in range(12)]),
        "off_grid_and_nan": np.vstack([_blob(rng, 200, 0.0, 0.0, 0.0, 0.1, 0.1),
                                       [[np.nan, 0, 0], [0, np.inf, 0], [0, 0, np.nan], [5.0, 0, 0], [0, -2.5, 1.0],
                                        [-2.0 - 1e-6, 0, 0]]]),
        "one_pose": np.array([[0.3, -0.4, 1.0]]),
        "one_bin": np.tile([[0.11, -0.07, 0.2]], (256, 1)),
        "ties": np.vstack([_blob(rng, 100, cx, cy, 0.0, 0.02, 0.02) for cx, cy in ((-1.5, -1.5), (1.5, -1.5), (-1.5, 1.5),
                                                                                   (1.5, 1.5))]),
        "all_excluded": np.full((8, 3), np.nan),
    }
    return {k: np.asarray(v, np.float32) for k, v in cases.items()}


@pytest.mark.parametrize("case", list(_hand_placed().keys()))
def test_hand_placed_generations_against_oracle(case):
    xyt = _hand_placed()[case]
    cfg = GridMapSlamConfig(position=PRESET.position, width=PRESET.width, height=PRESET.height,
                            resolution=PRESET.resolution, n_particles=xyt.shape[0])
    prob = scene_map(reference_scene(1.0), cfg)
    with GridMapLocalizer(cfg, prob, placement=GpuPlacement(seed=SEED)) as loc:
        loc.set_poses(xyt)
        for cl in (Clustering(bin_xy=0.2, theta_bins=36, max_clusters=16), Clustering(bin_xy=0.5, theta_bins=1, max_clusters=3),
                   Clustering(bin_xy=0.1, theta_bins=2, max_clusters=64), Clustering(bin_xy=0.2, theta_bins=36, max_clusters=2)):
            overall, clusters = _against_oracle(loc, cfg, cl)
            if case == "pi_blob" and cl.theta_bins == 36:
                assert clusters[0]["count"] >= 490 and abs(abs(clusters[0]["mean"][2]) - math.pi) < 0.05
            if case == "corner_chain" and cl.bin_xy == 0.2 and cl.theta_bins == 36:
                assert overall["n_bins"] == 12 and overall["n_clusters"] == 1
            if case == "ties" and cl.max_clusters == 2:
                assert overall["n_clusters"] == 4 and [c["count"] for c in clusters] == [100, 100]
            if case == "one_bin":
                assert overall["n_bins"] == 1 and clusters[0]["count"] == 256 and np.all(clusters[0]["cov"][:2, :2] == 0)
            if case == "all_excluded":
                assert overall["n_excluded"] == 8 and overall["n_clusters"] == 0 and clusters == []
        raw = _raw(loc, Clustering(max_clusters=64))
        if case == "all_excluded":   # every entry zeroed
            assert raw[32:] == bytes(len(raw) - 32)


@pytest.mark.parametrize("n", [4096, 1 << 20])
def test_random_clouds_against_oracle(n):
    cfg = at_scale_config(n)
    prob = scene_map(reference_scene(10.0), cfg)
    with GridMapLocalizer(cfg, prob, placement=GpuPlacement(seed=SEED)) as loc:
        loc.init_uniform((-11.0, -11.0, 11.0, 11.0))
        for cl in (Clustering(), Clustering(bin_xy=0.25, theta_bins=18, max_clusters=64)):
            _against_oracle(loc, cfg, cl)
        # clustered: 7 blobs of different spreads, a tenth of the poses off the grid
        rng = np.random.default_rng(n)
        k = rng.integers(0, 7, n)
        c = rng.uniform(-9.0, 9.0, (7, 3))
        xyt = np.column_stack([c[k, 0] + rng.normal(0, 0.1 + 0.1 * k), c[k, 1] + rng.normal(0, 0.1 + 0.1 * k),
                               c[k, 2] + rng.normal(0, 0.1, n)]).astype(np.float32)
        xyt[rng.random(n) < 0.1, 0] = 40.0
        loc.set_poses(xyt)
        overall, clusters = _against_oracle(loc, cfg, Clustering(max_clusters=8))
        assert overall["n_clusters"] >= 2


def test_shrunk_kld_population_against_oracle():
    """With KLD-sampling the call clusters the N poses of the current generation, not the capacity."""
    cfg = at_scale_config(4096)
    prob = room_map(reference_scene(10.0), cfg)
    obs, odo = make_scans(10.0, 360, 6.0, 1)[0]
    with GridMapLocalizer(cfg, prob, FIELD, GpuPlacement(seed=SEED)) as loc:
        loc.set_kld(Kld(n_min=100, err=1.0))
        loc.init_uniform((-0.3, -0.3, 0.3, 0.3))
        loc.update(obs, odo)
        n = loc.population
        assert 100 <= n < 4096
        overall, _ = _against_oracle(loc, cfg, Clustering())
        assert overall["n_poses"] == n
        for c in (overall,):
            assert c["count"] + c["n_excluded"] == n


def test_reproducible_across_calls_and_twins():
    cfg = at_scale_config(1 << 18)
    prob = room_map(reference_scene(10.0), cfg)
    scans = make_scans(10.0, 360, 6.0, 3)
    with GridMapLocalizer(cfg, prob, FIELD, GpuPlacement(seed=SEED)) as a, \
            GridMapLocalizer(cfg, prob, FIELD, GpuPlacement(seed=SEED)) as b:
        for h in (a, b):
            h.init_uniform((-9.0, -9.0, 9.0, 9.0))
        for obs, odo in scans:
            for h in (a, b):
                h.update(obs, odo)
            for cl in (Clustering(), Clustering(bin_xy=0.2, theta_bins=72, max_clusters=64)):
                ra = _raw(a, cl)
                assert ra == _raw(a, cl) == _raw(b, cl)


def _state(loc):
    ep = loc.estimated_pose()
    norm, raw = loc.weights()
    return (_bits(loc.poses()).tobytes(), _bits(norm).tobytes(), _bits(raw).tobytes(), loc.resample_indices().tobytes(),
            loc.max_particle, (ep.x, ep.y, ep.theta), loc.recovery_state(), loc.kld_state(), loc.population,
            loc.number_of_effective_particles())


def test_calling_after_every_step_changes_nothing():
    cfg = at_scale_config(4096)
    segments = reference_scene(10.0)
    prob = room_map(segments, cfg)
    scans = make_scans(10.0, 360, 6.0, 20)
    with GridMapLocalizer(cfg, prob, FIELD, GpuPlacement(seed=SEED)) as a, \
            GridMapLocalizer(cfg, prob, FIELD, GpuPlacement(seed=SEED)) as b:
        for h in (a, b):
            h.set_recovery(Recovery(alpha_slow=0.05, alpha_fast=0.5))
            h.set_kld(Kld(n_min=64, err=0.05, bin_xy=0.25, theta_bins=18))
            h.init_uniform((-9.0, -9.0, 9.0, 9.0))
        a.pose_clusters()
        for step, (obs, odo) in enumerate(scans):
            la, lb = a.launch_count, b.launch_count
            if step % 2:
                a.upload_scan(obs); a.step_async(odo)
                b.upload_scan(obs); b.step_async(odo)
            else:
                a.update(obs, odo)
                b.update(obs, odo)
            assert a.launch_count - la == b.launch_count - lb, step
            a.pose_clusters(Clustering(max_clusters=1 + step))   # straight behind the step, no sync
            assert _state(a) == _state(b), step
            assert a.recovery_state()["w_slow"] > 0 and a.kld_state()["k"] > 0, step


@pytest.mark.parametrize("what", ["slam", "null_c", "null_out", "null_clusters", "bin_cells_0", "theta_bins_0",
                                  "theta_bins_3601", "max_clusters_0", "max_clusters_65", "bin_space", "struct_size"])
def test_argument_checks(what):
    cfg = at_scale_config(256)
    prob = scene_map(reference_scene(1.0), cfg)
    filt = GridMapSlam(cfg) if what == "slam" else GridMapLocalizer(cfg, prob)
    msg = {"slam": "SLAM handle", "null_c": "null", "null_out": "null", "null_clusters": "null", "struct_size": "struct_size",
           "bin_space": "2^28"}.get(what, "clustering")
    c = Clustering().to_struct(cfg.resolution)
    if what == "bin_cells_0": c.bin_cells = 0
    elif what == "theta_bins_0": c.theta_bins = 0
    elif what == "theta_bins_3601": c.theta_bins = 3601
    elif what == "max_clusters_0": c.max_clusters = 0
    elif what == "max_clusters_65": c.max_clusters = 65
    elif what == "bin_space": c.bin_cells, c.theta_bins = 1, 3600   # 512^2 x 3600 bins
    elif what == "struct_size": c.struct_size = 20
    st = _lib.PoseStats()
    arr = (_lib.PoseCluster * 64)()
    with filt:
        rc = filt._L.slamrs_gpu_pose_clusters(filt._h, None if what == "null_c" else C.byref(c),
                                               None if what == "null_out" else C.byref(st),
                                               None if what == "null_clusters" else arr)
        assert rc == _lib.E_INVALID_ARG and msg.encode() in filt._L.slamrs_gpu_last_error(filt._h), \
            filt._L.slamrs_gpu_last_error(filt._h)
        if what not in ("slam",):   # the bounds themselves are valid
            for ok in (Clustering(bin_xy=0.05, theta_bins=1024, max_clusters=64), Clustering(bin_xy=100.0, theta_bins=3600,
                                                                                              max_clusters=1)):
                filt.pose_clusters(ok)


# Behaviour at 2^20 particles: the scenes and seed of test_global_localisation_with_kld (tests/test_gpu_localize_kld.py)
# and test_kidnapped_robot (tests/test_gpu_localize_recovery.py). Each scan records the error of estimated_pose() and
# of cluster 0's mean against the true pose, and the overall covariance. DESIGN.md section 11.3 has the measured run.
def _err(x, y, t, pose):
    return (math.hypot(x - float(pose[0]), y - float(pose[1])), _angle_diff(t, float(pose[2])))


def _global(kld, scans=40):
    cfg = at_scale_config(1 << 20)
    segments = reference_scene(5.0)
    sim = Simulator(segments, n_beams=360, scanner_range=6.0, wheel_base=0.1)
    trace = []
    with GridMapLocalizer(cfg, scene_map(segments, cfg), FIELD, GpuPlacement(seed=SEED)) as loc:
        loc.set_kld(kld)
        loc.init_uniform((-4.5, -4.5, 4.5, 4.5))
        start, _ = loc.pose_clusters()
        for _ in range(scans):
            obs, odo = sim.next_scan(0.08, 0.10)
            loc.update(obs, odo)
            ep = loc.estimated_pose()
            overall, clusters = loc.pose_clusters()
            trace.append((_err(ep.x, ep.y, ep.theta, sim.pose), _err(*clusters[0]["mean"], sim.pose),
                          float(overall["cov"][0, 0] + overall["cov"][1, 1]), overall["n_clusters"],
                          clusters[0]["weight"]))
    return float(start["cov"][0, 0] + start["cov"][1, 1]), trace


def _mean(tr, j, k):
    return sum(t[j][k] for t in tr[20:40]) / 20.0


def test_global_localisation_cluster_mean():
    """From a uniform start at 2^20 particles, with and without Kld(): the overall covariance falls from the uniform
    spread (9 m box: trace 2 * 81 / 12 = 13.5 m^2) to below 1e-3 of it once the cloud has converged, and cluster 0 then
    tracks the pose. The measured run (DESIGN.md section 11.3), fixed 2^20: over scans 20-39 cluster 0's mean is
    0.0644 m / 0.0008 rad off against estimated_pose()'s 0.0647 m / 0.0024 rad; asserted with a 10 % margin on the
    position and a factor 2 on the heading."""
    for kld in (None, Kld()):
        start, tr = _global(kld)
        print("Kld()" if kld else "fixed 2^20", "per scan (est err m, rad), (cluster 0 err m, rad), trace(cov xy),"
              " n_clusters, weight 0:", [(round(a[0], 4), round(a[1], 4), round(b[0], 4), round(b[1], 4), round(c, 4), d,
                                          round(w, 3)) for a, b, c, d, w in tr])
        print("mean over scans 20-39: estimate %.4f m %.4f rad, cluster 0 %.4f m %.4f rad"
              % (_mean(tr, 0, 0), _mean(tr, 0, 1), _mean(tr, 1, 0), _mean(tr, 1, 1)))
        # the overall covariance shrinks as the cloud converges: from the uniform spread to a tight cloud
        assert start > 10.0 and max(t[2] for t in tr[20:40]) < 1e-3 * start, (start, [t[2] for t in tr])
        assert max(t[1][0] for t in tr[20:40]) < 0.3 and max(t[1][1] for t in tr[20:40]) < 0.1, tr[20:40]
        if kld is None:
            assert _mean(tr, 1, 0) <= 1.1 * _mean(tr, 0, 0) and _mean(tr, 1, 1) <= 0.5 * _mean(tr, 0, 1), tr[20:40]


def test_kidnapped_cluster_mean():
    cfg = at_scale_config(1 << 20)
    segments = reference_scene(5.0)
    sim = Simulator(segments, n_beams=360, scanner_range=6.0, wheel_base=0.1)
    trace = []
    with GridMapLocalizer(cfg, room_map(segments, cfg), FIELD, GpuPlacement(seed=SEED)) as loc:
        loc.set_recovery(Recovery())
        loc.init_uniform((-4.5, -4.5, 4.5, 4.5))
        for k in range(60):
            if k == 20:
                t = float(sim.pose[2])
                sim.pose = [np.float32(3.5), np.float32(3.0), np.float32(t + 2.0)]
            obs, odo = sim.next_scan(0.08, 0.10)
            loc.update(obs, odo)
            ep = loc.estimated_pose()
            overall, clusters = loc.pose_clusters()
            trace.append((_err(ep.x, ep.y, ep.theta, sim.pose), _err(*clusters[0]["mean"], sim.pose), overall["n_clusters"],
                          clusters[0]["weight"], loc.recovery_state()["injected"]))
    print("kidnap per scan (est err m, rad), (cluster 0 err m, rad), n_clusters, weight 0, injected:",
          [(k, round(a[0], 3), round(a[1], 3), round(b[0], 3), round(b[1], 3), c, round(w, 3), i)
           for k, (a, b, c, w, i) in enumerate(trace)])
    assert trace[19][1][0] < 0.2
    assert all(t[1][0] > 1.0 for t in trace[20:55])   # carried away: cluster 0 is lost as the estimate is
    # The measured run: the injected particles find the pose at scan 56 (estimate 0.22 m off); cluster 0 is 0.65, 6.6,
    # 8.8 and 5.3 m off at scans 56-59, because with 0.5 m bins the injected cloud, spread over the room, joins into
    # one cluster that holds (nearly) every pose. Asserted: cluster 0 stays more than 0.3 m off and holds more than
    # 90 % of the poses at each of these scans.
    assert all(t[1][0] > 0.3 and t[3] > 0.9 for t in trace[56:60]), trace[55:60]
