"""The C++ host mirror of the reference interface (slamrs_b200/csrc/host/grid_map_slam.hpp):
CPU: it compiles against the C ABI and fails loudly without a GPU. GPU: driven like
GridMapSlamNode::update it gives the same poses and maps as the Python binding."""
import os
import subprocess

import numpy as np
import pytest

from slamrs_b200 import GridMapSlam, GridMapSlamConfig, Odometry
from slamrs_b200 import _lib

from common import gpu_present, make_scans

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _build(out_dir):
    """Compiles the check program into out_dir (a test's temporary directory: the source tree may be read-only)."""
    _lib.load()
    libdir = os.path.join(ROOT, "slamrs_b200")
    src = os.path.join(ROOT, "tests", "cpp", "host_mirror_check.cpp")
    exe = os.path.join(str(out_dir), "host_mirror_check")
    cmd = ["g++", "-std=c++17", "-O2", src, "-o", exe, "-L" + libdir, "-lslamrs_gpu", "-Wl,-rpath," + libdir]
    env = dict(os.environ); env.pop("CXX", None)
    subprocess.run(cmd, check=True, env=env)
    return exe


@pytest.mark.skipif(gpu_present(), reason="GPU present")
def test_cpp_mirror_builds_and_refuses_to_run_without_gpu(tmp_path):
    out = subprocess.run([_build(tmp_path), "--no-gpu"], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "no CPU fallback" in out.stdout


@pytest.mark.gpu
def test_cpp_mirror_matches_python_binding(tmp_path):
    (obs, _), = make_scans(1.0, 360, 1.0, 1)
    scan = tmp_path / "scan.txt"
    with open(scan, "w") as f:
        for a, d, v in zip(obs.angle, obs.distance, obs.valid):
            f.write(f"{float(np.float32(a))!r} {float(np.float32(d))!r} {int(v)}\n")
    out = subprocess.run([_build(tmp_path), str(scan)], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout + out.stderr
    lines = [ln.split() for ln in out.stdout.strip().splitlines()]
    assert len(lines) == 6
    with GridMapSlam(GridMapSlamConfig()) as g:          # same preset, same default seed
        for s in range(3):
            g.update(obs, Odometry.new(np.float32(0.08), np.float32(0.10), np.float32(0.1)))
            p = g.estimated_pose()
            m = g.estimated_likelihood().data
            for cycle in (0, 1):                          # destroy/create cycle gives the same run
                ln = lines[cycle * 3 + s]
                assert [float(ln[5]), float(ln[6]), float(ln[7])] == pytest.approx([p.x, p.y, p.theta], rel=1e-7)
                assert ln[9] == "200x200"
                assert float(ln[11]) == float((m > 0.5).sum()) and float(ln[13]) == float((m < 0.5).sum())
