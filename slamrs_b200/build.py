"""Builds libslamrs_gpu.so (the C-ABI product library) in-tree with nvcc for sm_100a."""
from __future__ import annotations

import os
import shutil
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libslamrs_gpu.so")
SOURCES = ["kernels_likelihood.cu", "kernels_ray.cu", "kernels_resample.cu", "kernels_copy.cu", "kernels_misc.cu",
           "kernels_localize.cu", "kernels_cluster.cu", "kernels_scan_match.cu", "comm.cu", "api.cu"]
HEADERS = ["kernels.cuh", "kernels_common.cuh", "slam_device.cuh", "libm_f32.cuh", "shared_stream.cuh", "comm.h",
           os.path.join("..", "..", "include", "slamrs_gpu.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",   # B200 only, no PTX for other archs
    "-O3", "-lineinfo", "-std=c++17",
    "-fmad=false",                                  # rustc never contracts a*b+c; neither may we
    "-Xcompiler", "-fPIC", "-shared",
]


def nvcc_path() -> str:
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: the slamrs_b200 CUDA library cannot be built")


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False, defines: tuple = (), out: str = LIB) -> str:
    """`defines` / `out`: tuning variants (tools/tune_variants.sh); the product library takes neither."""
    if not force and not needs_build():
        return LIB
    cmd = [nvcc_path()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-D" + d for d in defines] + \
          ["-o", out] + [os.path.join(CSRC, s) for s in SOURCES] + ["-ldl"]
    env = dict(os.environ)
    env.pop("CC", None); env.pop("CXX", None)   # the image's CC wrapper is not a usable nvcc host compiler
    res = subprocess.run(cmd, cwd=HERE, env=env, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
    if verbose:
        print(res.stdout + res.stderr)
    return LIB


if __name__ == "__main__":
    import sys
    defs = tuple(a[2:] for a in sys.argv[1:] if a.startswith("-D"))
    outs = [a[6:] for a in sys.argv[1:] if a.startswith("--out=")]
    print(build(force="--force" in sys.argv or bool(defs or outs), verbose="-v" in sys.argv, defines=defs,
                out=outs[0] if outs else LIB))
