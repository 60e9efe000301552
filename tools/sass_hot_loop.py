#!/usr/bin/env python
"""Shape of a packed ray kernel's free-run loop in the built library's SASS (no GPU needed).

    python tools/sass_hot_loop.py [slamrs_b200/libslamrs_gpu.so] [k_ray_update_packed | k_ray_update_half] [-v]

The walk both packed kernels share (ray_walk_packed) spends its time in one loop: classify the cell, one
shared-memory add, one step of the reference's ray iterator. ptxas compiles it to a single predicated block of 25
instructions -- or, after changes elsewhere in the kernel, to a branchy form that rebuilds the row table's shared
address inside the loop (S2UR + ULEA per y-step, 31 instructions, +15 % kernel time measured on B200). This script
takes the smallest loop around an ATOMS.ADD whose body contains an FMUL -- the tested free run recomputes dx^2 or
dy^2 at every step; the test-free loop over the first cells of a walk has no distance arithmetic -- and prints its
size and whether it contains an S2UR or local memory; tests/test_abi_and_host.py fails the build on the slow form."""
import re
import subprocess
import sys

KERNELS = ("k_ray_update_packed", "k_ray_update_half")


def opcode(text):
    """mnemonic of one SASS instruction, without its predicate guard"""
    return re.sub(r"^@!?U?P\w+\s+", "", text).split()[0]


def hot_loop(lib, kernel="k_ray_update_packed"):
    out = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout
    lines = out.split("\n")
    mangled = "_ZN6slamrs%d%s" % (len(kernel), kernel)
    start = next(i for i, l in enumerate(lines) if "Function : " + mangled in l)
    end = next((i for i, l in enumerate(lines[start + 1:], start + 1) if "Function :" in l), len(lines))
    ins = []
    for l in lines[start:end]:
        m = re.match(r"\s*/\*([0-9a-f]+)\*/\s+(.*?);", l)
        if m:
            ins.append((int(m.group(1), 16), m.group(2).strip()))
    loops = []   # (first, last) addresses of every backward branch's body
    for a, t in ins:
        m = re.search(r"BRA\S*\s+(?:\S+,\s*)?0x([0-9a-f]+)", t)
        if m and int(m.group(1), 16) <= a:
            loops.append((int(m.group(1), 16), a))
    best = None
    for lo, hi in loops:
        body = [(a, t) for a, t in ins if lo <= a <= hi]
        ops = [opcode(t) for _, t in body]
        if any(o.startswith("ATOMS.ADD") for o in ops) and any(o.startswith("FMUL") for o in ops):
            if best is None or len(body) < len(best):
                best = body
    if best is None:
        raise RuntimeError("no loop around an ATOMS.ADD with an FMUL in " + kernel)
    ops = [opcode(t) for _, t in best]
    return {"instructions": len(best), "s2ur": any(o.startswith("S2UR") for o in ops),
            "local_memory": any(o.startswith(("LDL", "STL")) for o in ops), "body": best}


if __name__ == "__main__":
    args = [a for a in sys.argv[1:] if not a.startswith("-")]
    lib = next((a for a in args if a.endswith(".so")), "slamrs_b200/libslamrs_gpu.so")
    kernels = [a for a in args if a in KERNELS] or list(KERNELS)
    for k in kernels:
        r = hot_loop(lib, k)
        print(k, {key: v for key, v in r.items() if key != "body"})
        if "-v" in sys.argv:
            for a, t in r["body"]:
                print(f"{a:06x}  {t}")
