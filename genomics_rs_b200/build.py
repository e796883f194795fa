"""Builds libgxalign.so (C ABI + CUDA kernels, sm_100a) in-tree with nvcc.  No torch involved.
The fill kernel is instantiated once per (K, CHAIN1) in its own object so that the objects compile in parallel."""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
# Tagged builds: GX_BUILD_TAG=chk GX_BUILD_DEFS="-DGX_CHECKED" python -m genomics_rs_b200.build  ->  libgxalign_chk.so
TAG = os.environ.get("GX_BUILD_TAG", "")
OBJ = os.path.join(HERE, "csrc", "_obj" + ("_" + TAG if TAG else ""))
OUT = os.path.join(HERE, "libgxalign" + ("_" + TAG if TAG else "") + ".so")
HEADERS = sorted(f for f in os.listdir(CSRC) if f.endswith(".cuh")) + [os.path.join("..", "..", "include", "gxalign.h")]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
CFLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-Xcompiler", "-fPIC"] + os.environ.get("GX_BUILD_DEFS", "").split()
# columns per lane of the fill kernel -- keep in step with GX_COMBOS in csrc/gx_api.cu
COMBOS = [4, 8, 16]
# (object name, source, extra flags)
UNITS = [("gx_api.o", "gx_api.cu", []), ("gx_k0.o", "gx_k0.cu", [])] + [
    (f"gx_fill_k{k}_c{c}.o", "gx_fill_inst.cu", [f"-DGX_INST_K={k}", f"-DGX_INST_CHAIN={c}"])
    for k in COMBOS for c in (0, 1)]


def _newest_header() -> float:
    return max(os.path.getmtime(os.path.join(CSRC, h)) for h in HEADERS)


def stale() -> bool:
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    srcs = {u[1] for u in UNITS}
    return any(os.path.getmtime(os.path.join(CSRC, f)) > t for f in srcs) or _newest_header() > t


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not stale():
        return OUT
    os.makedirs(OBJ, exist_ok=True)
    hdr_t = _newest_header()
    jobs = []
    for obj, src, extra in UNITS:
        o, s = os.path.join(OBJ, obj), os.path.join(CSRC, src)
        if force or not os.path.exists(o) or os.path.getmtime(o) < max(os.path.getmtime(s), hdr_t):
            jobs.append([NVCC] + CFLAGS + (["-Xptxas", "-v"] if verbose else []) + extra + ["-c", "-o", o, s])
    with ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1)) as ex:
        list(ex.map(subprocess.check_call, jobs))
    subprocess.check_call([NVCC, "-shared", "-cudart", "static", "-gencode", "arch=compute_100a,code=sm_100a", "-o", OUT] +
                          [os.path.join(OBJ, u[0]) for u in UNITS])
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
