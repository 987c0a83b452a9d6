"""Build the product library svn_icp_b200/lib/libsvnicp_b200.so for sm_100a with nvcc (in-tree, so the
.so travels to the GPU box with the gpurun snapshot).  `python -m svn_icp_b200.build [--force]`."""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIBDIR, "libsvnicp_b200.so")
SOURCES = ["cand_build.cu", "iter_kernels.cu", "stein_kernels.cu", "tail2.cu", "svgd_class.cu", "eval_kernels.cu", "voxel_map.cu", "preprocess.cu", "capi.cu"]
HEADERS = ["block_scan.cuh", "common.cuh", "kernels.h", "ptx.cuh", "voxel_hash.cuh", os.path.join("..", "..", "include", "svnicp_b200.h")]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
# extra -D switches for A/B builds (e.g. SVNICP_NVCC_DEFS="-DSVN_GN_ACC2_FP32 -DSVN_GN_MINBLOCKS=3")
EXTRA = os.environ.get("SVNICP_NVCC_DEFS", "").split()
FLAGS = EXTRA + ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-Xcompiler", "-fPIC",
         "-ccbin", "/usr/bin/g++", "-I", "/usr/include"]


def _stale(target: str, deps: list[str]) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False, debug_bounds: bool = False) -> str:
    """debug_bounds=True builds lib/libsvnicp_b200_dbg.so with -DSVN_DEBUG_BOUNDS (device-side bounds checks, see common.cuh);
    tests load it through SVNICP_B200_LIB."""
    os.makedirs(LIBDIR, exist_ok=True)
    objdir = os.path.join(LIBDIR, "obj_dbg" if debug_bounds else "obj")
    lib = LIB.replace(".so", "_dbg.so") if debug_bounds else LIB
    flags = FLAGS + (["-DSVN_DEBUG_BOUNDS"] if debug_bounds else [])
    os.makedirs(objdir, exist_ok=True)
    hdrs = [os.path.join(CSRC, h) for h in HEADERS]
    objs, procs = [], []
    for s in SOURCES:
        src = os.path.join(CSRC, s)
        obj = os.path.join(objdir, s.replace(".cu", ".o"))
        objs.append(obj)
        if force or _stale(obj, [src] + hdrs):
            cmd = [NVCC] + flags + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj]
            procs.append((s, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for name, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write(f"--- nvcc {name} ---\n{out}\n")
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed")
    if force or procs or _stale(lib, objs):
        cmd = [NVCC, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", lib] + objs + ["-ldl", "-ccbin", "/usr/bin/g++"]
        subprocess.check_call(cmd)
    return lib


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv, debug_bounds="--debug-bounds" in sys.argv))
