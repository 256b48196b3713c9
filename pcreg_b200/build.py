"""Builds libpcreg_b200.so (hand-written CUDA for sm_100a + the C ABI of include/pcreg.h) in-tree.

    python -m pcreg_b200.build            # incremental
    python -m pcreg_b200.build --force

nvcc cross-compiles without a GPU.  The .so is git-ignored but travels to the GPU box with gpurun.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
# PCREG_LIB_OUT / PCREG_NVCC_EXTRA: build a VARIANT of the library (other output file, extra nvcc flags such as -DUPD_THREADS_OVERRIDE=384)
# for same-session A/B timing with PCREG_LIB=<variant>; the default build ignores both
LIB = os.environ.get("PCREG_LIB_OUT") or os.path.join(HERE, "libpcreg_b200.so")
OBJDIR = os.path.join(HERE, "build" if not os.environ.get("PCREG_LIB_OUT") else "build_" + os.path.basename(os.environ["PCREG_LIB_OUT"]))
SOURCES = ["model.cu", "nn_brute.cu", "nn_grid.cu", "nn_vox.cu", "icp.cu", "icp_fused.cu", "normals.cu", "kabsch_ransac.cu", "align.cu", "local_points.cu", "descriptor.cu", "match.cu"]
HEADERS = ["pcreg_internal.h", "pcreg_dev.cuh", "pcreg_math.cuh", "pcreg_select.cuh", "pcreg_grid.cuh", "pcreg_vox.cuh", "pcreg_icp.cuh", os.path.join("..", "..", "include", "pcreg.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC"] + os.environ.get("PCREG_NVCC_EXTRA", "").split()


def _nvcc() -> str:
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: libpcreg_b200.so cannot be built (there is no CPU fallback)")


def _newest(paths):
    return max(os.path.getmtime(p) for p in paths)


def build_library(force: bool = False, verbose: bool = False) -> str:
    srcs = [os.path.join(CSRC, s) for s in SOURCES]
    hdrs = [os.path.join(CSRC, h) for h in HEADERS]
    if not force and os.path.exists(LIB) and os.path.getmtime(LIB) >= _newest(srcs + hdrs):
        return LIB
    nvcc = _nvcc()
    os.makedirs(OBJDIR, exist_ok=True)
    hdr_time = _newest(hdrs)

    def compile_one(src):
        obj = os.path.join(OBJDIR, os.path.basename(src).replace(".cu", ".o"))
        if not force and os.path.exists(obj) and os.path.getmtime(obj) >= max(os.path.getmtime(src), hdr_time):
            return obj
        cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s\n%s" % (src, r.stdout, r.stderr))
        if verbose:
            sys.stderr.write(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=min(8, len(srcs))) as ex:
        objs = list(ex.map(compile_one, srcs))
    cmd = [nvcc, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n%s\n%s" % (r.stdout, r.stderr))
    return LIB


def build_hostmath(force: bool = False) -> str:
    """Host-only build of pcreg_math.cuh behind a tiny C ABI (tests/hostmath): lets the CPU test
    suite check the 3x3 SVD / eigen / Kabsch code that the kernels inline, without a GPU."""
    root = os.path.dirname(HERE)
    srcs = [os.path.join(root, "tests", "hostmath", f) for f in ("hostmath.cpp", "hostmath_plane.cpp", "hostmath_gicp.cpp", "hostmath_extrap.cpp", "hostmath_polar.cpp", "hostmath_cov.cpp")]
    out = os.path.join(root, "tests", "hostmath", "libhostmath.so")
    deps = srcs + [os.path.join(CSRC, "pcreg_math.cuh")]
    if not force and os.path.exists(out) and os.path.getmtime(out) >= _newest(deps):
        return out
    cmd = ["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-x", "c++"] + srcs + ["-o", out]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("g++ failed for hostmath:\n%s\n%s" % (r.stdout, r.stderr))
    return out


if __name__ == "__main__":
    f = "--force" in sys.argv
    print(build_library(force=f, verbose="-v" in sys.argv))
    print(build_hostmath(force=f))
