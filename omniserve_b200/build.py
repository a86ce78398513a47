"""Build libomniserve_b200.so (all hand-written sm_100a kernels + the C ABI) in-tree with nvcc.

    python -m omniserve_b200.build [--force]

Output: omniserve_b200/lib/libomniserve_b200.so (git-ignored; travels to the GPU box with gpurun).
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, os.environ.get("OB_BUILD_LIBDIR", "lib"))     # e.g. lib_timing for an instrumented variant (OB_LIB_PATH)
LIB = os.path.join(LIBDIR, "libomniserve_b200.so")
SOURCES = ["w4a8_gemm.cu", "w4a8_gemm_decode.cu", "w8a8_gemm.cu", "small_ops.cu", "kv4_attention.cu", "lserve_ops.cu", "prefill_attention.cu",
           "moe_ops.cu", "c_api.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "--compiler-options", "-fPIC", "-Xptxas", "-v",
] + (["-DOB_GEMM_TIMING"] if os.environ.get("OB_GEMM_TIMING") == "1" else []) + (
    ["-DOB_DEC_TIMING"] if os.environ.get("OB_DEC_TIMING") == "1" else []) + (
    ["-DOB_ATT_TIMING"] if os.environ.get("OB_ATT_TIMING") == "1" else []) + (
    [f"-DOB_DEC_KPS={os.environ['OB_DEC_KPS']}"] if os.environ.get("OB_DEC_KPS") else []) + (
    ["-DOB_DEC_WAIT_FIRST"] if os.environ.get("OB_DEC_WAIT_FIRST") == "1" else [])  # per-role wait counters (tools/gemm_waits.py)


def _newest_src() -> float:
    t = os.path.getmtime(os.path.join(HERE, "..", "include", "omniserve_b200.h"))
    for f in os.listdir(CSRC):
        t = max(t, os.path.getmtime(os.path.join(CSRC, f)))
    return t


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(LIBDIR, exist_ok=True)
    srcs = [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    if not force and os.path.exists(LIB) and os.path.getmtime(LIB) >= _newest_src():
        return LIB
    objdir = os.path.join(LIBDIR, "obj")
    os.makedirs(objdir, exist_ok=True)

    def cc(src):
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        cmd = ["nvcc", "-c", os.path.join(CSRC, src), "-o", obj] + NVCC_FLAGS
        r = subprocess.run(cmd, capture_output=True, text=True)
        return src, obj, r

    with ThreadPoolExecutor(4) as ex:
        results = list(ex.map(cc, srcs))
    objs = []
    for src, obj, r in results:
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stderr[-6000:]}")
        if verbose:
            print(r.stderr)
        objs.append(obj)
    r = subprocess.run(["nvcc", "-shared", "-cudart", "shared", "-o", LIB] + objs, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stderr[-4000:]}")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
