"""In-tree build of libneurons_mm.so (sm_100a only) with plain nvcc -- no torch C++ extension, no JIT cache.

    python -m neurons_b200.build [--force] [--verbose]

The shared object lands next to this file (neurons_b200/libneurons_mm.so) so that it travels with the repo
snapshot to the GPU box.  nvcc cross-compiles without a GPU; the CUDA runtime is linked statically and the one
driver entry point the library needs (cuTensorMapEncodeTiled) is resolved at run time through
cudaGetDriverEntryPoint, so the .so also loads on a machine without a driver (symbol-export tests).
"""
from __future__ import annotations

import argparse
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
BUILD = os.path.join(HERE, "build")
LIB = os.path.join(HERE, "libneurons_mm.so")
SOURCES = ["api.cu", "norm_kernels.cu", "attention_kernel.cu", "gemm_simt.cu", "gemm_tcgen05.cu", "sampler_kernels.cu", "fused_module.cu", "spatial_attention.cu", "spatial_attention_tc.cu", "spatial_attention_x3.cu", "spatial_attention_x6.cu", "spatial_attention_f32.cu", "spatial_api.cu", "decoder_attention.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden",
    "--expt-relaxed-constexpr",
]


def find_nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.isfile(cand):
            return cand
    raise RuntimeError("nvcc not found (set NVCC=/path/to/nvcc)")


def _newer(target: str, deps) -> bool:
    if not os.path.isfile(target):
        return False
    t = os.path.getmtime(target)
    return all(os.path.getmtime(d) <= t for d in deps)


def _headers():
    hs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    hs.append(os.path.join(os.path.dirname(HERE), "include", "neurons_mm.h"))
    return hs


def build(force: bool = False, verbose: bool = False, trace: bool = False) -> str:
    """trace=True builds a development variant (libneurons_mm_trace.so, -DNMM_TRACE: per-tile timestamps in the GEMM)."""
    nvcc = find_nvcc()
    global BUILD, LIB
    if trace:
        BUILD, LIB = os.path.join(HERE, "build_trace"), os.path.join(HERE, "libneurons_mm_trace.so")
    os.makedirs(BUILD, exist_ok=True)
    headers = _headers()
    objs, jobs = [], []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(BUILD, src.replace(".cu", ".o"))
        objs.append(o)
        if force or not _newer(o, [s, __file__] + headers):
            cmd = [nvcc] + NVCC_FLAGS + (["-DNMM_TRACE"] if trace else []) + (["-Xptxas", "-v"] if verbose else []) + ["-c", s, "-o", o]
            jobs.append(cmd)

    def run(cmd):
        r = subprocess.run(cmd, capture_output=True, text=True)
        return cmd, r

    if jobs:
        with ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 4)) as ex:
            for cmd, r in ex.map(run, jobs):
                if verbose or r.returncode != 0:
                    sys.stderr.write(" ".join(cmd) + "\n" + r.stdout + r.stderr)
                if r.returncode != 0:
                    raise RuntimeError(f"nvcc failed for {cmd[-3]}")
    if jobs or force or not _newer(LIB, objs):
        cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-cudart", "static", "-o", LIB] + objs
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            sys.stderr.write(" ".join(cmd) + "\n" + r.stdout + r.stderr)
            raise RuntimeError("link failed")
    return LIB


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--force", action="store_true")
    ap.add_argument("--verbose", action="store_true")
    ap.add_argument("--trace", action="store_true")
    a = ap.parse_args()
    print(build(a.force, a.verbose, a.trace))
