"""Builds bpl_next_b200/lib/libbplx.so (nvcc, sm_100a only) -- in-tree, so it travels with the repo."""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "lib", "libbplx.so")
SOURCES = ["api.cu", "logdensity.cu", "logdensity_dynamic.cu", "score_grid.cu", "loo.cu", "markets.cu", "simulate.cu", "simulate_cond.cu", "ppc.cu", "dynamic_predict.cu", "nuts.cu", "peer_sum.cu", "plan.cc"]
HEADERS = ["common.cuh", "k1_common.cuh", "plan.h", "plan_dynamic.inc", "problem.h", "score_grid.h", "loo.h", "markets.h", "radix_select.cuh", "simulate.h", "simulate_body.inc", "simulate_device.cuh", "sample_score.cuh", "ppc.h", "dynamic_predict.h", "nuts.h", os.path.join("..", "..", "include", "bplx_nuts.h"), os.path.join("..", "..", "include", "bplx.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared"]


def _stale() -> bool:
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    return any(os.path.getmtime(os.path.join(CSRC, f)) > t for f in SOURCES + HEADERS)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not _stale():
        return OUT
    os.makedirs(os.path.dirname(OUT), exist_ok=True)
    nvcc = os.environ.get("NVCC", "nvcc")
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", OUT] + SOURCES
    r = subprocess.run(cmd, cwd=CSRC, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("nvcc failed building libbplx.so")
    if verbose:
        sys.stderr.write(r.stderr)
    return OUT


BENCH_SRC = os.path.join(HERE, "..", "bench_kernels", "fp32_peak.cu")
BENCH_OUT = os.path.join(HERE, "lib", "libbplx_bench.so")


def build_bench(force: bool = False) -> str:
    """Measurement helper for bench.py (FFMA / shared-memory peaks); not part of the product."""
    if not force and os.path.exists(BENCH_OUT) and os.path.getmtime(BENCH_OUT) >= os.path.getmtime(BENCH_SRC):
        return BENCH_OUT
    os.makedirs(os.path.dirname(BENCH_OUT), exist_ok=True)
    nvcc = os.environ.get("NVCC", "nvcc")
    r = subprocess.run([nvcc] + NVCC_FLAGS + ["-o", BENCH_OUT, BENCH_SRC], capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("nvcc failed building libbplx_bench.so")
    return BENCH_OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
    print(build_bench(force="--force" in sys.argv))
