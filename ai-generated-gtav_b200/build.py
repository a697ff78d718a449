"""Builds libgtav_b200.so in-tree with nvcc for sm_100a (no torch headers, no CUTLASS).

    python ai-generated-gtav_b200/build.py [--force]

The .so is git-ignored but travels to the GPU box with the gpurun snapshot.
"""
from __future__ import annotations

import concurrent.futures
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
BUILD = os.path.join(HERE, "build")
LIB = os.path.join(HERE, "libgtav_b200.so")
SOURCES = ["gemm_sm100.cu", "gemm_sm100_2cta.cu", "gemm_sm100_splitk.cu", "gemm_skinny.cu", "norm_mod.cu", "attn_mma.cu", "attn_tc.cu", "attn_temporal.cu", "attn_temporal_long.cu", "elementwise.cu", "dit_engine.cu",
           "vae_engine.cu", "sampler.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "--cudart", "shared",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden", "-Xptxas", "-v"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", shutil.which("nvcc")):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def _stale(target: str, deps: list[str]) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(BUILD, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".h", ".cuh"))]
    headers.append(os.path.join(os.path.dirname(HERE), "include", "gtav_b200.h"))
    nvcc = _nvcc()

    def compile_one(src: str):
        obj = os.path.join(BUILD, src.replace(".cu", ".o"))
        path = os.path.join(CSRC, src)
        if force or _stale(obj, [path] + headers):
            r = subprocess.run([nvcc, *NVCC_FLAGS, "-c", path, "-o", obj], capture_output=True, text=True)
            with open(obj + ".log", "w") as f:
                f.write(r.stdout + r.stderr)
            if r.returncode != 0:
                raise RuntimeError(f"nvcc failed on {src}:\n{r.stdout}\n{r.stderr}")
            if verbose:
                print(r.stderr)
        return obj

    with concurrent.futures.ThreadPoolExecutor(max_workers=min(8, len(SOURCES))) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    if force or _stale(LIB, objs):
        cmd = [nvcc, "-shared", "--cudart", "shared", "-o", LIB, *objs, "-Xlinker", "-rpath=/usr/local/cuda/lib64"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
