"""Builds gp_b200/lib/libgpb200.so (hand-written CUDA for sm_100a + the C ABI) with nvcc, in-tree.

nvcc cross-compiles without a GPU, so this runs in the build container; the .so travels to the GPU
box with the gpurun snapshot (it is git-ignored, not gpurun-ignored).
"""
from __future__ import annotations

import concurrent.futures as cf
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
TAG = os.environ.get("GPB_BUILD_TAG", "")            # experiment builds: libgpb200_<tag>.so with extra -D flags
SO = os.path.join(LIBDIR, "libgpb200%s.so" % ("_" + TAG if TAG else ""))
EXTRA = os.environ.get("GPB_EXTRA_NVCC", "").split()
SOURCES = ["gemm.cu", "panel.cu", "gram.cu", "solve.cu", "engine.cu", "api_core.cu", "api_gp.cu", "api_mg.cu", "rng.cu", "api_sample.cu", "small.cu", "api_latent.cu"]
HEADERS = ["common.cuh", "gemm_tile_body.cuh", "gram.cuh", "host.cuh", "fastexp.cuh", "panel_ll.cuh", os.path.join("..", "..", "include", "gpb200.h")]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
         "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden", "--expt-relaxed-constexpr"]


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(LIBDIR, exist_ok=True)
    objdir = os.path.join(LIBDIR, "obj" + ("_" + TAG if TAG else ""))
    os.makedirs(objdir, exist_ok=True)
    hdrs = [os.path.join(CSRC, h) for h in HEADERS]
    jobs = []
    for s in SOURCES:
        src = os.path.join(CSRC, s)
        obj = os.path.join(objdir, s.replace(".cu", ".o"))
        if force or _stale(obj, [src] + hdrs):
            jobs.append((src, obj))

    def compile_one(job):
        src, obj = job
        cmd = [NVCC] + FLAGS + EXTRA + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        return job, r

    with cf.ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        for job, r in ex.map(compile_one, jobs):
            if verbose or r.returncode != 0:
                sys.stderr.write(r.stdout + r.stderr)
            if r.returncode != 0:
                raise RuntimeError("nvcc failed for %s" % job[0])
    objs = [os.path.join(objdir, s.replace(".cu", ".o")) for s in SOURCES]
    if force or jobs or _stale(SO, objs):
        cmd = [NVCC, "-shared", "-o", SO] + objs + ["-gencode", "arch=compute_100a,code=sm_100a"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            sys.stderr.write(r.stdout + r.stderr)
            raise RuntimeError("link failed")
    return SO


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
