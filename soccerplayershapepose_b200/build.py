"""In-tree build of libb200smpl.so (hand-written CUDA for sm_100a, C-ABI in include/b200smpl.h).

nvcc cross-compiles without a GPU, so this runs in the build container; the resulting .so is
git-ignored but travels to the GPU box with the repo snapshot.  No JIT, no torch extension
machinery: plain `nvcc -c` per translation unit + one `nvcc -shared` link.
"""
from __future__ import annotations

import concurrent.futures
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
BUILD = os.path.join(HERE, "csrc", "build")
LIB = os.path.join(HERE, "libb200smpl.so")

SOURCES = ["api.cu", "pack.cu", "pose.cu", "blend_simt.cu", "blend_umma.cu", "fused_fwd.cu", "lbs.cu", "joints.cu", "aux_ops.cu", "fit.cu", "loss.cu"]
HEADERS = [os.path.join(CSRC, h) for h in sorted(os.listdir(CSRC)) if h.endswith(".cuh")] + [
    os.path.join(HERE, "..", "include", "b200smpl.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC",
    "-Xcompiler", "-fvisibility=hidden",
    "--expt-relaxed-constexpr",
    "-Xptxas", "-v",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", shutil.which("nvcc")):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found (needed to build libb200smpl.so)")


def _stale(target: str, deps) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build_library(force: bool = False, verbose: bool = False) -> str:
    nvcc = _nvcc()
    os.makedirs(BUILD, exist_ok=True)
    jobs = []
    objs = []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(BUILD, src.replace(".cu", ".o"))
        objs.append(o)
        if force or _stale(o, [s] + HEADERS):
            jobs.append((s, o))

    def compile_one(job):
        s, o = job
        cmd = [nvcc] + NVCC_FLAGS + os.environ.get("B200_NVCC_EXTRA", "").split() + ["-c", s, "-o", o]
        r = subprocess.run(cmd, capture_output=True, text=True)
        log = os.path.join(BUILD, os.path.basename(o) + ".log")
        with open(log, "w") as f:
            f.write(" ".join(cmd) + "\n" + r.stdout + r.stderr)
        return s, r.returncode, r.stdout + r.stderr

    if jobs:
        with concurrent.futures.ThreadPoolExecutor(max_workers=min(8, len(jobs))) as ex:
            for s, rc, out in ex.map(compile_one, jobs):
                if verbose or rc != 0:
                    print(out, file=sys.stderr)
                if rc != 0:
                    raise RuntimeError("nvcc failed on " + s)
    if jobs or force or _stale(LIB, objs):
        cmd = [nvcc, "-shared", "-o", LIB] + objs + ["-cudart", "static", "-gencode",
                                                      "arch=compute_100a,code=sm_100a"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            print(r.stdout + r.stderr, file=sys.stderr)
            raise RuntimeError("link failed")
    return LIB


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose="-v" in sys.argv))
