"""In-tree nvcc build of libp3tok.so (sm_100a only).  The built library is git-ignored but
travels to the GPU box with the gpurun snapshot; nothing is JIT-compiled at run time."""
from __future__ import annotations

import concurrent.futures as cf
import os
import shutil
import subprocess
from typing import List

_PKG = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(os.path.dirname(_PKG))
CSRC = os.path.join(os.path.dirname(_PKG), "csrc")
INCLUDE = os.path.join(_ROOT, "include")
LIB_PATH = os.path.join(_PKG, "libp3tok.so")
OBJ_DIR = os.path.join(CSRC, "_obj")

SOURCES = ["capi.cu", "fps.cu", "fps_nd.cu", "sqdist.cu", "knn.cu", "group.cu", "mlp_f32.cu", "embed_tc.cu", "embed_fused.cu", "embed_stage.cu", "embed_gather.cu", "vit.cu", "train.cu", "train_vit.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "--expt-extended-lambda", "--expt-relaxed-constexpr", "-Xcompiler", "-fPIC",
    "-Xcompiler", "-fvisibility=hidden", "-I", INCLUDE, "-I", CSRC,
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.isfile(cand):
            return cand
    raise RuntimeError("nvcc not found; libp3tok.so must be built where the CUDA toolkit is installed")


def _newer(target: str, deps: List[str]) -> bool:
    if not os.path.isfile(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build_library(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(OBJ_DIR, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    headers += [os.path.join(INCLUDE, f) for f in os.listdir(INCLUDE)]
    nvcc = _nvcc()
    jobs = []
    objs = []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(OBJ_DIR, src.replace(".cu", ".o"))
        objs.append(o)
        if force or _newer(o, [s] + headers):
            jobs.append([nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", s, "-o", o])

    def run(cmd):
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + r.stdout + r.stderr)
        return r.stderr

    if jobs:
        with cf.ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 1)) as ex:
            for out in ex.map(run, jobs):
                if verbose and out:
                    print(out)
    if jobs or force or _newer(LIB_PATH, objs):
        run([nvcc, "-shared", "-o", LIB_PATH] + objs + ["-gencode", "arch=compute_100a,code=sm_100a"])
    return LIB_PATH


if __name__ == "__main__":
    import sys
    print(build_library(force="--force" in sys.argv, verbose="-v" in sys.argv))
