"""Build libemojivoice_b200.so in-tree with nvcc for sm_100a (no torch extension machinery, no JIT cache).

    python -m emojivoice_b200.build [--force]

The shared object lands in emojivoice_b200/lib/ (git-ignored, shipped to the GPU box by gpurun).
"""
from __future__ import annotations

import concurrent.futures as cf
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "build")
LIBDIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIBDIR, "libemojivoice_b200.so")
SOURCES = ["api.cu", "weights.cu", "conv_simt.cu", "conv_tc.cu", "resblock_tc.cu", "elementwise.cu", "attention.cu", "attention_tc.cu", "attention_enc_tc.cu", "align.cu",
           "matcha.cu", "hifigan.cu", "denoiser.cu", "mas.cu", "ragged.cu", "ff_tc.cu", "resnet_tc.cu", "train_forward.cu",
           "noise.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC",
              "-Xcompiler", "-fvisibility=hidden", "--expt-relaxed-constexpr"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def _stale(target: str, deps: list[str]) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(OBJ, exist_ok=True)
    os.makedirs(LIBDIR, exist_ok=True)
    nvcc = _nvcc()
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    headers.append(os.path.join(os.path.dirname(HERE), "include", "emojivoice_b200.h"))
    jobs = []
    for src in SOURCES:
        s, o = os.path.join(CSRC, src), os.path.join(OBJ, src.replace(".cu", ".o"))
        if force or _stale(o, [s] + headers):
            jobs.append((s, o))

    def compile_one(job):
        s, o = job
        cmd = [nvcc, *NVCC_FLAGS, *os.environ.get("EV_NVCC_EXTRA", "").split(), "-c", s, "-o", o]   # e.g. EV_NVCC_EXTRA=-DEV_RB_TRACE
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {s}:\n{r.stdout}\n{r.stderr}")
        if verbose and r.stderr.strip():
            print(r.stderr, file=sys.stderr)
        return o

    if jobs:
        with cf.ThreadPoolExecutor(max_workers=min(8, len(jobs))) as ex:
            list(ex.map(compile_one, jobs))
    objs = [os.path.join(OBJ, s.replace(".cu", ".o")) for s in SOURCES]
    if force or jobs or _stale(LIB, objs):
        cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB, *objs, "-cudart", "static"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
