"""In-tree build of libtmae_b200.so (sm_100a only).  nvcc cross-compiles without a GPU.

    python -m textmae_image_compression_b200.build [--force]
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

PKG = Path(__file__).resolve().parent
CSRC = PKG / "csrc"
LIB = PKG / "libtmae_b200.so"
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden"]
# mask.cu restates fp32 ATen CPU arithmetic bit for bit: no implicit FMA contraction there.
SOURCES = {
    "gemm_tc.cu": [],
    "attention.cu": [],
    "elementwise.cu": [],
    "mask.cu": ["-fmad=false"],
    "scores.cu": ["-fmad=false"],
    "rans.cu": [],
    "container.cu": [],
    "picture.cu": [],
    "huffman.cpp": [],
    "tmae_api.cu": [],
}


def _stale(target: Path, deps) -> bool:
    if not target.exists():
        return True
    t = target.stat().st_mtime
    return any(Path(d).stat().st_mtime > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> Path:
    headers = list(CSRC.glob("*.cuh")) + list(CSRC.glob("*.h")) + [PKG.parent / "include" / "tmae.h"]
    obj_dir = CSRC / "_obj"
    obj_dir.mkdir(exist_ok=True)
    jobs = []
    for src, extra in SOURCES.items():
        obj = obj_dir / (src + ".o")
        if force or _stale(obj, [CSRC / src] + headers):
            cmd = [NVCC] + ARCH + COMMON + extra + ["-c", str(CSRC / src), "-o", str(obj)]
            jobs.append(cmd)
    def run(cmd):
        if verbose:
            print(" ".join(cmd), flush=True)
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed: {' '.join(cmd)}\n{r.stdout}\n{r.stderr}")
        return r
    if jobs:
        with ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 1)) as ex:
            list(ex.map(run, jobs))
    objs = [str(obj_dir / (s + ".o")) for s in SOURCES]
    if force or jobs or _stale(LIB, objs):
        run([NVCC] + ARCH + ["-shared", "-Xcompiler", "-fPIC", "-o", str(LIB)] + objs + ["-cudart", "static"])
    return LIB


if __name__ == "__main__":
    p = build(force="--force" in sys.argv, verbose=True)
    print(p)
