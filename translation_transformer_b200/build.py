"""Build libttb200.so in-tree with nvcc for sm_100a (no JIT cache: the .so travels with the repo)."""
from __future__ import annotations

import os
import subprocess
import sys
from pathlib import Path

CSRC = Path(__file__).resolve().parent / "csrc"
LIB = Path(__file__).resolve().parent / "libttb200.so"
SOURCES = ["elementwise.cu", "gemm_simt.cu", "gemm_tcgen05.cu", "attention.cu", "attention_mma.cu", "drafting.cu", "greedy.cu", "beam.cu", "std_beam.cu", "scoring.cu", "sampling.cu", "engine.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr"]


def _stale() -> bool:
    if not LIB.exists():
        return True
    t = LIB.stat().st_mtime
    deps = list(CSRC.glob("*.cu")) + list(CSRC.glob("*.cuh")) + [CSRC.parent.parent / "include" / "ttb200.h"]
    return any(p.stat().st_mtime > t for p in deps)


def build(force: bool = False, verbose: bool = False) -> Path:
    if not force and not _stale():
        return LIB
    nvcc = os.environ.get("NVCC", "nvcc")
    objs = []
    procs = []
    out_dir = CSRC / "build"
    out_dir.mkdir(exist_ok=True)
    for src in SOURCES:
        obj = out_dir / (src + ".o")
        cmd = [nvcc, *NVCC_FLAGS, *os.environ.get("TTB_NVCC_EXTRA", "").split(), "-c", str(CSRC / src), "-o", str(obj)]
        if verbose:
            print(" ".join(cmd))
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(str(obj))
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            failed = True
            print(f"nvcc failed for {src}:\n{out}", file=sys.stderr)
        elif verbose and out.strip():
            print(out)
    if failed:
        raise RuntimeError("libttb200 build failed")
    cmd = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", str(LIB), *objs, "-lcudart"]
    subprocess.run(cmd, check=True)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
