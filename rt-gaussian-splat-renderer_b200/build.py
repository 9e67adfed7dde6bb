"""Build librtgs_b200.so (the C-ABI CUDA library) in-tree with nvcc for sm_100a.

    python rt-gaussian-splat-renderer_b200/build.py [--force] [--verbose]

nvcc cross-compiles without a GPU.  The .so lands in rt-gaussian-splat-renderer_b200/lib/ (git-ignored,
but shipped to the GPU box by gpurun).  Rebuilds only when a source is newer than the library.
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

HERE = Path(__file__).resolve().parent
CSRC = HERE / "csrc"
LIBDIR = HERE / "lib"
LIB = LIBDIR / os.environ.get("RTGS_LIB_NAME", "librtgs_b200.so")
SOURCES = ["abi.cu", "lbvh.cu", "render.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC",
    "-Xptxas", "-v",
] + os.environ.get("RTGS_NVCC_EXTRA", "").split()


def _stale() -> bool:
    if not LIB.exists():
        return True
    t = LIB.stat().st_mtime
    deps = list(CSRC.glob("*.cu")) + list(CSRC.glob("*.cuh")) + [HERE.parent / "include" / "rtgs_b200.h",
                                                                  Path(__file__)]
    return any(p.stat().st_mtime > t for p in deps)


def build(force: bool = False, verbose: bool = False) -> Path:
    if not force and not _stale():
        return LIB
    LIBDIR.mkdir(exist_ok=True)
    objdir = HERE / "build"
    objdir.mkdir(exist_ok=True)

    def compile_one(src: str):
        obj = objdir / (src + ".o")
        cmd = [NVCC, *FLAGS, "-c", str(CSRC / src), "-o", str(obj)]
        r = subprocess.run(cmd, capture_output=True, text=True)
        return src, obj, r

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        results = list(ex.map(compile_one, SOURCES))
    log = []
    for src, obj, r in results:
        log.append(f"==== {src}\n{r.stdout}{r.stderr}")
        if r.returncode != 0:
            bad = [l for l in (r.stdout + r.stderr).splitlines() if not l.startswith("ptxas info") and l.strip()]
            sys.stderr.write(f"==== {src}\n" + "\n".join(bad[-60:]) + "\n")
            raise RuntimeError(f"nvcc failed on {src}")
    (objdir / "ptxas.log").write_text("\n".join(log))
    if verbose:
        print("\n".join(log))
    cmd = [NVCC, "-shared", "-o", str(LIB), *[str(o) for _, o, _ in results],
           "-gencode", "arch=compute_100a,code=sm_100a"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("link failed")
    return LIB


if __name__ == "__main__":
    p = build(force="--force" in sys.argv, verbose="--verbose" in sys.argv)
    print(p)
