"""Builds libsphmw.so (hand-written CUDA for sm_100a + the C ABI) in-tree with nvcc.

No torch, no JIT cache: the .so lands next to this file so that it travels to the
GPU box with the repo snapshot.  `python -m sph_mountain_waves_b200.build` rebuilds.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

PKG = Path(__file__).resolve().parent
ROOT = PKG.parent
CSRC = PKG / "csrc"
LIB = PKG / "libsphmw.so"

ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
# -fmad=false: the reference (Julia without @fastmath) never contracts a*b+c into
# an FMA; bit-exact neighbour sets and reproducible FP64 sums depend on it.
NVCC_FLAGS = ARCH + ["-O3", "-std=c++17", "-lineinfo", "-fmad=false", "-Xcompiler", "-fPIC,-O2",
                     "-Xcudafe", "--diag_suppress=177", f"-I{ROOT / 'include'}", f"-I{CSRC}"]
SOURCES = ["api.cu", "cell_list.cu", "pair_ops.cu", "halo.cu", "slab_comm.cu", "frame_async.cu", "lattice.cu", "point_sum.cu", "frame_io.cpp", "grid_setup.cpp"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and Path(cand).exists():
            return cand
    raise RuntimeError("nvcc not found; libsphmw cannot be built (there is no CPU fallback)")


def _stale(target: Path, deps) -> bool:
    if not target.exists():
        return True
    t = target.stat().st_mtime
    return any(Path(d).stat().st_mtime > t for d in deps)


def build_lib(force: bool = False, verbose: bool = False) -> Path:
    nvcc = _nvcc()
    headers = list(CSRC.glob("*.h")) + list(CSRC.glob("*.cuh")) + [ROOT / "include" / "sphmw.h"]
    objdir = PKG / "build"
    objdir.mkdir(exist_ok=True)
    env = dict(os.environ)
    ccbin = "/usr/bin/g++" if Path("/usr/bin/g++").exists() else shutil.which("g++")

    def compile_one(src: str) -> Path:
        obj = objdir / (src.rsplit(".", 1)[0] + ".o")
        if force or _stale(obj, [CSRC / src, Path(__file__)] + headers):
            cmd = [nvcc, "-ccbin", ccbin] + NVCC_FLAGS + ["-c", str(CSRC / src), "-o", str(obj)]
            if verbose:
                cmd.insert(1, "-Xptxas=-v")
            r = subprocess.run(cmd, capture_output=True, text=True, env=env)
            if verbose or r.returncode != 0:
                sys.stderr.write(r.stdout + r.stderr)
            if r.returncode != 0:
                raise RuntimeError(f"nvcc failed on {src}")
        return obj

    with ThreadPoolExecutor(max_workers=4) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    if force or _stale(LIB, objs):
        cmd = [nvcc, "-ccbin", ccbin, "-shared"] + ARCH + ["-o", str(LIB)] + [str(o) for o in objs] + \
              ["-lcudart", "-lz", "-ldl"]
        r = subprocess.run(cmd, capture_output=True, text=True, env=env)
        if r.returncode != 0:
            sys.stderr.write(r.stdout + r.stderr)
            raise RuntimeError("link of libsphmw.so failed")
    return LIB


if __name__ == "__main__":
    p = build_lib(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print(p)
