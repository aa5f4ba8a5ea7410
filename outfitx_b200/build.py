"""Builds ``outfitx_b200/libofx.so`` (the C-ABI CUDA library, sm_100a only) in-tree with nvcc.

    python -m outfitx_b200.build [--force] [-v] [--debug]

``--debug`` builds the INSTRUMENTED library ``libofx_debug.so`` (``-DOFX_DEBUG``: role-cycle counters and
timing experiments that allocate, synchronise or skip work -- none of that exists in the product library);
load it with ``OFX_LIB_PATH=outfitx_b200/libofx_debug.so``.

nvcc cross-compiles without a GPU, so this runs in the build container; the built ``.so`` is
git-ignored but travels to the GPU box with the repo snapshot.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "build")
LIB = os.path.join(HERE, "libofx.so")
SOURCES = ["common.cu", "gemm.cu", "encoder_ops.cu", "encoder.cu", "search.cu", "ffn_block.cu", "pool_search.cu", "losses.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found (set NVCC or put it on PATH)")


def _deps() -> list[str]:
    out = [os.path.join(HERE, "..", "include", "ofx.h")]
    for f in os.listdir(CSRC):
        out.append(os.path.join(CSRC, f))
    return out


def up_to_date() -> bool:
    if not os.path.exists(LIB):
        return False
    t = os.path.getmtime(LIB)
    return all(os.path.getmtime(d) <= t for d in _deps() if os.path.exists(d))


def build(force: bool = False, verbose: bool = False, debug: bool = False) -> str:
    if not debug and not force and up_to_date():
        return LIB
    nvcc = _nvcc()
    obj_dir = OBJ + ("_debug" if debug else "")
    lib = LIB.replace("libofx.so", "libofx_debug.so") if debug else LIB
    os.makedirs(obj_dir, exist_ok=True)

    def compile_one(src: str) -> str:
        obj = os.path.join(obj_dir, src.replace(".cu", ".o"))
        cmd = [nvcc, *NVCC_FLAGS, *(["-DOFX_DEBUG"] if debug else []), "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            print(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    tmp = lib + ".tmp"
    r = subprocess.run([nvcc, "-shared", "-o", tmp, *objs, "-gencode", "arch=compute_100a,code=sm_100a",
                        "-cudart", "static"], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    os.replace(tmp, lib)
    return lib


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv, debug="--debug" in sys.argv))
