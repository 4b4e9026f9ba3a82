"""In-tree build of the C-ABI library `libsmt_b200.so` for sm_100a.

`nvcc` cross-compiles without a GPU; the resulting `.so` is git-ignored but travels to the GPU box with
the repo snapshot.  Objects are rebuilt only when a source (or header) is newer than the library.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT_DIR = os.path.join(HERE, "_C")
LIB_PATH = os.path.join(OUT_DIR, "libsmt_b200.so")
SOURCES = ["capi.cu", "score_kernels.cu", "topk_kernel.cu", "block_copy_kernels.cu", "channel_kernels.cu", "adam_kernels.cu",
           "block_grad_gemm.cu", "block_grad_runs.cu", "dense_gemm.cu", "decoder_kernels.cu", "loss_kernels.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; cannot build libsmt_b200.so")


def _deps() -> list[str]:
    files = [os.path.join(CSRC, s) for s in SOURCES]
    files += [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    files.append(os.path.join(HERE, "..", "include", "smt_b200.h"))
    return files


def needs_build() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    return any(os.path.getmtime(f) > t for f in _deps())


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every .cu under csrc/ for sm_100a and link libsmt_b200.so. Returns its path."""
    if not force and not needs_build():
        return LIB_PATH
    nvcc = _nvcc()
    os.makedirs(OUT_DIR, exist_ok=True)
    obj_dir = os.path.join(OUT_DIR, "obj")
    os.makedirs(obj_dir, exist_ok=True)

    def compile_one(src: str) -> str:
        obj = os.path.join(obj_dir, src.replace(".cu", ".o"))
        cmd = [nvcc, *NVCC_FLAGS, *os.environ.get("SMT_NVCC_EXTRA", "").split(), "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            sys.stderr.write(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=min(8, len(SOURCES))) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    tmp = LIB_PATH + ".tmp"
    r = subprocess.run([nvcc, "-shared", "-o", tmp, *objs, "-gencode", "arch=compute_100a,code=sm_100a",
                        "-cudart", "static", "-Xlinker", "--exclude-libs,ALL"], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    os.replace(tmp, LIB_PATH)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
