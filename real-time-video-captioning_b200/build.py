"""In-tree nvcc build of libgitb200.so (sm_100a only).  No torch dependency: the library is a plain
C-ABI shared object loaded with ctypes (include/gitb200.h).  Run as a script or call build()."""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
ROOT = os.path.dirname(HERE)
OBJ_DIR = os.path.join(ROOT, "build", "obj")
LIB_PATH = os.path.join(HERE, "libgitb200.so")
SOURCES = ["gemm_tcgen05.cu", "gemm2_tcgen05.cu", "gemv_skinny.cu", "elementwise.cu", "attention.cu", "attention_tc.cu", "search.cu", "decode_mega.cu", "preprocess.cu", "student.cu", "student_train.cu", "api.cu"]
HEADERS = ["common.cuh", "kernels.h", "student_ops.h", "student_internal.cuh", "search_step.cuh", "philox.cuh", "text_attention_dev.cuh", os.path.join("..", "..", "include", "gitb200.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC",
              "-DGITB200_BUILD"]


def _nvcc() -> str:
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found: cannot build libgitb200.so")
    return nvcc


def _digest() -> str:
    h = hashlib.sha256()
    for f in SOURCES + HEADERS:
        with open(os.path.join(CSRC, f), "rb") as fh:
            h.update(fh.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every .cu for sm_100a and link libgitb200.so next to this file.  Returns its path."""
    os.makedirs(OBJ_DIR, exist_ok=True)
    stamp = os.path.join(OBJ_DIR, "digest.txt")
    digest = _digest()
    if not force and os.path.exists(LIB_PATH) and os.path.exists(stamp) and open(stamp).read() == digest:
        return LIB_PATH
    nvcc = _nvcc()

    def compile_one(src: str) -> str:
        obj = os.path.join(OBJ_DIR, src.replace(".cu", ".o"))
        cmd = [nvcc, *NVCC_FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            sys.stderr.write(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    r = subprocess.run([nvcc, "-shared", "-o", LIB_PATH, *objs, "-gencode", "arch=compute_100a,code=sm_100a"],
                       capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    with open(stamp, "w") as fh:
        fh.write(digest)
    return LIB_PATH


def build_test_gemm() -> str:
    """Standalone tcgen05 GEMM bring-up binary (tests/cuda/test_gemm.cu)."""
    out = os.path.join(ROOT, "build", "test_gemm")
    os.makedirs(os.path.dirname(out), exist_ok=True)
    cmd = [_nvcc(), "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-o", out,
           os.path.join(ROOT, "tests", "cuda", "test_gemm.cu"), os.path.join(CSRC, "gemm_tcgen05.cu"), os.path.join(CSRC, "gemm2_tcgen05.cu"), os.path.join(CSRC, "gemv_skinny.cu"),
           os.path.join(ROOT, "tests", "cuda", "note_launch_stub.cu")]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"nvcc failed for test_gemm:\n{r.stdout}\n{r.stderr}")
    return out


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
