"""Builds and loads the test-only shims over the internal launchers of libgitb200.so: tests/cuda/op_modes.cpp (kernels.h) and
tests/cuda/student_ops.cpp (student_ops.h, the student decoder's kernels).

A shim is host C++ linked against the built library; it compiles no kernel.  The output goes to build/ (a temporary directory
if the tree is read-only), named by a hash of the shim, the headers it includes and the library's directory, so a changed
argument struct or launcher signature rebuilds it."""
import ctypes
import hashlib
import os
import shutil
import subprocess
import tempfile
from ctypes import c_float, c_int, c_longlong, c_void_p

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "real-time-video-captioning_b200")
LIB = os.path.join(PKG, "libgitb200.so")
CSRC = os.path.join(PKG, "csrc")
SRC = os.path.join(ROOT, "tests", "cuda", "op_modes.cpp")
HEADER = os.path.join(CSRC, "kernels.h")
CUDA_INCLUDE = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "include")

P = c_void_p
SIGNATURES = {
    "opm_gemm": (c_int, [P, c_int, P, c_int, c_int, c_int, c_int, P, P, c_int, c_int, c_int, P, c_int, P, c_int, c_int, c_int, c_int,
                         P, P, c_float, P, c_int, P, c_int, c_int, P, c_int, c_int, c_int, c_int, P]),
    "opm_layernorm": (c_int, [P, c_int, c_int, c_int, P, P, c_float, P, c_int, c_int, P, c_int, P, c_int, P, c_int, P, c_int, P]),
    "opm_text_attention": (c_int, [P, c_int, c_int, c_int, c_int, P, c_int, c_int, c_int, c_int, P, c_int, c_int, P, c_int, P, c_int,
                                   c_int, c_float, P, c_int, P, c_int, P]),
    "opm_text_attention_workspace_floats": (c_longlong, [c_int, c_int, c_int]),
    "opm_store_text_kv": (c_int, [P, c_int, c_int, c_int, c_int, P, c_int, c_int, c_int, P, P]),
}

STUDENT_SRC = os.path.join(ROOT, "tests", "cuda", "student_ops.cpp")
STUDENT_HEADERS = (HEADER, os.path.join(CSRC, "student_ops.h"))
STUDENT_SIGNATURES = {
    "sto_embed": (c_int, [P, P, c_int, c_int, c_int, c_int, P, P]),
    "sto_ln": (c_int, [P, P, c_int, c_int, P, P, P, c_int, P]),
    "sto_attn": (c_int, [P, P, c_int, c_int, c_int, P, c_int, c_int, c_int, c_int, c_int, c_int, P, c_int, c_int, P, c_int, P]),
    "sto_transpose": (c_int, [P, P, c_int, c_int, c_int, P, c_int, c_int, P]),
    "sto_colsum": (c_int, [P, P, c_int, c_int, c_int, P, P]),
    "sto_weight_grad": (c_int, [P, P, c_int, c_int, P, c_int, c_int, c_int, c_int, P, P, P, P]),
    "sto_ln_bwd": (c_int, [P, P, P, c_int, P, P, P, P, P, P]),
    "sto_attn_bwd": (c_int, [P, P, c_int, c_int, P, c_int, c_int, c_int, c_int, c_int, c_int, P, c_int, c_int, P, P, c_int, P, c_int,
                             c_int, c_int, P]),
    "sto_distill_loss": (c_int, [P, P, c_int, P, c_int, P, c_int, c_int, c_float, P, P, P, P, P]),
    "sto_relu_bwd": (c_int, [P, P, P, c_longlong, P]),
    "sto_embed_bwd": (c_int, [P, P, c_int, P, c_int, P, P]),
}


def compiler():
    return shutil.which(os.environ.get("CXX", "g++")) or shutil.which("c++")


def _out_dir():
    d = os.path.join(ROOT, "build")
    try:
        os.makedirs(d, exist_ok=True)
        if os.access(d, os.W_OK):
            return d
    except OSError:
        pass
    d = os.path.join(tempfile.gettempdir(), "gitb200_op_modes")
    os.makedirs(d, exist_ok=True)
    return d


def build(src=SRC, headers=(HEADER,)):
    """Compile the shim `src` (if it or one of `headers` changed) and return its path."""
    h = hashlib.sha256(PKG.encode())  # the library's directory is baked into the shim as its run path
    for f in (src, *headers):
        with open(f, "rb") as fh:
            h.update(fh.read())
    name = os.path.splitext(os.path.basename(src))[0]
    out = os.path.join(_out_dir(), f"{name}_{h.hexdigest()[:16]}.so")
    if os.path.exists(out):
        return out
    tmp = f"{out}.{os.getpid()}.tmp"
    cmd = [compiler(), "-shared", "-fPIC", "-std=c++17", "-O1", f"-I{CUDA_INCLUDE}", f"-I{CSRC}", src,
           f"-L{PKG}", "-l:libgitb200.so", f"-Wl,-rpath,{PKG}", "-o", tmp]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"{name} shim failed to build:\n{' '.join(cmd)}\n{r.stdout}\n{r.stderr}")
    os.replace(tmp, out)
    return out


def load(src=SRC, headers=(HEADER,), signatures=SIGNATURES):
    """Build and load a shim; libgitb200.so must already be loaded (gitb200 imported) so both share one copy of it."""
    lib = ctypes.CDLL(build(src, headers))
    for name, (res, args) in signatures.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    return lib


def load_student():
    """tests/cuda/student_ops.cpp: the student decoder's launchers (student_ops.h)."""
    return load(STUDENT_SRC, STUDENT_HEADERS, STUDENT_SIGNATURES)
