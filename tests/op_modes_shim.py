"""Builds and loads tests/cuda/op_modes.cpp: test-only C entry points over the internal launchers of libgitb200.so (kernels.h).

The shim is host C++ linked against the built library; it compiles no kernel.  The output goes to build/ (a temporary directory
if the tree is read-only), named by a hash of the shim, kernels.h and the library's directory, so a changed argument struct
rebuilds it."""
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
SRC = os.path.join(ROOT, "tests", "cuda", "op_modes.cpp")
HEADER = os.path.join(PKG, "csrc", "kernels.h")
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


def build():
    """Compile the shim (if its source or kernels.h changed) and return its path."""
    h = hashlib.sha256(PKG.encode())  # the library's directory is baked into the shim as its run path
    for f in (SRC, HEADER):
        with open(f, "rb") as fh:
            h.update(fh.read())
    out = os.path.join(_out_dir(), f"op_modes_{h.hexdigest()[:16]}.so")
    if os.path.exists(out):
        return out
    tmp = f"{out}.{os.getpid()}.tmp"
    cmd = [compiler(), "-shared", "-fPIC", "-std=c++17", "-O1", f"-I{CUDA_INCLUDE}", f"-I{os.path.dirname(HEADER)}", SRC,
           f"-L{PKG}", "-l:libgitb200.so", f"-Wl,-rpath,{PKG}", "-o", tmp]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"op_modes shim failed to build:\n{' '.join(cmd)}\n{r.stdout}\n{r.stderr}")
    os.replace(tmp, out)
    return out


def load():
    """Build and load the shim; libgitb200.so must already be loaded (gitb200 imported) so both share one copy of it."""
    lib = ctypes.CDLL(build())
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    return lib
