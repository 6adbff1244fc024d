"""ctypes wrapper of tests/kb_oracle.c, the CPU restatement of the kernel-basis extraction -- TEST INFRASTRUCTURE.

The C file is compiled on first use into a temporary directory (keyed by its content), never into the tree.
"""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "kb_oracle.c")

_u32p = np.ctypeslib.ndpointer(dtype=np.uint32, flags="C_CONTIGUOUS")
_i32p = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")
_lib = None


def _load():
    global _lib
    if _lib is not None:
        return _lib
    src = open(SRC, "rb").read()
    tag = hashlib.sha256(src).hexdigest()[:16]
    d = os.path.join(tempfile.gettempdir(), f"blk_kb_oracle_{os.getuid()}_{tag}")
    so = os.path.join(d, "libkboracle.so")
    if not os.path.exists(so):
        os.makedirs(d, exist_ok=True)
        part = f"{so}.{os.getpid()}"
        subprocess.check_call(["gcc", "-std=c99", "-O2", "-fPIC", "-shared", "-Wall", "-Wextra", "-o", part, SRC])
        os.replace(part, so)
    L = C.CDLL(so)
    L.kbo_kernel_basis.argtypes = [C.c_int, C.c_int, C.c_long, _i32p, _i32p, _u32p, _u32p, C.c_int,
                                   C.c_uint64, C.c_int, _u32p]
    L.kbo_kernel_basis.restype = C.c_int
    _lib = L
    return L


def kernel_basis(M, v, n: int, p: int, right: bool) -> np.ndarray:
    """The kernel vectors inside span(v) for the COO matrix M (values already reduced mod p): an N x k uint32
    array, k = its rank, exactly as DESIGN.md section 12 defines it."""
    L = _load()
    N = M.ncols if right else M.nrows
    v = np.ascontiguousarray(np.asarray(v, dtype=np.uint32).ravel()[:N * n])
    X = np.zeros(N * n, dtype=np.uint32)
    k = L.kbo_kernel_basis(M.nrows, M.ncols, M.nnz, np.ascontiguousarray(M.i, dtype=np.int32),
                           np.ascontiguousarray(M.j, dtype=np.int32), np.ascontiguousarray(M.x, dtype=np.uint32),
                           v, n, p, int(right), X)
    return X.reshape(N, n)[:, :k].copy()
