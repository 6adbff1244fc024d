"""ctypes wrapper of tests/solve_oracle.c, the CPU restatement of the inhomogeneous solve -- TEST INFRASTRUCTURE.

The C file (which includes tests/kb_oracle.c) is compiled on first use into a temporary directory keyed by the
content of both, never into the tree.
"""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "solve_oracle.c")
DEPS = (SRC, os.path.join(HERE, "kb_oracle.c"))

_u32p = np.ctypeslib.ndpointer(dtype=np.uint32, flags="C_CONTIGUOUS")
_i32p = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")
_lib = None


def _load():
    global _lib
    if _lib is not None:
        return _lib
    h = hashlib.sha256()
    for f in DEPS:
        h.update(open(f, "rb").read())
    d = os.path.join(tempfile.gettempdir(), f"blk_solve_oracle_{os.getuid()}_{h.hexdigest()[:16]}")
    so = os.path.join(d, "libsolveoracle.so")
    if not os.path.exists(so):
        os.makedirs(d, exist_ok=True)
        part = f"{so}.{os.getpid()}"
        subprocess.check_call(["gcc", "-std=c99", "-O2", "-fPIC", "-shared", "-Wall", "-Wextra", "-I", HERE,
                               "-o", part, SRC])
        os.replace(part, so)
    L = C.CDLL(so)
    L.svo_solve.argtypes = [C.c_int, C.c_int, C.c_long, _i32p, _i32p, _u32p, _u32p, C.c_int, _u32p, C.c_int,
                            C.c_uint64, C.c_int, _u32p, _i32p]
    L.svo_solve.restype = C.c_int
    _lib = L
    return L


def reduce_rhs(B, p: int) -> np.ndarray:
    """B as the library ingests it: integers taken mod 2^32 (-k is 2^32 - k), then reduced mod p; Mc x r."""
    b = np.asarray(B)
    if b.ndim == 1:
        b = b.reshape(-1, 1)
    if b.dtype.kind == "i":
        b = b.astype(np.int64) % (1 << 32)
    return np.ascontiguousarray(b.astype(np.uint64) % p, dtype=np.uint32)


def solve(M, B, v, n: int, p: int, right: bool):
    """(x, found) for the COO matrix M (values already reduced mod p), the Mc x r block B and the block v of the
    loop on the augmented matrix ((N + r) x n), exactly as DESIGN.md section 13 defines them."""
    L = _load()
    b = reduce_rhs(B, p)
    r = b.shape[1]
    N = M.ncols if right else M.nrows
    v = np.ascontiguousarray(np.asarray(v, dtype=np.uint32).ravel()[:(N + r) * n])
    x = np.zeros(N * r, dtype=np.uint32)
    found = np.zeros(r, dtype=np.int32)
    L.svo_solve(M.nrows, M.ncols, M.nnz, np.ascontiguousarray(M.i, dtype=np.int32),
                np.ascontiguousarray(M.j, dtype=np.int32), np.ascontiguousarray(M.x, dtype=np.uint32),
                b, r, v, n, p, int(right), x, found)
    return x.reshape(N, r), found.astype(bool)


def augmented(M, B, p: int, right: bool):
    """The augmented matrix [M | -B] (right) or [M ; -B^T] as a SparseCOO (same triplet order as the library)."""
    import blk_lanczos_b200 as Bk
    b = reduce_rhs(B, p)
    Mc, r = b.shape
    N = M.ncols if right else M.nrows
    ii, jj = np.nonzero(b)
    vals = ((p - b[ii, jj].astype(np.int64)) % p).astype(np.uint32)
    rows, cols = (ii, N + jj) if right else (N + jj, ii)
    return Bk.SparseCOO(M.nrows + (0 if right else r), M.ncols + (r if right else 0),
                        np.concatenate([M.i, rows]).astype(np.int32), np.concatenate([M.j, cols]).astype(np.int32),
                        np.concatenate([M.x, vals]).astype(np.uint32))
