"""ctypes wrapper of tests/prune_oracle.c, the CPU restatement of the pruning of DESIGN.md section 14 -- TEST
INFRASTRUCTURE.

The C file is compiled on first use into a temporary directory (keyed by its content), never into the tree.
"""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "prune_oracle.c")
STATS = ("N", "Mc", "nnz", "free", "rounds")

_u32p = np.ctypeslib.ndpointer(dtype=np.uint32, flags="C_CONTIGUOUS")
_i32p = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")
_i64p = np.ctypeslib.ndpointer(dtype=np.int64, flags="C_CONTIGUOUS")
_lib = None


def _load():
    global _lib
    if _lib is not None:
        return _lib
    src = open(SRC, "rb").read()
    tag = hashlib.sha256(src).hexdigest()[:16]
    d = os.path.join(tempfile.gettempdir(), f"blk_prune_oracle_{os.getuid()}_{tag}")
    so = os.path.join(d, "libpruneoracle.so")
    if not os.path.exists(so):
        os.makedirs(d, exist_ok=True)
        part = f"{so}.{os.getpid()}"
        subprocess.check_call(["gcc", "-std=c99", "-O2", "-fPIC", "-shared", "-Wall", "-Wextra", "-o", part, SRC])
        os.replace(part, so)
    L = C.CDLL(so)
    L.pro_prune.argtypes = [C.c_int, C.c_int, C.c_long, _i32p, _i32p, _u32p, C.c_uint64, C.c_int, _i32p, _i32p, _i64p,
                            _i32p, _i32p, _u32p]
    L.pro_prune.restype = C.c_int
    _lib = L
    return L


def prune(M, p: int, right: bool) -> dict:
    """dict(unknowns, constraints, M, stats) for the COO matrix M (values not necessarily reduced): the original
    indices of the kept unknowns and constraints (ascending int32), M' as a SparseCOO, and the stats N, Mc, nnz, free,
    rounds, exactly as DESIGN.md section 14 defines them."""
    import blk_lanczos_b200 as Bk
    L = _load()
    N, Mc = (M.ncols, M.nrows) if right else (M.nrows, M.ncols)
    uk, ck = np.zeros(N, dtype=np.int32), np.zeros(Mc, dtype=np.int32)
    st = np.zeros(len(STATS), dtype=np.int64)
    cap = max(M.nnz, 1)
    oi, oj, ox = np.zeros(cap, np.int32), np.zeros(cap, np.int32), np.zeros(cap, np.uint32)
    rc = L.pro_prune(M.nrows, M.ncols, M.nnz, np.ascontiguousarray(M.i, dtype=np.int32),
                     np.ascontiguousarray(M.j, dtype=np.int32), np.ascontiguousarray(M.x, dtype=np.uint32), p, int(right),
                     uk, ck, st, oi, oj, ox)
    if rc:
        raise ValueError("prune_oracle: index out of range")
    stats = {k: int(st[i]) for i, k in enumerate(STATS)}
    z = stats["nnz"]
    nr, nc = (stats["Mc"], stats["N"]) if right else (stats["N"], stats["Mc"])
    Mp = Bk.SparseCOO(nr, nc, oi[:z].copy(), oj[:z].copy(), ox[:z].copy())
    return dict(unknowns=np.nonzero(uk)[0].astype(np.int32), constraints=np.nonzero(ck)[0].astype(np.int32), M=Mp,
                stats=stats)


def lift(x, unknowns, N: int) -> np.ndarray:
    """An N' x w block on the kept unknowns as the N x w block of the original matrix (zeros elsewhere)."""
    x = np.asarray(x, dtype=np.uint32)
    out = np.zeros((N, x.shape[1]), dtype=np.uint32)
    out[unknowns] = x
    return out
