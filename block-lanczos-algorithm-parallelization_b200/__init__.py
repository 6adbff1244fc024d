"""B200-native block-Lanczos mod-p hot path -- Python host side over the C ABI.

The product is ``libblklanczos.so`` (hand-written sm_100a CUDA behind ``include/blk_lanczos.h``)
and the C driver in ``driver/``.  This module is the ctypes mirror of the reference's per-iteration
functions (same names and argument meaning as sequential/lanczos_modp.c) used by the parity tests
and by bench.py.  There is NO CPU fallback: if the shared library is missing the import of the
binding fails loudly, and without a CUDA device ``BlockLanczos(...)`` raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import synth                                   # noqa: F401  (re-export)
from .synth import SparseCOO                          # noqa: F401

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(PKG_DIR, "libblklanczos.so")

BLK_ABI_VERSION = 2
BLK_MAX_N = 64
BLK_NCCL_ID_BYTES = 128
BLK_RANK_ALL = -1          # blk_params.rank: one context (one process) drives all `world` GPUs
PRUNE_STATS = ("N", "Mc", "nnz", "free", "rounds")     # BLK_PR_N ... BLK_PR_ROUNDS
PHASES = ("spmv1", "spmv2", "dots", "small", "ortho", "exchange")

# every symbol include/blk_lanczos.h declares
ABI_SYMBOLS = (
    "blk_abi_version", "blk_last_error", "blk_device_count", "blk_nccl_unique_id", "blk_create", "blk_create_system",
    "blk_create_pruned", "blk_pruned_index",
    "blk_destroy", "blk_plan_shards", "blk_plan_grid", "blk_plan_heavy", "blk_block_pad", "blk_set_state", "blk_iterate", "blk_get_state", "blk_get_state_local", "blk_final_check",
    "blk_check_kernel_block", "blk_kernel_basis", "blk_solve", "blk_get_small",
    "blk_spmv", "blk_block_dot_products", "blk_semi_inverse", "blk_orthogonalize",
    "blk_set_profiling", "blk_get_phase_times", "blk_time_spmv", "blk_kernel_launches", "blk_get_info",
)


class BlkError(RuntimeError):
    pass


class blk_params(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32), ("nrows", C.c_int32), ("ncols", C.c_int32), ("nnz", C.c_int64),
        ("Mi", C.c_void_p), ("Mj", C.c_void_p), ("Mx", C.c_void_p), ("coo_on_device", C.c_int32),
        ("n", C.c_int32), ("prime", C.c_uint32), ("right_kernel", C.c_int32), ("device", C.c_int32),
        ("rank", C.c_int32), ("world", C.c_int32), ("nccl_id", C.c_void_p), ("stream", C.c_void_p),
        ("chunk_len", C.c_int32), ("use_graph", C.c_int32),
    ]


class blk_info(C.Structure):
    _fields_ = [
        ("N", C.c_int64), ("Mc", C.c_int64), ("local_N0", C.c_int64), ("local_N1", C.c_int64),
        ("local_M0", C.c_int64), ("local_M1", C.c_int64), ("nnz_local", C.c_int64 * 2),
        ("stored_local", C.c_int64 * 2), ("tiles", C.c_int64 * 2), ("n", C.c_int32), ("n_pad", C.c_int32),
        ("chunk_len", C.c_int32 * 2), ("groups_per_warp", C.c_int32), ("device_bytes", C.c_int64),
        ("loop_mode", C.c_int32), ("nrhs", C.c_int32), ("bands", C.c_int32 * 2),
        ("heavy_rows", C.c_int64), ("heavy_bands", C.c_int32),
    ]


_lib = None


def load_library(path: str | None = None) -> C.CDLL:
    """dlopen the CUDA library.  Raises (never falls back) when it has not been built."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    path = path or LIB_PATH
    if not os.path.exists(path):
        raise BlkError(f"{path} not found: build it with `python __graft_entry__.py build` "
                       "(nvcc, sm_100a). There is no CPU fallback.")
    L = C.CDLL(path)
    vp, i32, i64 = C.c_void_p, C.c_int32, C.c_int64
    L.blk_abi_version.restype = C.c_int
    L.blk_last_error.restype = C.c_char_p
    L.blk_device_count.argtypes = [C.POINTER(C.c_int)]
    L.blk_nccl_unique_id.argtypes = [vp]
    L.blk_create.argtypes = [C.POINTER(vp), C.POINTER(blk_params)]
    L.blk_create_system.argtypes = [C.POINTER(vp), C.POINTER(blk_params), vp, i32, i32]
    L.blk_create_pruned.argtypes = [C.POINTER(vp), C.POINTER(blk_params), vp]
    L.blk_pruned_index.argtypes = [vp, vp, vp]
    L.blk_destroy.argtypes = [vp]
    L.blk_plan_shards.argtypes = [vp, i64, i64, i32, vp]
    L.blk_plan_grid.argtypes = [vp, vp, i64, i32, i32, i32, i32, vp, vp, vp, vp, vp, vp]
    L.blk_plan_heavy.argtypes = [vp, i64, i64, i32, i64, i64, i64, i32, C.POINTER(i64), C.POINTER(i32)]
    L.blk_block_pad.argtypes = [i32, i32, i32, i32]
    L.blk_block_pad.restype = i64
    L.blk_set_state.argtypes = [vp, vp, vp, i32]
    L.blk_iterate.argtypes = [vp, i32, C.POINTER(i32), C.POINTER(i32)]
    L.blk_get_state.argtypes = [vp, vp, vp, vp, vp]
    L.blk_get_state_local.argtypes = [vp, vp, vp, vp]
    L.blk_final_check.argtypes = [vp, C.POINTER(i32), C.POINTER(i32)]
    L.blk_check_kernel_block.argtypes = [vp, vp, C.POINTER(i32)]
    L.blk_kernel_basis.argtypes = [vp, vp, C.POINTER(i32)]
    L.blk_solve.argtypes = [vp, vp, vp]
    L.blk_get_small.argtypes = [vp, vp, vp, vp, vp, C.POINTER(i32)]
    L.blk_spmv.argtypes = [vp, vp, vp, i32]
    L.blk_block_dot_products.argtypes = [vp, vp, vp, i64, vp, vp]
    L.blk_semi_inverse.argtypes = [vp, vp, vp, vp, C.POINTER(i32)]
    L.blk_orthogonalize.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, i64, vp]
    L.blk_set_profiling.argtypes = [vp, i32]
    L.blk_get_phase_times.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(i64)]
    L.blk_time_spmv.argtypes = [vp, i32, i32, C.POINTER(C.c_double)]
    L.blk_kernel_launches.argtypes = [vp]
    L.blk_kernel_launches.restype = i64
    L.blk_get_info.argtypes = [vp, C.POINTER(blk_info)]
    if L.blk_abi_version() != BLK_ABI_VERSION:
        raise BlkError("libblklanczos.so ABI version mismatch")
    if path == LIB_PATH:
        _lib = L
    return L


def _u32(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.uint32)


def _ptr(a) -> C.c_void_p:
    return C.c_void_p(a.ctypes.data) if a is not None else C.c_void_p(None)


def block_pad(nrows: int, ncols: int, n: int, right: bool) -> int:
    return int(load_library().blk_block_pad(nrows, ncols, n, int(right)))


def plan_shards(idx, dim: int, world: int) -> np.ndarray:
    """Row-block boundaries (world+1 offsets) blk_create uses along one dimension (host only)."""
    L = load_library()
    idx = np.ascontiguousarray(idx, dtype=np.int32)
    off = np.zeros(world + 1, dtype=np.int64)
    if L.blk_plan_shards(_ptr(idx), idx.size, dim, world, _ptr(off)):
        raise BlkError(L.blk_last_error().decode())
    return off


def plan_heavy(deg, cols: int, n_pad: int, l2_bytes: int, min_deg: int, band_bytes: int, force: bool = False):
    """(H, K) of blk_plan_heavy (host only): the high-degree row prefix of product 2 run as K column bands."""
    L = load_library()
    deg = _u32(deg)
    H, K = C.c_int64(0), C.c_int32(0)
    if L.blk_plan_heavy(_ptr(deg), deg.size, cols, n_pad, l2_bytes, min_deg, band_bytes, int(force), C.byref(H), C.byref(K)):
        raise BlkError(L.blk_last_error().decode())
    return H.value, K.value


def plan_grid(M, right: bool, world: int, grid=(0, 0)) -> dict:
    """The P x Q block grid of blk_plan_grid (host only): dict(P, Q, n_off, m_off, n_sub[P][Q+1],
    m_sub[Q][P+1], block_nnz[P][Q]).  grid=(0, 0) chooses the factorisation like MPI_Dims_create."""
    L = load_library()
    i = np.ascontiguousarray(M.i, dtype=np.int32)
    j = np.ascontiguousarray(M.j, dtype=np.int32)
    g = (C.c_int32 * 2)(int(grid[0]), int(grid[1]))
    if grid[0] and grid[1]:
        P, Q = int(grid[0]), int(grid[1])
    else:
        P = Q = world          # upper bounds for the output buffers
    n_off, m_off = np.zeros(P + 1, np.int64), np.zeros(Q + 1, np.int64)
    n_sub, m_sub = np.zeros(P * (Q + 1) + world + 1, np.int64), np.zeros(Q * (P + 1) + world + 1, np.int64)
    bn = np.zeros(P * Q, np.int64)
    if L.blk_plan_grid(_ptr(i), _ptr(j), i.size, M.nrows, M.ncols, int(bool(right)), world, g, _ptr(n_off), _ptr(m_off),
                       _ptr(n_sub), _ptr(m_sub), _ptr(bn)):
        raise BlkError(L.blk_last_error().decode())
    P, Q = int(g[0]), int(g[1])
    return dict(P=P, Q=Q, n_off=n_off[:P + 1].copy(), m_off=m_off[:Q + 1].copy(),
                n_sub=n_sub[:P * (Q + 1)].reshape(P, Q + 1).copy(), m_sub=m_sub[:Q * (P + 1)].reshape(Q, P + 1).copy(),
                block_nnz=bn[:P * Q].reshape(P, Q).copy())


def nccl_unique_id() -> bytes:
    L = load_library()
    buf = C.create_string_buffer(BLK_NCCL_ID_BYTES)
    if L.blk_nccl_unique_id(buf):
        raise BlkError(L.blk_last_error().decode())
    return buf.raw


class BlockLanczos:
    """One GPU-resident problem: the matrix, the modulus, the blocking factor, the four blocks.

    Mirrors what block_lanczos() holds on its stack (sequential/lanczos_modp.c:585-669).  The
    method names are the reference's function names; ``n`` and ``prime`` are bound at creation
    the way the reference binds them as globals.
    """

    def __init__(self, M=None, *, n: int, prime: int, right: bool = False, device: int = 0,
                 rank: int = 0, world: int = 1, nccl_id: bytes | None = None, stream: int | None = None,
                 chunk_len: int = 0, use_graph: int = -1, device_coo=None, rhs=None, rhs_device=None,
                 prune: bool = False):
        """`M` is a host SparseCOO; alternatively `device_coo=(nrows, ncols, nnz, i_ptr, j_ptr, x_ptr)`
        gives raw CUDA device pointers (int32, int32, uint32) on `device`.  `rank=BLK_RANK_ALL` with
        `world=W` makes ONE context drive W GPUs (devices device..device+W-1) from this process.

        `rhs` (an Mc x r integer array, 1 <= r <= n; Mc = nrows for --right, ncols for --left) makes the context of
        the system M x = b (x M = b for --left), blk_create_system: the loop then runs on the augmented matrix, so
        `nrows` / `ncols` / `N` / `pad` are its sizes; `N0` is the original length and `nrhs` = r.  Negative
        entries are taken like the MatrixMarket loader takes them (-k is 2^32 - k before the reduction mod p).
        `rhs_device=(ptr, r)` gives that block instead as a raw CUDA device pointer (uint32, Mc x r) on `device`.

        `prune=True` removes the empty and singleton constraints first (blk_create_pruned, DESIGN.md section 14): the
        loop then runs on M', so `nrows` / `ncols` / `N` / `Mc` / `pad` are its sizes, `orig_N` / `orig_Mc` the
        original ones; `prune_stats`, `pruned_index()` and `lift()` relate the two.  Not with `rhs`."""
        self.L = load_library()
        self.n, self.prime, self.right = int(n), int(prime), bool(right)
        self.pruned, self.prune_stats = bool(prune), None
        if prune and (rhs is not None or rhs_device is not None):
            raise BlkError("prune=True cannot be combined with rhs= (a singleton constraint forces a value in a system)")
        prm = blk_params()
        prm.abi_version = BLK_ABI_VERSION
        keep = []
        if device_coo is not None:
            prm.nrows, prm.ncols, prm.nnz = device_coo[0], device_coo[1], device_coo[2]
            prm.Mi, prm.Mj, prm.Mx = device_coo[3], device_coo[4], device_coo[5]
            prm.coo_on_device = 1
        else:
            mi = np.ascontiguousarray(M.i, dtype=np.int32)
            mj = np.ascontiguousarray(M.j, dtype=np.int32)
            mx = _u32(M.x)
            keep = [mi, mj, mx]
            prm.nrows, prm.ncols, prm.nnz = M.nrows, M.ncols, M.nnz
            prm.Mi, prm.Mj, prm.Mx = mi.ctypes.data, mj.ctypes.data, mx.ctypes.data
        self.nrows, self.ncols, self.nnz = int(prm.nrows), int(prm.ncols), int(prm.nnz)
        self.nrhs = 0
        b_ptr, b_dev = None, 0
        if rhs_device is not None:
            b_ptr, b_dev, self.nrhs = C.c_void_p(rhs_device[0]), 1, int(rhs_device[1])
        elif rhs is not None:
            b = np.asarray(rhs)
            if b.ndim == 1:
                b = b.reshape(-1, 1)
            if b.ndim != 2 or b.shape[0] != (self.nrows if right else self.ncols):
                raise BlkError(f"rhs must be an Mc x r array (Mc = {self.nrows if right else self.ncols}), "
                               f"got shape {b.shape}")
            b = _u32(b.astype(np.int64) % (1 << 32) if b.dtype.kind == "i" else b)
            keep.append(b)
            b_ptr, self.nrhs = _ptr(b), int(b.shape[1])
        prm.n, prm.prime, prm.right_kernel, prm.device = n, prime, int(right), device
        prm.rank, prm.world = rank, world
        idbuf = None
        if nccl_id is not None:
            idbuf = C.create_string_buffer(nccl_id, BLK_NCCL_ID_BYTES)
            prm.nccl_id = C.cast(idbuf, C.c_void_p)
        prm.stream = stream
        prm.chunk_len, prm.use_graph = chunk_len, use_graph
        h = C.c_void_p()
        stats = (C.c_int64 * len(PRUNE_STATS))()
        if self.nrhs:
            rc = self.L.blk_create_system(C.byref(h), C.byref(prm), b_ptr, self.nrhs, b_dev)
        elif prune:
            rc = self.L.blk_create_pruned(C.byref(h), C.byref(prm), stats)
        else:
            rc = self.L.blk_create(C.byref(h), C.byref(prm))
        del keep, idbuf
        if rc:
            raise BlkError(self.L.blk_last_error().decode())
        self.h = h
        self.N0 = self.ncols if right else self.nrows
        self.orig_N, self.orig_Mc = self.N0, (self.nrows if right else self.ncols)
        if prune:
            self.prune_stats = {k: int(stats[i]) for i, k in enumerate(PRUNE_STATS)}
            self.N0 = self.prune_stats["N"]
            Mc = self.prune_stats["Mc"]
            self.nrows, self.ncols = (Mc, self.N0) if right else (self.N0, Mc)
            self.nnz = self.prune_stats["nnz"]
        if right:
            self.ncols += self.nrhs
        else:
            self.nrows += self.nrhs
        self.N = self.ncols if right else self.nrows
        self.Mc = self.nrows if right else self.ncols
        self.pad = block_pad(self.nrows, self.ncols, n, right)

    # -- lifetime ---------------------------------------------------------
    def close(self):
        if getattr(self, "h", None):
            self.L.blk_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _ck(self, rc):
        if rc:
            raise BlkError(self.L.blk_last_error().decode())

    # -- the reference's functions (host arrays in, host arrays out) -------
    def sparse_matrix_vector_product(self, x, transpose: bool) -> np.ndarray:
        """y <- M x (transpose False) or M^T x (True); sequential/lanczos_modp.c:266."""
        rows = self.ncols if transpose else self.nrows
        cols = self.nrows if transpose else self.ncols
        x = _u32(x)
        assert x.size >= cols * self.n
        y = np.empty(rows * self.n, dtype=np.uint32)
        self._ck(self.L.blk_spmv(self.h, _ptr(y), _ptr(x), int(transpose)))
        return y

    def block_dot_products(self, N: int, Av, v):
        """(vtAv, vtAAv); sequential/lanczos_modp.c:443."""
        Av, v = _u32(Av), _u32(v)
        a = np.empty(self.n * self.n, dtype=np.uint32)
        b = np.empty(self.n * self.n, dtype=np.uint32)
        self._ck(self.L.blk_block_dot_products(self.h, _ptr(a), _ptr(b), N, _ptr(Av), _ptr(v)))
        return a, b

    def semi_inverse(self, U):
        """(npiv, winv, d); sequential/lanczos_modp.c:342."""
        U = _u32(U)
        winv = np.empty(self.n * self.n, dtype=np.uint32)
        d = np.empty(self.n, dtype=np.uint32)
        npiv = C.c_int32(0)
        self._ck(self.L.blk_semi_inverse(self.h, _ptr(U), _ptr(winv), _ptr(d), C.byref(npiv)))
        return npiv.value, winv, d

    def orthogonalize(self, v, p_blk, d, vtAv, vtAAv, winv, N: int, Av):
        """(next v rows [0,N), new p); sequential/lanczos_modp.c:456."""
        v, Av, d = _u32(v), _u32(Av), _u32(d)
        vtAv, vtAAv, winv = _u32(vtAv), _u32(vtAAv), _u32(winv)
        pn = np.array(p_blk[:N * self.n], dtype=np.uint32, copy=True)
        tmp = np.empty(N * self.n, dtype=np.uint32)
        self._ck(self.L.blk_orthogonalize(self.h, _ptr(v), _ptr(tmp), _ptr(pn), _ptr(d), _ptr(vtAv),
                                          _ptr(vtAAv), _ptr(winv), N, _ptr(Av)))
        return tmp, pn

    # -- the loop -----------------------------------------------------------
    def set_state(self, v, p_blk=None, n_iterations: int = 0):
        v = _u32(v)
        assert v.size >= self.N * self.n
        pb = _u32(p_blk) if p_blk is not None else None
        self._ck(self.L.blk_set_state(self.h, _ptr(v), _ptr(pb), n_iterations))

    def iterate(self, max_iters: int):
        """Run up to max_iters iterations on the device.  Returns (n_iterations, stopped)."""
        it, st = C.c_int32(0), C.c_int32(0)
        self._ck(self.L.blk_iterate(self.h, max_iters, C.byref(it), C.byref(st)))
        return it.value, bool(st.value)

    def get_state(self, which=("v", "tmp", "Av", "p")) -> dict:
        out = {k: np.empty(self.pad, dtype=np.uint32) for k in which}
        self._ck(self.L.blk_get_state(self.h, _ptr(out.get("v")), _ptr(out.get("tmp")),
                                      _ptr(out.get("Av")), _ptr(out.get("p"))))
        return out

    def get_state_local(self, v=None, Av=None, p_blk=None):
        """Multi-process jobs: write only this rank's rows of v / Av / p into the given padded blocks."""
        self._ck(self.L.blk_get_state_local(self.h, _ptr(v), _ptr(Av), _ptr(p_blk)))

    def final_check(self):
        """(v != 0, M^T v == 0) evaluated on the device; sequential/lanczos_modp.c:560-582."""
        a, b = C.c_int32(0), C.c_int32(0)
        self._ck(self.L.blk_final_check(self.h, C.byref(a), C.byref(b)))
        return bool(a.value), bool(b.value)

    def check_kernel_block(self, x) -> bool:
        """checker_modp's verdict (checker_modp.c:146-204) for a block of N*n residues."""
        x = _u32(x)
        assert x.size >= self.N * self.n
        ok = C.c_int32(0)
        self._ck(self.L.blk_check_kernel_block(self.h, _ptr(x), C.byref(ok)))
        return bool(ok.value)

    def kernel_basis(self) -> np.ndarray:
        """The kernel vectors inside span(v) (blk_kernel_basis): an N x k uint32 array of independent columns,
        each annihilated by M (x^T M == 0 for --left, M x == 0 for --right); k may be 0."""
        x = np.empty(self.N * self.n, dtype=np.uint32)
        k = C.c_int32(0)
        self._ck(self.L.blk_kernel_basis(self.h, _ptr(x), C.byref(k)))
        return x.reshape(self.N, self.n)[:, :k.value].copy()

    def solve(self):
        """The solutions inside span(v) of a context made with `rhs` (blk_solve): (x, found), x an N0 x r uint32
        array, found a bool array of r flags.  M x[:, j] == b_j (x[:, j]^T M == b_j for --left) for every found j;
        the other columns are zero (no solution in span(v): the system may be inconsistent)."""
        if not self.nrhs:
            raise BlkError("solve() needs a context created with rhs=")
        x = np.empty(self.N0 * self.nrhs, dtype=np.uint32)
        found = np.zeros(self.nrhs, dtype=np.int32)
        self._ck(self.L.blk_solve(self.h, _ptr(x), _ptr(found)))
        return x.reshape(self.N0, self.nrhs), found.astype(bool)

    def pruned_index(self):
        """(unknowns, constraints) of a context made with prune=True: the original indices of the N' kept unknowns and
        the Mc' kept constraints, ascending int32 arrays (blk_pruned_index)."""
        if not self.pruned:
            raise BlkError("pruned_index() needs a context created with prune=True")
        u = np.empty(self.N, dtype=np.int32)
        c = np.empty(self.Mc, dtype=np.int32)
        self._ck(self.L.blk_pruned_index(self.h, _ptr(u), _ptr(c)))
        return u, c

    def lift(self, x) -> np.ndarray:
        """An N' x w block on the kept unknowns as the orig_N x w block of the original matrix, zero on the removed
        unknowns (a kernel vector of M' lifts to a kernel vector of M)."""
        x = np.asarray(x, dtype=np.uint32)
        if x.ndim == 1:
            x = x.reshape(self.N, -1)
        if x.shape[0] != self.N:
            raise BlkError(f"lift() takes an N' x w block (N' = {self.N}), got shape {x.shape}")
        u, _ = self.pruned_index()
        out = np.zeros((self.orig_N, x.shape[1]), dtype=np.uint32)
        out[u] = x
        return out

    def get_small(self):
        n = self.n
        a, b, w = (np.empty(n * n, dtype=np.uint32) for _ in range(3))
        d = np.empty(n, dtype=np.uint32)
        npiv = C.c_int32(0)
        self._ck(self.L.blk_get_small(self.h, _ptr(a), _ptr(b), _ptr(w), _ptr(d), C.byref(npiv)))
        return dict(vtAv=a, vtAAv=b, winv=w, d=d, npiv=npiv.value)

    def block_lanczos(self, v0, stop_after: int = -1, batch: int = 256, p0=None, n_iterations: int = 0):
        """The main loop of block_lanczos (sequential/lanczos_modp.c:631-659) from the start block
        v0.  Returns dict(v,tmp,Av,p,iters,stopped) with the reference's padded blocks."""
        self.set_state(v0, p0, n_iterations)
        it, stopped = n_iterations, False
        while not stopped:
            if stop_after > 0:
                if it >= stop_after:
                    break
                step = min(batch, stop_after - it)
            else:
                step = batch
            it, stopped = self.iterate(step)
        st = self.get_state()
        st.update(iters=it, stopped=stopped)
        return st

    # -- measurement ----------------------------------------------------------
    def set_profiling(self, on: bool):
        self._ck(self.L.blk_set_profiling(self.h, int(on)))

    def phase_times(self) -> dict:
        ms = (C.c_double * len(PHASES))()
        ln = (C.c_int64 * len(PHASES))()
        self._ck(self.L.blk_get_phase_times(self.h, ms, ln))
        return {PHASES[k]: dict(ms=ms[k], launches=ln[k]) for k in range(len(PHASES))}

    def time_spmv(self, transpose: bool, reps: int = 10) -> float:
        ms = C.c_double(0)
        self._ck(self.L.blk_time_spmv(self.h, int(transpose), reps, C.byref(ms)))
        return ms.value

    def kernel_launches(self) -> int:
        return int(self.L.blk_kernel_launches(self.h))

    def info(self) -> dict:
        inf = blk_info()
        self._ck(self.L.blk_get_info(self.h, C.byref(inf)))
        out = {}
        for name, _ in blk_info._fields_:
            val = getattr(inf, name)
            out[name] = list(val) if hasattr(val, "__len__") else val
        return out
