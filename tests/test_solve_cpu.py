"""CPU suite: the CPU restatement of the inhomogeneous solve (svo_solve in tests/solve_oracle.c, DESIGN.md section 13).
The reference has no such step, so the restatement is pinned by the properties that define a solution, with ranks
from an independent elimination:

* M x_j == b_j (--right) or x_j^T M == b_j^T (--left) for every found j; unsolved columns are zero;
* found[j] == (e_j lies in the column space of T), T the tail rows of the kernel basis of the augmented matrix;
* planted consistent systems are solved completely after the loop, at small and large primes, on both sides;
* b non-zero where M has an empty row (--right) or column (--left) is not solved;
* relabelling both dimensions of the problem permutes the rows of x and nothing else.
"""
import numpy as np
import pytest

import kb_oracle
import solve_oracle
from test_kernel_basis_cpu import rank_mod_p

import blk_lanczos_b200 as B

P31 = 2147483647
# (p, n, r): the blocking factor has to leave room for the kernel vectors at small p (DESIGN.md section 13)
CASES = [(2, 64, 8), (2, 32, 4), (3, 16, 4), (7, 16, 4), (65537, 16, 4), (65537, 4, 2), (P31, 16, 8), (P31, 2, 1)]


def product(oracle, M, x, right, p):
    """M x (--right) or M^T x (--left) as an (Mc x w) array."""
    x = np.asarray(x, dtype=np.uint32)
    if x.ndim == 1:
        x = x.reshape(-1, 1)
    w = x.shape[1]
    y = oracle.sparse_matrix_vector_product(M, np.ascontiguousarray(x).ravel(), not right, w, p)
    return y.reshape(-1, w)


def random_block(rows, cols, p, seed):
    return np.random.default_rng(seed).integers(0, p, size=(rows, cols), dtype=np.int64).astype(np.uint32)


def planted(oracle, M, r, p, right, seed):
    """B = M X0 (--right) or M^T X0 (--left) for a random X0: a consistent system."""
    N = M.ncols if right else M.nrows
    X0 = random_block(N, r, p, seed)
    return product(oracle, M, X0, right, p)


def run_loop(oracle, M, Bm, n, p, right):
    """The loop on the augmented matrix from the driver's start block: the final v ((N + r) x n)."""
    A = solve_oracle.augmented(M, Bm, p, right)
    st = oracle.lanczos_run(A, n, p, right)
    Np = A.ncols if right else A.nrows
    return st["v"][:Np * n].reshape(Np, n)


def check_properties(oracle, M, Bm, v, n, p, right):
    x, found = solve_oracle.solve(M, Bm, v, n, p, right)
    b = solve_oracle.reduce_rhs(Bm, p)
    N = M.ncols if right else M.nrows
    r = b.shape[1]
    assert x.shape == (N, r) and found.shape == (r,) and (x < p).all()
    y = product(oracle, M, x, right, p)
    for j in range(r):
        if found[j]:
            assert np.array_equal(y[:, j], b[:, j]), j
        else:
            assert not x[:, j].any(), j
    # found against an independent rank test of the tail of the kernel basis
    X = kb_oracle.kernel_basis(solve_oracle.augmented(M, Bm, p, right), v, n, p, right)
    T = X[N:N + r].astype(np.int64)
    rt = rank_mod_p(T, p) if T.size else 0
    for j in range(r):
        e = np.zeros((r, 1), dtype=np.int64)
        e[j] = 1
        assert found[j] == (rank_mod_p(np.hstack([T, e]), p) == rt), j
    return x, found


@pytest.mark.parametrize("p,n,r", CASES)
@pytest.mark.parametrize("right", [False, True])
def test_oracle_solves_planted_systems(oracle, p, n, r, right):
    M = B.synth.uniform_rows(400, 400, 5, seed=3).reduced(p)
    Bm = planted(oracle, M, r, p, right, seed=n + r)
    v = run_loop(oracle, M, Bm, n, p, right)
    _, found = check_properties(oracle, M, Bm, v, n, p, right)
    assert found.all(), found


@pytest.mark.parametrize("p,n,r", [(65537, 16, 8), (P31, 16, 16), (2, 64, 8)])
def test_oracle_solves_rectangular_systems(oracle, p, n, r):
    """A wide matrix (--right: more unknowns than equations) and its transpose (--left)."""
    W = B.synth.uniform_rows(560, 600, 5, seed=8).reduced(p)
    for right, M in ((True, W), (False, B.SparseCOO(W.ncols, W.nrows, W.j, W.i, W.x))):
        Bm = planted(oracle, M, r, p, right, seed=r)
        v = run_loop(oracle, M, Bm, n, p, right)
        _, found = check_properties(oracle, M, Bm, v, n, p, right)
        assert found.all(), (right, found)


@pytest.mark.parametrize("p,n", [(65537, 8), (2, 32), (P31, 4)])
@pytest.mark.parametrize("right", [False, True])
def test_oracle_inconsistent_system(oracle, p, n, right):
    """b_0 non-zero on an empty row of M (--right) or column (--left): no solution exists, found[0] is 0."""
    M = B.synth.uniform_rows(300, 300, 5, seed=5)
    empty = 17
    keep = (M.i != empty) if right else (M.j != empty)
    M = B.SparseCOO(M.nrows, M.ncols, M.i[keep], M.j[keep], M.x[keep]).reduced(p)
    Bm = planted(oracle, M, 2, p, right, seed=1)
    Bm[empty, 0] = 1
    v = run_loop(oracle, M, Bm, n, p, right)
    x, found = check_properties(oracle, M, Bm, v, n, p, right)
    assert not found[0] and not x[:, 0].any()


@pytest.mark.parametrize("p,n,r", [(2, 32, 4), (3, 16, 3), (65537, 8, 8), (P31, 5, 2)])
@pytest.mark.parametrize("right", [False, True])
def test_oracle_solve_row_order_free(oracle, p, n, r, right):
    """Relabelling the N rows of the problem (with v) and the Mc rows (with B) permutes the rows of x only."""
    M = B.synth.uniform_rows(300, 300, 5, seed=9).reduced(p)
    Bm = planted(oracle, M, r, p, right, seed=2)
    v = run_loop(oracle, M, Bm, n, p, right)
    x, found = solve_oracle.solve(M, Bm, v, n, p, right)
    rng = np.random.default_rng(n)
    N, Mc = (M.ncols, M.nrows) if right else (M.nrows, M.ncols)
    pn, pm = rng.permutation(N), rng.permutation(Mc)           # new label of old row r: pn[r]
    if right:
        M2 = B.SparseCOO(M.nrows, M.ncols, pm[M.i].astype(np.int32), pn[M.j].astype(np.int32), M.x)
    else:
        M2 = B.SparseCOO(M.nrows, M.ncols, pn[M.i].astype(np.int32), pm[M.j].astype(np.int32), M.x)
    B2 = np.empty_like(Bm)
    B2[pm] = Bm
    v2 = v.copy()
    v2[pn] = v[:N]                                             # the r tail rows stay where they are
    x2, found2 = solve_oracle.solve(M2, B2, v2, n, p, right)
    assert np.array_equal(found2, found)
    assert np.array_equal(x2[pn], x)


def test_rhs_ingest_semantics():
    """-k is 2^32 - k before the reduction, like the MatrixMarket loader."""
    b = solve_oracle.reduce_rhs(np.array([[-1], [5], [-65537]]), 65537)
    assert b.ravel().tolist() == [(2**32 - 1) % 65537, 5, (2**32 - 65537) % 65537]
