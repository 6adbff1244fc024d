"""CPU suite: the CPU restatement of the kernel-basis extraction (kbo_kernel_basis in tests/kb_oracle.c, the final
Gaussian elimination of block Lanczos).  The reference has no such step, so the oracle is pinned by its defining properties, with
ranks from an independent elimination written here:

* every column of X is annihilated: x^T M == 0 (--left) or M x == 0 (--right);
* rank X == k, and the columns of X lie in span(v);
* k == rank([T; V]) - rank(T), T = M^T v (--left) or M v (--right);
* permuting the rows of V together with the matrix permutes the rows of X and changes nothing else.
"""
import numpy as np
import pytest

import kb_oracle

import blk_lanczos_b200 as B

PRIMES = [2, 3, 7, 65537, 2147483647]
NS = [1, 2, 5, 16, 64]


def rank_mod_p(a, p):
    """Rank over GF(p) by plain Gaussian elimination (int64 arithmetic: p < 2^31)."""
    a = np.array(a, dtype=np.int64) % p
    rows, cols = a.shape
    r = 0
    for c in range(cols):
        if r == rows:
            break
        nz = np.nonzero(a[r:, c])[0]
        if nz.size == 0:
            continue
        i = r + int(nz[0])
        a[[r, i]] = a[[i, r]]
        a[r] = (a[r] * pow(int(a[r, c]), p - 2, p)) % p
        col = a[:, c].copy()
        col[r] = 0
        hit = np.nonzero(col)[0]
        for h in hit:
            a[h] = (a[h] - int(col[h]) * a[r]) % p
        r += 1
    return r


def product(oracle, M, x, right, p):
    """T = M^T x (--left) or M x (--right) as an (Mc x w) array."""
    w = x.shape[1]
    y = oracle.sparse_matrix_vector_product(M, np.ascontiguousarray(x, dtype=np.uint32).ravel(), not right, w, p)
    return y.reshape(-1, w)


def planted_case(n, p, right, seed):
    """A tall problem (Mc < n when n > 1) with a v of deficient rank: kernel vectors exist inside span(v)."""
    rng = np.random.default_rng(seed)
    N = 90 + 3 * n
    Mc = max(1, n // 2)
    M = B.synth.uniform_rows(N, Mc, 3, seed=seed) if not right else B.synth.uniform_rows(Mc, N, 40, seed=seed)
    M = M.reduced(p)
    r = max(1, n - n // 4)
    v = (rng.integers(0, p, size=(N, r), dtype=np.int64) @ rng.integers(0, p, size=(r, n), dtype=np.int64) % p
         if p < 2**31 // 2 else None)
    if v is None:           # keep the product exact in int64 for the largest primes
        a = rng.integers(0, p, size=(N, r)).astype(object)
        b = rng.integers(0, p, size=(r, n)).astype(object)
        v = np.array((a.dot(b)) % p, dtype=np.int64)
    return M, v.astype(np.uint32)


def check_properties(oracle, M, v, n, p, right):
    X = kb_oracle.kernel_basis(M, v, n, p, right)
    N = M.ncols if right else M.nrows
    k = X.shape[1]
    assert X.shape == (N, k) and X.dtype == np.uint32
    assert (X < p).all()
    if k:
        assert not product(oracle, M, X, right, p).any()
    assert rank_mod_p(X, p) == k
    # the columns of X lie in span(v)
    assert rank_mod_p(np.hstack([v, X]), p) == rank_mod_p(v, p)
    T = product(oracle, M, v, right, p)
    assert k == rank_mod_p(np.vstack([T, v]), p) - rank_mod_p(T, p)
    return X


@pytest.mark.parametrize("p", PRIMES)
@pytest.mark.parametrize("n", NS)
@pytest.mark.parametrize("right", [False, True])
def test_oracle_kernel_basis_planted(oracle, p, n, right):
    M, v = planted_case(n, p, right, seed=7 * n + p % 1000)
    X = check_properties(oracle, M, v, n, p, right)
    if n > 1:
        assert X.shape[1] > 0


@pytest.mark.parametrize("p,n", [(2, 16), (3, 16), (2, 5), (7, 2), (65537, 5), (2147483647, 1)])
@pytest.mark.parametrize("right", [False, True])
def test_oracle_kernel_basis_after_the_loop(oracle, p, n, right):
    """On the block the loop ends with (the case the option is for)."""
    M = (B.synth.uniform_rows(420, 400, 5, seed=3) if not right else B.synth.uniform_rows(400, 420, 5, seed=3)).reduced(p)
    st = oracle.lanczos_run(M, n, p, right)
    N = M.ncols if right else M.nrows
    check_properties(oracle, M, st["v"][:N * n].reshape(N, n), n, p, right)


@pytest.mark.parametrize("p", PRIMES)
@pytest.mark.parametrize("n", NS)
def test_oracle_kernel_basis_row_order_free(oracle, p, n):
    """Relabelling both dimensions of the problem permutes the rows of X and nothing else."""
    right = n % 2 == 1
    M, v = planted_case(n, p, right, seed=11 * n + 1)
    X = kb_oracle.kernel_basis(M, v, n, p, right)
    rng = np.random.default_rng(n)
    N, Mc = (M.ncols, M.nrows) if right else (M.nrows, M.ncols)
    pn, pm = rng.permutation(N), rng.permutation(Mc)       # new label of old row r: pn[r]
    if right:
        M2 = B.SparseCOO(M.nrows, M.ncols, pm[M.i].astype(np.int32), pn[M.j].astype(np.int32), M.x)
    else:
        M2 = B.SparseCOO(M.nrows, M.ncols, pn[M.i].astype(np.int32), pm[M.j].astype(np.int32), M.x)
    v2 = np.empty_like(v)
    v2[pn] = v
    X2 = kb_oracle.kernel_basis(M2, v2, n, p, right)
    assert X2.shape == X.shape
    assert np.array_equal(X2[pn], X)


def test_rank_helper():
    assert rank_mod_p([[1, 1], [1, 1]], 2) == 1
    assert rank_mod_p([[1, 2], [2, 1]], 3) == 1
    assert rank_mod_p([[1, 2], [2, 1]], 7) == 2
