"""CPU suite: the CPU restatement of the pruning (pro_prune in tests/prune_oracle.c, DESIGN.md section 14), pinned by
the properties that make it exact and by an independent restatement of the synchronous rounds:

* dim ker M == dim ker M' (dense elimination), and the lift of a basis of ker M' is a basis of ker M;
* pruning M' removes nothing (idempotence);
* a permutation of the triplets changes nothing;
* a vectorised numpy restatement of the rounds gives the same kept sets, M' and stats;
* duplicates are counted, not merged, even when they cancel mod p.
"""
import numpy as np
import pytest

import prune_oracle

import blk_lanczos_b200 as B

PRIMES = [2, 3, 7, 65537]


def dense(M, p, right):
    """The constraints x unknowns matrix A (duplicates summed mod p): the kernel is {x : A x = 0}."""
    N, Mc = (M.ncols, M.nrows) if right else (M.nrows, M.ncols)
    iu, ic = (M.j, M.i) if right else (M.i, M.j)
    A = np.zeros((Mc, N), dtype=np.int64)
    np.add.at(A, (ic.astype(np.int64), iu.astype(np.int64)), M.x.astype(np.int64) % p)
    return A % p


def null_basis(A, p):
    """A basis of {x : A x = 0 mod p} as the columns of an N x k array (reduced row echelon form)."""
    a = np.array(A, dtype=np.int64) % p
    rows, cols = a.shape
    piv, r = [], 0
    for c in range(cols):
        if r == rows:
            break
        nz = np.nonzero(a[r:, c])[0]
        if nz.size == 0:
            continue
        i = r + int(nz[0])
        a[[r, i]] = a[[i, r]]
        a[r] = (a[r] * pow(int(a[r, c]), p - 2, p)) % p
        for h in np.nonzero(a[:, c])[0]:
            if h != r:
                a[h] = (a[h] - int(a[h, c]) * a[r]) % p
        piv.append(c)
        r += 1
    free = [c for c in range(cols) if c not in set(piv)]
    X = np.zeros((cols, len(free)), dtype=np.int64)
    for k, f in enumerate(free):
        X[f, k] = 1
        for t, c in enumerate(piv):
            X[c, k] = (-a[t, f]) % p
    return X


def rank(A, p):
    return A.shape[1] - null_basis(A, p).shape[1] if A.size else 0


def numpy_rounds(M, p, right):
    """The synchronous rounds of the definition, vectorised: (kept unknowns, kept constraints, M', stats)."""
    N, Mc = (M.ncols, M.nrows) if right else (M.nrows, M.ncols)
    iu, ic = ((M.j, M.i) if right else (M.i, M.j))
    iu, ic = iu.astype(np.int64), ic.astype(np.int64)
    counting = M.x.astype(np.uint64) % p != 0
    ua, ca = np.ones(N, bool), np.ones(Mc, bool)
    rounds = 0
    while True:
        live = counting & ua[iu] & ca[ic]
        cnt = np.bincount(ic[live], minlength=Mc)
        D = ca & (cnt <= 1)
        if not D.any():
            break
        rounds += 1
        ua[iu[live & D[ic]]] = False          # a constraint of D with count 1 has exactly one live triplet
        ca[D] = False
    keep = counting & ua[iu] & ca[ic]
    unew, cnew = np.cumsum(ua) - 1, np.cumsum(ca) - 1
    u2, c2 = unew[iu[keep]].astype(np.int32), cnew[ic[keep]].astype(np.int32)
    x2 = (M.x[keep].astype(np.uint64) % p).astype(np.uint32)
    n1, m1 = int(ua.sum()), int(ca.sum())
    Mp = B.SparseCOO(m1, n1, c2, u2, x2) if right else B.SparseCOO(n1, m1, u2, c2, x2)
    used = np.zeros(n1, bool)
    used[u2] = True
    stats = dict(N=n1, Mc=m1, nnz=int(keep.sum()), free=int((~used).sum()), rounds=rounds)
    return np.nonzero(ua)[0], np.nonzero(ca)[0], Mp, stats


def small_matrices(right):
    """Up to 60 x 60: sparse uniform (many singletons), power law with empty rows, a matrix with empty columns, and a
    planted chain; oriented so that the unknowns are the first dimension for --left."""
    s = B.synth
    mats = [s.uniform_rows(60, 60, 2, seed=1), s.uniform_rows(50, 60, 3, seed=2),
            s.powerlaw_rows(60, 55, mean=3, seed=3, with_empty_rows=5), s.uniform_rows(40, 60, 4, seed=4, order="file")]
    # empty columns: the entries of 10 columns removed
    M = s.uniform_rows(60, 60, 3, seed=5)
    keep = M.j % 6 != 0
    mats.append(B.SparseCOO(M.nrows, M.ncols, M.i[keep], M.j[keep], M.x[keep]))
    mats.append(chain(30, seed=6))
    if right:
        mats = [B.SparseCOO(M.ncols, M.nrows, M.j, M.i, M.x) for M in mats]
    return mats


def chain(k, seed=0, extra=None):
    """A --left chain: constraint c (column) holds unknowns (rows) c and c + 1, constraint k - 1 only row k - 1; each
    round removes the last constraint of the chain and its lone unknown, k rounds in all.  `extra` appends a dense
    square block that survives."""
    rng = np.random.default_rng(seed)
    i = [c for c in range(k)] + [c + 1 for c in range(k - 1)]
    j = [c for c in range(k)] + [c for c in range(k - 1)]
    nr, nc = k, k
    if extra:
        for a in range(extra):
            for b in range(extra):
                i.append(k + a)
                j.append(k + b)
        nr, nc = k + extra, k + extra
    x = rng.integers(1, 100, size=len(i))
    return B.SparseCOO(nr, nc, np.array(i, np.int32), np.array(j, np.int32), x.astype(np.uint32))


def coo_equal(A, Bm):
    return (A.nrows, A.ncols) == (Bm.nrows, Bm.ncols) and np.array_equal(A.i, Bm.i) and np.array_equal(A.j, Bm.j) and \
        np.array_equal(A.x, Bm.x)


@pytest.mark.parametrize("right", [False, True])
@pytest.mark.parametrize("p", PRIMES)
def test_prune_keeps_the_kernel(p, right):
    for mi, M in enumerate(small_matrices(right)):
        N = M.ncols if right else M.nrows
        r = prune_oracle.prune(M, p, right)
        K = null_basis(dense(M, p, right), p)
        if r["stats"]["Mc"] == 0:
            assert K.shape[1] == r["stats"]["N"], mi
            continue
        K2 = null_basis(dense(r["M"], p, right), p)
        assert K.shape[1] == K2.shape[1], mi
        X = prune_oracle.lift(K2.astype(np.uint32), r["unknowns"], N).astype(np.int64)
        assert not (dense(M, p, right) @ X % p).any(), mi
        assert rank(X.T, p) == K.shape[1], mi


@pytest.mark.parametrize("right", [False, True])
@pytest.mark.parametrize("p", PRIMES)
def test_prune_agrees_with_the_synchronous_rounds(p, right):
    for mi, M in enumerate(small_matrices(right)):
        r = prune_oracle.prune(M, p, right)
        u, c, Mp, stats = numpy_rounds(M, p, right)
        assert np.array_equal(r["unknowns"], u) and np.array_equal(r["constraints"], c), mi
        assert r["stats"] == stats, (mi, r["stats"], stats)
        assert coo_equal(r["M"], Mp), mi


@pytest.mark.parametrize("right", [False, True])
@pytest.mark.parametrize("p", PRIMES)
def test_prune_is_idempotent_and_order_free(p, right):
    rng = np.random.default_rng(p)
    for mi, M in enumerate(small_matrices(right)):
        r = prune_oracle.prune(M, p, right)
        if r["stats"]["Mc"]:
            again = prune_oracle.prune(r["M"], p, right)
            assert again["stats"]["rounds"] == 0 and coo_equal(again["M"], r["M"]), mi
        perm = rng.permutation(M.nnz)
        P = B.SparseCOO(M.nrows, M.ncols, M.i[perm], M.j[perm], M.x[perm])
        rp = prune_oracle.prune(P, p, right)
        assert np.array_equal(rp["unknowns"], r["unknowns"]) and np.array_equal(rp["constraints"], r["constraints"]), mi
        assert rp["stats"] == r["stats"], mi


def test_prune_chain_rounds():
    r = prune_oracle.prune(chain(50, extra=4), 65537, False)
    assert r["stats"] == dict(N=4, Mc=4, nnz=16, free=0, rounds=50)
    assert r["unknowns"].tolist() == [50, 51, 52, 53]
    assert numpy_rounds(chain(50, extra=4), 65537, False)[3] == r["stats"]


@pytest.mark.parametrize("right", [False, True])
def test_prune_duplicates_count_twice(right):
    """Two triplets (c, u) whose values cancel mod p still give cnt(c) = 2: c and u stay, although column c of the
    summed matrix is zero.  A triplet whose value is 0 mod p does not count at all."""
    p = 7
    # --left: rows are unknowns.  Constraint 0: (0, 0) twice, 3 + 4 = 0 mod 7.  Constraints 1, 2: a 2 x 2 block on
    # unknowns 1, 2.  Constraint 3: (1, 3) = 7 and (2, 3) = 14, both 0 mod p: empty.  Unknown 3 has no entry: free.
    i = np.array([0, 0, 1, 1, 2, 2, 1, 2], np.int32)
    j = np.array([0, 0, 1, 2, 1, 2, 3, 3], np.int32)
    x = np.array([3, 4, 1, 2, 3, 5, 7, 14], np.uint32)
    M = B.SparseCOO(4, 4, i, j, x)
    if right:
        M = B.SparseCOO(4, 4, j, i, x)
    r = prune_oracle.prune(M, p, right)
    assert r["unknowns"].tolist() == [0, 1, 2, 3] and r["constraints"].tolist() == [0, 1, 2]
    assert r["stats"] == dict(N=4, Mc=3, nnz=6, free=1, rounds=1)
    assert numpy_rounds(M, p, right)[3] == r["stats"]
    # one of the two duplicates alone: constraint 0 is a singleton, unknown 0 goes with it
    M1 = B.SparseCOO(4, 4, M.i[1:], M.j[1:], M.x[1:])
    r1 = prune_oracle.prune(M1, p, right)
    assert r1["unknowns"].tolist() == [1, 2, 3] and r1["constraints"].tolist() == [1, 2]


def test_prune_everything_removed():
    r = prune_oracle.prune(chain(20), 65537, False)
    assert r["stats"]["N"] == 0 and r["stats"]["Mc"] == 0 and r["stats"]["rounds"] == 20
    # free unknowns only: every constraint goes, the free unknowns stay
    M = B.SparseCOO(5, 3, np.array([0, 1], np.int32), np.array([0, 1], np.int32), np.array([1, 1], np.uint32))
    r = prune_oracle.prune(M, 3, False)
    assert r["stats"] == dict(N=3, Mc=0, nnz=0, free=3, rounds=1)
