"""Product 2 split into a heavy row prefix run as column bands and a light remainder (SpOp::split, DESIGN.md section 4).

The split applies on its own only to blocks far larger than L2; here BLK_HEAVY_FORCE=1 with a small band slice forces it on
test-sized matrices, and BLK_HOT_MIN_BYTES=0 forces the degree-sorted labels it depends on.  Everything is compared with the
CPU oracle bit for bit.  The first test is host-only (blk_plan_heavy) and runs without a GPU."""
import ctypes

import numpy as np
import pytest

P_FERMAT, P_MERSENNE = 65537, 2147483647
P_WIDE = 1000000007          # 2^32 mod p is large: the full 64-bit Barrett reduction and a fold every 8 products
MB = 1 << 20


def test_plan_heavy_choice(lib):
    deg = np.array([5000, 900, 400, 200, 199, 50, 3, 0], np.uint32)
    big = 50_000_000
    # H = rows with degree >= min_deg (a prefix of the sorted degrees), K = ceil(x block / slice)
    assert lib.plan_heavy(deg, big, 16, 126 * MB, 200, 48 * MB) == (4, (big * 64 + 48 * MB - 1) // (48 * MB))
    assert lib.plan_heavy(deg, big, 16, 126 * MB, 400, 32 * MB)[0] == 3
    assert lib.plan_heavy(deg, big, 32, 126 * MB, 1, 48 * MB)[0] == 7
    assert lib.plan_heavy(deg, big, 16, 126 * MB, 0, 48 * MB)[0] == 8
    assert lib.plan_heavy(deg, big, 16, 126 * MB, 6000, 48 * MB) == (0, 0)            # no row that heavy
    assert lib.plan_heavy(deg, big, 16, 126 * MB, 200, 4096)[1] == 256                 # at most 256 bands
    # not applied: n_pad < 8, a gathered block that fits L2, a single band
    assert lib.plan_heavy(deg, big, 4, 126 * MB, 200, 48 * MB) == (0, 0)
    assert lib.plan_heavy(deg, 1_000_000, 16, 126 * MB, 200, 48 * MB) == (0, 0)
    assert lib.plan_heavy(deg, 1_000_000, 16, 126 * MB, 200, 512 * MB, force=True) == (0, 0)
    # force skips the L2 and cost checks, nothing else
    assert lib.plan_heavy(deg, 1_000_000, 16, 126 * MB, 200, 4096, force=True) == (4, 256)
    # the cost check: light rows in many bands cost more partial traffic than their lines save
    flat = np.full(1000, 40, np.uint32)
    assert lib.plan_heavy(flat, big, 16, 126 * MB, 30, 16 * MB) == (0, 0)
    assert lib.plan_heavy(flat, big, 16, 126 * MB, 30, 16 * MB, force=True)[0] == 1000
    assert lib.plan_heavy(np.full(10, 4000, np.uint32), big, 16, 126 * MB, 30, 16 * MB)[0] == 10
    H, K = ctypes.c_int64(0), ctypes.c_int32(0)
    assert lib.load_library().blk_plan_heavy(None, 3, 10, 16, 0, 0, 4096, 0, ctypes.byref(H), ctypes.byref(K)) != 0


def force(monkeypatch, min_deg, band_bytes=4096):
    monkeypatch.setenv("BLK_HOT_MIN_BYTES", "0")
    monkeypatch.setenv("BLK_HEAVY_FORCE", "1")
    monkeypatch.setenv("BLK_HEAVY_MIN_DEG", str(min_deg))
    monkeypatch.setenv("BLK_HEAVY_BAND_BYTES", str(band_bytes))


def giant_rows(lib, nrows, ncols, seed):
    """Power-law rows plus two rows far longer than a warp tile and a few empty rows."""
    M = lib.synth.powerlaw_rows(nrows, ncols, mean=8, seed=seed, cap=600, with_empty_rows=9)
    rng = np.random.default_rng(seed)
    gi = np.concatenate([M.i, np.full(5000, 3, np.int32), np.full(2500, nrows - 1, np.int32)])
    gj = np.concatenate([M.j, rng.integers(0, ncols, 7500).astype(np.int32)])
    gx = np.concatenate([M.x, rng.integers(1, 1 << 30, 7500).astype(np.uint32)])
    return lib.SparseCOO(nrows, ncols, gi, gj, gx)


def check_against_oracle(lib, oracle, M, n, p, right, stop_after, expect_split, rng, graphs=(0, 1)):
    Mp = M.reduced(p)
    N = M.ncols if right else M.nrows
    Mc = M.nrows if right else M.ncols
    for graph in graphs:
        with lib.BlockLanczos(Mp, n=n, prime=p, right=right, use_graph=graph) as ctx:
            inf = ctx.info()
            if expect_split:
                assert 0 < inf["heavy_rows"] <= N and inf["heavy_bands"] >= 2, inf
            else:
                assert inf["heavy_rows"] == 0 and inf["heavy_bands"] == 0, inf
            if graph == 0:
                for tr in (False, True):
                    cols = M.nrows if tr else M.ncols
                    x = rng.integers(0, p, size=cols * n).astype(np.uint32)
                    x[rng.integers(0, x.size, size=max(1, x.size // 50))] = p - 1
                    assert np.array_equal(ctx.sparse_matrix_vector_product(x, tr),
                                          oracle.sparse_matrix_vector_product(Mp, x, tr, n, p)), (n, p, right, tr)
            got = ctx.block_lanczos(oracle.start_block(N * n, p), stop_after=stop_after, batch=3)
            fc = ctx.final_check()
        want = oracle.lanczos_run(Mp, n, p, right, stop_after=stop_after)
        assert got["iters"] == want["iters"] and got["stopped"] == want["stopped"]
        for k in ("v", "tmp", "Av", "p"):
            assert np.array_equal(got[k], want[k]), (n, p, right, graph, k)
    return inf, fc, N, Mc


@pytest.mark.gpu
@pytest.mark.parametrize("right", [False, True])
@pytest.mark.parametrize("p", [P_FERMAT, P_MERSENNE, P_WIDE])
@pytest.mark.parametrize("n", [8, 12, 16, 32])
def test_heavy_split_matches_oracle(lib, oracle, monkeypatch, n, p, right):
    """Single products in both directions and whole loops (chain and graph), Mc > N and Mc < N."""
    force(monkeypatch, 12)
    rng = np.random.default_rng(n * 31 + p % 1000 + right)
    for M in (giant_rows(lib, 1500, 2300, 1), giant_rows(lib, 2600, 1700, 2)):
        check_against_oracle(lib, oracle, M, n, p, right, 5, True, rng)


@pytest.mark.gpu
@pytest.mark.parametrize("min_deg,which", [(10 ** 9, "none"), (0, "all"), (20, "some")])
def test_heavy_prefix_edges(lib, oracle, monkeypatch, min_deg, which):
    """H = 0 (no split is made), H = N (the light operator has no rows), and heavy rows with fewer entries than there
    are bands (empty in most bands: a dummy entry and a zero partial there)."""
    force(monkeypatch, min_deg)
    rng = np.random.default_rng(7)
    M = giant_rows(lib, 1800, 2100, 3)
    inf, _, N, _ = check_against_oracle(lib, oracle, M, 16, P_MERSENNE, False, 4, which != "none", rng)
    if which == "all":
        assert inf["heavy_rows"] == N
    if which == "some":
        deg = np.bincount(M.i, minlength=M.nrows)
        assert inf["heavy_rows"] == int((deg >= min_deg).sum()) < N
        assert int(deg[deg >= min_deg].min()) < inf["heavy_bands"]


@pytest.mark.gpu
def test_heavy_split_leaves_state_api_alone(lib, oracle, monkeypatch):
    """get_state, blk_spmv and final_check give what the unsplit operator gives, mid-run and after it."""
    M = giant_rows(lib, 2000, 1900, 4).reduced(P_MERSENNE)
    n, p = 16, P_MERSENNE
    v0 = oracle.start_block(M.nrows * n, p)
    x = np.random.default_rng(3).integers(0, p, size=M.ncols * n).astype(np.uint32)
    out = {}
    for heavy in ("0", "1"):
        force(monkeypatch, 15)
        monkeypatch.setenv("BLK_HEAVY", heavy)
        with lib.BlockLanczos(M, n=n, prime=p) as ctx:
            assert (ctx.info()["heavy_rows"] > 0) == (heavy == "1")
            ctx.set_state(v0)
            ctx.iterate(3)
            mid = ctx.get_state()
            y = ctx.sparse_matrix_vector_product(x, False)
            ctx.iterate(2)
            out[heavy] = (mid, y, ctx.get_state(), ctx.final_check())
    a, b = out["0"], out["1"]
    for k in ("v", "tmp", "Av", "p"):
        assert np.array_equal(a[0][k], b[0][k]) and np.array_equal(a[2][k], b[2][k]), k
    assert np.array_equal(a[1], b[1]) and a[3] == b[3]


@pytest.mark.gpu
def test_heavy_split_not_made_where_it_does_not_apply(lib, monkeypatch):
    """n_pad <= 4 (column bands serve those), no degree-sorted labels, BLK_HEAVY=0, and blocks that fit L2 without force."""
    M = giant_rows(lib, 1500, 1600, 5).reduced(P_FERMAT)
    force(monkeypatch, 5)
    with lib.BlockLanczos(M, n=4, prime=P_FERMAT) as ctx:
        assert ctx.info()["heavy_rows"] == 0
    monkeypatch.setenv("BLK_HOT", "0")
    with lib.BlockLanczos(M, n=16, prime=P_FERMAT) as ctx:
        assert ctx.info()["heavy_rows"] == 0
    monkeypatch.delenv("BLK_HOT")
    monkeypatch.setenv("BLK_HEAVY", "0")
    with lib.BlockLanczos(M, n=16, prime=P_FERMAT) as ctx:
        assert ctx.info()["heavy_rows"] == 0
    monkeypatch.delenv("BLK_HEAVY")
    monkeypatch.delenv("BLK_HEAVY_FORCE")
    with lib.BlockLanczos(M, n=16, prime=P_FERMAT) as ctx:
        assert ctx.info()["heavy_rows"] == 0
    monkeypatch.setenv("BLK_HEAVY_FORCE", "1")
    with lib.BlockLanczos(M, n=16, prime=P_FERMAT) as ctx:
        assert ctx.info()["heavy_rows"] > 0


def gpus():
    import torch
    return torch.cuda.device_count()


@pytest.mark.gpu
def test_heavy_split_not_made_on_several_gpus(lib, oracle, monkeypatch):
    """With world > 1 the products are sharded and pieced: every rank keeps its full operator."""
    if gpus() < 2:
        pytest.skip("needs two GPUs")
    force(monkeypatch, 5)
    M = giant_rows(lib, 1500, 1600, 6)
    n, p = 16, P_MERSENNE
    Mp = M.reduced(p)
    with lib.BlockLanczos(Mp, n=n, prime=p, rank=lib.BLK_RANK_ALL, world=2) as ctx:
        assert ctx.info()["heavy_rows"] == 0
        got = ctx.block_lanczos(oracle.start_block(M.nrows * n, p), stop_after=4, batch=2)
    want = oracle.lanczos_run(Mp, n, p, False, stop_after=4)
    for k in ("v", "tmp", "Av", "p"):
        assert np.array_equal(got[k], want[k]), k
