"""GPU tests of the pruning (blk_create_pruned, BlockLanczos(prune=True), --prune): the kept indices, the stats and
M' equal the CPU restatement (pro_prune in tests/prune_oracle.c) at small and large primes on both sides, planted
chains of thousands of rounds and a 4M-row matrix whose first pass spans many CTAs included; whole loops on M' equal
the oracle's loop on M' bit for bit; lifted kernel bases are kernel vectors of M; through the driver and on several
GPUs."""
import os
import subprocess
import sys
import time

import numpy as np
import pytest

import kb_oracle
import prune_oracle
from test_gpu_cli import checker
from test_gpu_solve import matrices
from test_kernel_basis_cpu import rank_mod_p
from test_prune_cpu import chain

from conftest import ROOT

pytestmark = pytest.mark.gpu

DRIVER = os.path.join(ROOT, "block-lanczos-algorithm-parallelization_b200", "driver", "lanczos_modp")
PRIMES = [2, 3, 7, 65537, 2147483647]
NS = [1, 2, 8, 16, 32, 64]
ENV_KNOBS = ("BLK_HOT", "BLK_HOT_MIN_BYTES", "BLK_HOT_BYTES", "BLK_BANDS", "BLK_BAND_BYTES", "BLK_GPUS")


@pytest.fixture(autouse=True)
def _clean_env(monkeypatch):
    for k in ENV_KNOBS:
        monkeypatch.delenv(k, raising=False)


def cases(lib, right):
    """The matrices of test_gpu_solve (uniform, power law with empty rows, tall) and a sparse uniform one of column
    weight 3 that loses about a quarter of its unknowns."""
    M = lib.synth.uniform_rows(3000, 3000, 3, seed=7)
    if right:
        M = lib.SparseCOO(M.ncols, M.nrows, M.j, M.i, M.x)
    return matrices(lib, right) + [M]


def assert_same_operator(oracle, ctx, Mp, p, seed=0):
    """The device operator of the context is M' (both products, one random block each)."""
    rng = np.random.default_rng(seed)
    for transpose in (False, True):
        cols = Mp.nrows if transpose else Mp.ncols
        x = rng.integers(0, p, size=cols * ctx.n, dtype=np.int64).astype(np.uint32)
        got = ctx.sparse_matrix_vector_product(x, transpose)
        want = oracle.sparse_matrix_vector_product(Mp, x, transpose, ctx.n, p)
        assert np.array_equal(got, want), transpose


def assert_pruned_like_oracle(oracle, ctx, ref, p):
    assert ctx.prune_stats == ref["stats"], (ctx.prune_stats, ref["stats"])
    u, c = ctx.pruned_index()
    assert np.array_equal(u, ref["unknowns"]) and np.array_equal(c, ref["constraints"])
    info = ctx.info()
    assert info["N"] == ref["stats"]["N"] and info["Mc"] == ref["stats"]["Mc"]
    assert_same_operator(oracle, ctx, ref["M"], p)


@pytest.mark.parametrize("right", [False, True])
@pytest.mark.parametrize("p", PRIMES)
def test_prune_matches_oracle(lib, oracle, p, right):
    for mi, M in enumerate(cases(lib, right)):
        ref = prune_oracle.prune(M, p, right)
        with lib.BlockLanczos(M, n=2, prime=p, right=right, prune=True) as ctx:
            assert ctx.orig_N == (M.ncols if right else M.nrows) and ctx.orig_Mc == (M.nrows if right else M.ncols)
            assert_pruned_like_oracle(oracle, ctx, ref, p)
        if mi == 3:
            assert ref["stats"]["rounds"] > 2 and ref["stats"]["N"] < 0.9 * ctx.orig_N


@pytest.mark.parametrize("right", [False, True])
@pytest.mark.parametrize("n", NS)
@pytest.mark.parametrize("p", [2, 65537, 2147483647])
def test_loop_on_pruned_matrix_matches_oracle(lib, oracle, p, n, right):
    for mi, M in enumerate(cases(lib, right)):
        ref = prune_oracle.prune(M, p, right)
        with lib.BlockLanczos(M, n=n, prime=p, right=right, prune=True) as ctx:
            got = ctx.block_lanczos(oracle.start_block(ctx.N * n, p), batch=64)
            assert ctx.pad == len(got["v"])
        want = oracle.lanczos_run(ref["M"], n, p, right)
        assert got["iters"] == want["iters"] and got["stopped"] == want["stopped"], mi
        for k in ("v", "tmp", "Av", "p"):
            assert np.array_equal(got[k], want[k]), (mi, k)


@pytest.mark.parametrize("right", [False, True])
@pytest.mark.parametrize("p,n", [(2, 64), (3, 16)])
def test_lifted_kernel_basis_is_a_kernel_of_m(lib, oracle, p, n, right):
    for mi, M in enumerate(cases(lib, right)):
        ref = prune_oracle.prune(M, p, right)
        with lib.BlockLanczos(M, n=n, prime=p, right=right, prune=True) as ctx:
            ctx.block_lanczos(oracle.start_block(ctx.N * n, p), batch=64)
            X = ctx.kernel_basis()
            want = oracle.lanczos_run(ref["M"], n, p, right)
            assert np.array_equal(X, kb_oracle.kernel_basis(ref["M"], want["v"], n, p, right)), mi
            L = ctx.lift(X)
        assert L.shape == ((M.ncols if right else M.nrows), X.shape[1])
        if X.shape[1]:
            y = oracle.sparse_matrix_vector_product(M.reduced(p), np.ascontiguousarray(L).ravel(), not right, L.shape[1], p)
            assert not y.any(), mi
            assert rank_mod_p(L, p) == X.shape[1], mi


def test_prune_deep_chain(lib, oracle):
    """A planted chain of 3000 rounds in front of a block that survives: every round is one host round trip."""
    M = chain(3000, seed=2, extra=40)
    p = 65537
    ref = prune_oracle.prune(M, p, False)
    assert ref["stats"]["rounds"] == 3000
    with lib.BlockLanczos(M, n=4, prime=p, prune=True) as ctx:    # warm-up: module load
        pass
    t0 = time.perf_counter()
    with lib.BlockLanczos(M, n=4, prime=p, prune=True) as ctx:
        dt = time.perf_counter() - t0
        assert_pruned_like_oracle(oracle, ctx, ref, p)
    assert dt < 1.0, dt
    Mr = lib.SparseCOO(M.ncols, M.nrows, M.j, M.i, M.x)
    with lib.BlockLanczos(Mr, n=4, prime=p, right=True, prune=True) as ctx:
        assert_pruned_like_oracle(oracle, ctx, prune_oracle.prune(Mr, p, True), p)


def test_prune_free_unknowns_and_errors(lib, oracle):
    p = 65537
    M = lib.synth.powerlaw_rows(420, 400, mean=6, seed=4, with_empty_rows=9)
    ref = prune_oracle.prune(M, p, False)
    assert ref["stats"]["free"] == 9
    with lib.BlockLanczos(M, n=4, prime=p, prune=True) as ctx:
        assert_pruned_like_oracle(oracle, ctx, ref, p)
        u, _ = ctx.pruned_index()
        empty = np.setdiff1d(np.arange(M.nrows), M.i)
        assert np.isin(empty, u).all()
    with pytest.raises(lib.BlkError, match="the kernel is \\{0\\}"):
        lib.BlockLanczos(chain(50), n=2, prime=p, prune=True)
    only_free = lib.SparseCOO(5, 3, np.array([0, 1], np.int32), np.array([0, 1], np.int32), np.array([1, 1], np.uint32))
    with pytest.raises(lib.BlkError, match="every vector on the 3 surviving unknowns"):
        lib.BlockLanczos(only_free, n=2, prime=p, prune=True)
    with pytest.raises(lib.BlkError, match="rhs"):
        lib.BlockLanczos(M, n=4, prime=p, prune=True, rhs=np.ones((400, 1), np.uint32))
    with lib.BlockLanczos(M, n=4, prime=p) as ctx:
        with pytest.raises(lib.BlkError, match="prune=True"):
            ctx.pruned_index()
        assert ctx.L.blk_pruned_index(ctx.h, None, None) != 0
        assert b"blk_create_pruned" in ctx.L.blk_last_error()
    bad = lib.SparseCOO(5, 5, np.array([0, 7], np.int32), np.array([0, 1], np.int32), np.array([1, 1], np.uint32))
    with pytest.raises(lib.BlkError, match="out of range"):
        lib.BlockLanczos(bad, n=2, prime=p, prune=True)


@pytest.mark.parametrize("p,n,right", [(65537, 1, False), (2147483647, 8, True)])
def test_prune_removing_nothing_gives_the_plain_context(lib, oracle, p, n, right):
    """BASELINE config-1 shape (30 entries per row): nothing is removed, and the loop is that of blk_create."""
    M, _ = lib.synth.baseline_config(1)
    if right:
        M = lib.SparseCOO(M.ncols, M.nrows, M.j, M.i, M.x)
    N = M.ncols if right else M.nrows
    with lib.BlockLanczos(M, n=n, prime=p, right=right, prune=True) as a:
        assert a.prune_stats == dict(N=N, Mc=a.orig_Mc, nnz=M.nnz, free=0, rounds=0)
        u, c = a.pruned_index()
        assert np.array_equal(u, np.arange(N)) and np.array_equal(c, np.arange(a.orig_Mc))
        ga = a.block_lanczos(oracle.start_block(N * n, p), stop_after=12, batch=4)
    with lib.BlockLanczos(M, n=n, prime=p, right=right) as b:
        gb = b.block_lanczos(oracle.start_block(N * n, p), stop_after=12, batch=4)
    for k in ("v", "tmp", "Av", "p"):
        assert np.array_equal(ga[k], gb[k]), k


@pytest.mark.parametrize("p,right", [(2, False), (2147483647, True)])
def test_prune_many_ctas_planted(lib, oracle, p, right):
    """4M unknowns at column weight 3: round 0 and the decrement passes span thousands of CTAs."""
    M = lib.synth.uniform_rows(4_000_000, 4_000_000, 3, seed=9)
    if right:
        M = lib.SparseCOO(M.ncols, M.nrows, M.j, M.i, M.x)
    ref = prune_oracle.prune(M, p, right)
    assert ref["stats"]["rounds"] >= 10
    with lib.BlockLanczos(M, n=1, prime=p, right=right, prune=True) as ctx:
        assert_pruned_like_oracle(oracle, ctx, ref, p)


def test_prune_device_coo_equals_host(lib, oracle):
    import torch
    p, n = 7, 8
    M = lib.synth.uniform_rows(3000, 3000, 3, seed=7)
    dev = torch.device("cuda", 0)
    ti = torch.from_numpy(M.i.astype(np.int32)).to(dev)
    tj = torch.from_numpy(M.j.astype(np.int32)).to(dev)
    tx = torch.from_numpy(M.x.astype(np.int32)).to(dev)
    torch.cuda.synchronize()
    coo = (M.nrows, M.ncols, M.nnz, ti.data_ptr(), tj.data_ptr(), tx.data_ptr())
    ref = prune_oracle.prune(M, p, False)
    with lib.BlockLanczos(n=n, prime=p, device_coo=coo, prune=True) as a:
        assert_pruned_like_oracle(oracle, a, ref, p)
        ga = a.block_lanczos(oracle.start_block(a.N * n, p), batch=64)
    with lib.BlockLanczos(M, n=n, prime=p, prune=True) as b:
        gb = b.block_lanczos(oracle.start_block(b.N * n, p), batch=64)
    assert ga["iters"] == gb["iters"]
    for k in ("v", "tmp", "Av", "p"):
        assert np.array_equal(ga[k], gb[k]), k


# ---- the driver ----------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def driver(lib):
    if not os.path.exists(DRIVER):
        import __graft_entry__
        __graft_entry__.build()
    return DRIVER


def cli(args, env=None, cwd=None):
    return subprocess.run([DRIVER, *args], capture_output=True, text=True, env=env, cwd=cwd)


@pytest.mark.parametrize("side,p,n", [("--left", 65537, 8), ("--right", 2147483647, 16), ("--left", 7, 4)])
def test_cli_prune_output_file(driver, lib, oracle, tmp_path, side, p, n):
    right = side == "--right"
    M = lib.synth.uniform_rows(2000, 1900, 3, seed=3)
    mtx, out = str(tmp_path / "m.mtx"), str(tmp_path / "k.mtx")
    lib.synth.write_mtx(mtx, M)
    res = cli(["--matrix", mtx, "--prime", str(p), "--n", str(n), side, "--prune", "--output-file", out])
    assert res.returncode == 0, (res.stdout[-2000:], res.stderr[-2000:])
    ref = prune_oracle.prune(M, p, right)
    st = ref["stats"]
    N, Mc = (M.ncols, M.nrows) if right else (M.nrows, M.ncols)
    line = (f"  - Prune: kept {st['N']} of {N} unknowns ({st['free']} free), {st['Mc']} of {Mc} constraints, "
            f"{st['nnz']} of {M.nnz} entries in {st['rounds']} rounds, ")
    assert line in res.stdout, res.stdout[-2000:]
    assert f"Expecting {1 + st['Mc'] // n} iterations" in res.stdout or st["Mc"] // n >= 999
    want = oracle.lanczos_run(ref["M"], n, p, right)
    x = lib.synth.read_kernel_block(out)
    assert np.array_equal(x, prune_oracle.lift(want["v"][:st["N"] * n].reshape(-1, n), ref["unknowns"], N))
    assert checker(oracle, lib, M, mtx, p, out, side)


def test_cli_prune_kernel_basis(driver, lib, oracle, tmp_path):
    p, n = 2, 64
    M = lib.synth.uniform_rows(2000, 2000, 3, seed=5)
    mtx, out = str(tmp_path / "m.mtx"), str(tmp_path / "k.mtx")
    lib.synth.write_mtx(mtx, M)
    res = cli(["--matrix", mtx, "--prime", str(p), "--n", str(n), "--left", "--prune", "--kernel-basis", "--output-file", out])
    assert res.returncode == 0, (res.stdout[-2000:], res.stderr[-2000:])
    ref = prune_oracle.prune(M, p, False)
    want = oracle.lanczos_run(ref["M"], n, p, False)
    X = kb_oracle.kernel_basis(ref["M"], want["v"], n, p, False)
    assert f"Kernel basis: {X.shape[1]} independent vectors" in res.stdout and "  - OK: kernel basis" in res.stdout
    x = lib.synth.read_kernel_block(out)
    assert np.array_equal(x, prune_oracle.lift(X, ref["unknowns"], M.nrows))
    assert checker(oracle, lib, M, mtx, p, out, "--left")


def test_cli_prune_usage_errors_and_everything_removed(driver, lib, tmp_path):
    M = lib.synth.uniform_rows(200, 180, 4, seed=1)
    mtx, out = str(tmp_path / "m.mtx"), str(tmp_path / "x.mtx")
    lib.synth.write_mtx(mtx, M)
    base = ["--matrix", mtx, "--prime", "65537", "--n", "4", "--prune"]
    for extra in (["--rhs", mtx, "--output-file", out], ["--checkpoint", "5"], ["--load-checkpoint"]):
        res = cli(base + extra, cwd=str(tmp_path))
        assert res.returncode == 1 and "--prune cannot be combined" in res.stderr, (extra, res.stderr[-500:])
    ch = str(tmp_path / "chain.mtx")
    lib.synth.write_mtx(ch, chain(40))
    res = cli(["--matrix", ch, "--prime", "65537", "--n", "4", "--prune", "--output-file", out])
    assert res.returncode == 1 and "the kernel is {0}" in res.stderr, res.stderr[-500:]
    assert not os.path.exists(out)


# ---- several GPUs --------------------------------------------------------------------------------
def _ngpus():
    import torch
    return torch.cuda.device_count()


@pytest.mark.parametrize("world", [2, 4, 8])
def test_prune_all_gpus_one_process(lib, oracle, world):
    if _ngpus() < world:
        pytest.skip(f"needs {world} GPUs")
    p, n = 3, 32
    M = lib.synth.powerlaw_rows(2800, 2600, mean=6, seed=21, with_empty_rows=7)
    ref = prune_oracle.prune(M, p, False)
    with lib.BlockLanczos(M, n=n, prime=p, rank=lib.BLK_RANK_ALL, world=world, prune=True) as ctx:
        assert ctx.prune_stats == ref["stats"]
        u, c = ctx.pruned_index()
        assert np.array_equal(u, ref["unknowns"]) and np.array_equal(c, ref["constraints"])
        got = ctx.block_lanczos(oracle.start_block(ctx.N * n, p), batch=32)
    with lib.BlockLanczos(M, n=n, prime=p, prune=True) as one:
        want = one.block_lanczos(oracle.start_block(one.N * n, p), batch=32)
    assert got["iters"] == want["iters"]
    for k in ("v", "tmp", "Av", "p"):
        assert np.array_equal(got[k], want[k]), k


def test_cli_prune_several_gpus(driver, lib, tmp_path):
    if _ngpus() < 2:
        pytest.skip("needs 2 GPUs")
    M = lib.synth.uniform_rows(3000, 2900, 3, seed=2)
    mtx = str(tmp_path / "m.mtx")
    lib.synth.write_mtx(mtx, M)
    files = {}
    for g in [1, 2] + ([4] if _ngpus() >= 4 else []) + ([8] if _ngpus() >= 8 else []):
        out = tmp_path / f"k{g}.mtx"
        res = cli(["--matrix", mtx, "--prime", "3", "--n", "16", "--left", "--prune", "--output-file", str(out)],
                  env=dict(os.environ, BLK_GPUS=str(g)), cwd=str(tmp_path))
        assert res.returncode == 0, (g, res.stdout[-2000:], res.stderr[-2000:])
        files[g] = out.read_bytes()
    assert len(set(files.values())) == 1


@pytest.mark.parametrize("world", [2, 4, 8])
def test_prune_one_process_per_gpu(lib, world):
    if _ngpus() < world:
        pytest.skip(f"needs {world} GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", str(29800 + world), os.path.join(ROOT, "tests", "prune_worker.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0 and f"PRUNE_OK world={world}" in res.stdout, (res.stdout[-3000:], res.stderr[-3000:])
