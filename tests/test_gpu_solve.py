"""GPU tests of the inhomogeneous solve (blk_create_system + blk_solve, BlockLanczos(rhs=...).solve(), --rhs):
bit-identical to the CPU restatement (svo_solve in tests/solve_oracle.c), found included, after whole loops at small
and large primes, on planted multi-million-row problems whose dense right-hand side spans many tiles, with the state
left untouched, through the driver and on several GPUs."""
import os
import subprocess
import sys

import numpy as np
import pytest

import solve_oracle

from conftest import ROOT

pytestmark = pytest.mark.gpu

DRIVER = os.path.join(ROOT, "block-lanczos-algorithm-parallelization_b200", "driver", "lanczos_modp")
PRIMES = [2, 3, 7, 65537, 2147483647]
NS = [1, 2, 3, 8, 13, 16, 32, 64]
ENV_KNOBS = ("BLK_HOT", "BLK_HOT_MIN_BYTES", "BLK_HOT_BYTES", "BLK_BANDS", "BLK_BAND_BYTES", "BLK_GPUS")


@pytest.fixture(autouse=True)
def _clean_env(monkeypatch):
    for k in ENV_KNOBS:
        monkeypatch.delenv(k, raising=False)


def matrices(lib, right):
    """uniform, power law with empty rows, tall (Mc < N); oriented so that N is the first size for --left."""
    s = lib.synth
    mats = [s.uniform_rows(420, 400, 5, seed=3), s.powerlaw_rows(420, 400, mean=6, seed=4, with_empty_rows=9),
            s.uniform_rows(500, 150, 4, seed=5)]
    if right:
        mats = [lib.SparseCOO(M.ncols, M.nrows, M.j, M.i, M.x) for M in mats]
    return mats


def product(oracle, M, x, right, p):
    """M x (--right) or M^T x (--left) for an N x w block x: Mc x w."""
    x = np.ascontiguousarray(x, dtype=np.uint32)
    return oracle.sparse_matrix_vector_product(M, x.ravel(), not right, x.shape[1], p).reshape(-1, x.shape[1])


def planted_rhs(oracle, M, r, p, right, seed):
    N = M.ncols if right else M.nrows
    X0 = np.random.default_rng(seed).integers(0, p, size=(N, r), dtype=np.int64).astype(np.uint32)
    return product(oracle, M, X0, right, p)


def run_both(lib, oracle, M, Bm, n, p, right):
    A = solve_oracle.augmented(M, Bm, p, right)
    Np = A.ncols if right else A.nrows
    with lib.BlockLanczos(M, n=n, prime=p, right=right, rhs=Bm) as ctx:
        assert ctx.N == Np and ctx.N0 == Np - Bm.shape[1] and ctx.info()["nrhs"] == Bm.shape[1]
        got = ctx.block_lanczos(oracle.start_block(Np * n, p), batch=64)
        x, found = ctx.solve()
    want = oracle.lanczos_run(A, n, p, right)
    return A, Np, got, want, x, found


@pytest.mark.parametrize("right", [False, True])
@pytest.mark.parametrize("n", NS)
@pytest.mark.parametrize("p", PRIMES)
def test_solve_matches_oracle_after_the_loop(lib, oracle, p, n, right):
    for r in sorted({1, min(2, n), n}):
        for mi, M in enumerate(matrices(lib, right)):
            Mp = M.reduced(p)
            Bm = planted_rhs(oracle, Mp, r, p, right, seed=10 * mi + r)
            A, Np, got, want, x, found = run_both(lib, oracle, Mp, Bm, n, p, right)
            assert got["iters"] == want["iters"] and np.array_equal(got["v"], want["v"]), (mi, r)
            rx, rf = solve_oracle.solve(Mp, Bm, want["v"][:Np * n], n, p, right)
            assert np.array_equal(found, rf), (mi, r, found, rf)
            assert x.shape == rx.shape and np.array_equal(x, rx), (mi, r)
            y = product(oracle, Mp, x, right, p)
            for j in np.nonzero(found)[0]:
                assert np.array_equal(y[:, j], Bm[:, j] % p), (mi, r, j)


def mulmod(a, b, p):
    """(a @ b) mod p for uint32 blocks, exact for p < 2^31 (one % per product)."""
    out = np.zeros((a.shape[0], b.shape[1]), dtype=np.uint64)
    for k in range(a.shape[1]):
        out = (out + (a[:, k:k + 1].astype(np.uint64) * b[k:k + 1, :].astype(np.uint64)) % p) % p
    return out.astype(np.uint32)


def planted_block(N, Mc, n, r, p, right, seed, lib):
    """A sparse M with a dense consistent B = M X0 (M^T X0 for --left) and a block v ((N + r) x n) whose span holds
    the r solutions (X0_j ; e_j) and n - r random vectors, mixed by a random unit upper triangular matrix."""
    rng = np.random.default_rng(seed)
    M = lib.synth.uniform_rows(Mc, N, 3, seed=seed) if right else lib.synth.uniform_rows(N, Mc, 3, seed=seed)
    M = M.reduced(p)
    X0 = rng.integers(0, p, size=(N, r), dtype=np.int64).astype(np.uint32)
    S = np.zeros((N + r, n), dtype=np.uint32)
    S[:N, :r] = X0
    S[N + np.arange(r), np.arange(r)] = 1
    S[:, r:] = rng.integers(0, p, size=(N + r, n - r), dtype=np.int64).astype(np.uint32)
    G = np.triu(rng.integers(0, p, size=(n, n), dtype=np.int64), 1) + np.eye(n, dtype=np.int64)   # invertible
    v = mulmod(S, G.astype(np.uint32), p)
    return M, X0, v


@pytest.mark.parametrize("n,p,r,right,env", [
    (16, 65537, 4, False, {}),
    (16, 2147483647, 8, False, {"BLK_HOT_MIN_BYTES": "0", "BLK_HOT_BYTES": "8192"}),
    (8, 2, 3, True, {"BLK_HOT_MIN_BYTES": "0", "BLK_HOT_BYTES": "8192"}),
    (4, 3, 2, True, {"BLK_BAND_BYTES": "8192"}),
    (2, 7, 1, False, {"BLK_BAND_BYTES": "8192"}),
])
def test_solve_many_ctas_planted(lib, oracle, monkeypatch, n, p, r, right, env):
    """3M unknowns, 1.5M equations: each right-hand side is one row or column of about 1.5M entries of the
    augmented matrix, spanning thousands of tiles, and the reductions run on hundreds of CTAs."""
    for k, val in env.items():
        monkeypatch.setenv(k, val)
    N, Mc = 3_000_000, 1_500_000
    M, X0, v = planted_block(N, Mc, n, r, p, right, seed=n + r, lib=lib)
    Bm = product(oracle, M, X0, right, p)
    assert np.count_nonzero(Bm) > Mc * r // 4           # dense: at p = 2 about half the entries are zero
    with lib.BlockLanczos(M, n=n, prime=p, right=right, rhs=Bm) as ctx:
        ctx.set_state(v.ravel())
        x, found = ctx.solve()
    rx, rf = solve_oracle.solve(M, Bm, v, n, p, right)
    assert np.array_equal(found, rf) and found.all(), (found, rf)
    assert np.array_equal(x, rx)
    assert np.array_equal(product(oracle, M, x, right, p), Bm)


@pytest.mark.parametrize("n,p,right", [(8, 65537, False), (16, 2147483647, True), (4, 2, False)])
def test_solve_leaves_the_state_untouched(lib, oracle, n, p, right):
    M = matrices(lib, right)[1].reduced(p)
    Bm = planted_rhs(oracle, M, min(n, 3), p, right, seed=5)
    A = solve_oracle.augmented(M, Bm, p, right)
    Np = A.ncols if right else A.nrows
    with lib.BlockLanczos(M, n=n, prime=p, right=right, rhs=Bm) as ctx:
        ctx.set_state(oracle.start_block(Np * n, p))
        x0, f0 = ctx.solve()                          # nothing has run: T goes to scratch
        rx, rf = solve_oracle.solve(M, Bm, oracle.start_block(Np * n, p), n, p, right)
        assert np.array_equal(x0, rx) and np.array_equal(f0, rf)
        ctx.iterate(4)
        before = ctx.get_state()
        x, found = ctx.solve()
        after = ctx.get_state()
        for k in before:
            assert np.array_equal(before[k], after[k]), k
        want4 = oracle.lanczos_run(A, n, p, right, stop_after=4)
        rx, rf = solve_oracle.solve(M, Bm, want4["v"][:Np * n], n, p, right)
        assert np.array_equal(x, rx) and np.array_equal(found, rf)
        it, _ = ctx.iterate(3)
        got = ctx.get_state()
        want = oracle.lanczos_run(A, n, p, right, stop_after=7)
        assert it == want["iters"]
        for k in ("v", "tmp", "Av", "p"):
            assert np.array_equal(got[k], want[k]), k


def test_solve_needs_a_system_context(lib):
    M = lib.synth.uniform_rows(50, 40, 3).reduced(65537)
    with lib.BlockLanczos(M, n=2, prime=65537) as ctx:
        assert ctx.info()["nrhs"] == 0
        x = np.zeros(64, dtype=np.uint32)
        f = np.zeros(2, dtype=np.int32)
        assert ctx.L.blk_solve(ctx.h, x.ctypes.data, f.ctypes.data) != 0
        assert b"blk_create_system" in ctx.L.blk_last_error()
    with pytest.raises(lib.BlkError, match="right-hand sides"):
        lib.BlockLanczos(M, n=2, prime=65537, rhs=np.ones((40, 3), dtype=np.uint32))


# ---- the driver ----------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def driver(lib):
    if not os.path.exists(DRIVER):
        import __graft_entry__
        __graft_entry__.build()
    return DRIVER


def cli(args, env=None, cwd=None):
    return subprocess.run([DRIVER, *args], capture_output=True, text=True, env=env, cwd=cwd)


def write_array(path, a):
    """MatrixMarket array integer general, column-major (the format of the driver's output files)."""
    a = np.asarray(a)
    with open(path, "w") as f:
        f.write("%%MatrixMarket matrix array integer general\n%right-hand sides\n")
        f.write(f"{a.shape[0]} {a.shape[1]}\n")
        for col in range(a.shape[1]):
            f.write("\n".join(str(int(t)) for t in a[:, col]) + "\n")


@pytest.mark.parametrize("side,p,n,r", [("--right", 65537, 16, 4), ("--left", 2147483647, 16, 1), ("--left", 2, 64, 8),
                                        ("--right", 3, 16, 3)])
def test_cli_rhs(driver, lib, oracle, tmp_path, side, p, n, r):
    right = side == "--right"
    M = lib.synth.uniform_rows(2000, 1900, 5, seed=1)
    Mp = M.reduced(p)
    b = planted_rhs(oracle, Mp, r, p, right, seed=r)
    # every 7th row written as a negative number of the same residue: -k is read as 2^32 - k, like the matrix loader
    Bm = b.astype(np.int64)
    k = ((1 << 32) - Bm[::7]) % p
    Bm[::7] = np.where(k > 0, -k, Bm[::7])
    mtx, rhs, out = str(tmp_path / "m.mtx"), str(tmp_path / "b.mtx"), str(tmp_path / "x.mtx")
    lib.synth.write_mtx(mtx, M)
    write_array(rhs, Bm)
    res = cli(["--matrix", mtx, "--prime", str(p), "--n", str(n), side, "--rhs", rhs, "--output-file", out])
    assert res.returncode == 0, (res.stdout[-2000:], res.stderr[-2000:])
    assert f"Solve: {r} of {r} right-hand sides solved" in res.stdout and "  - OK: " in res.stdout, res.stdout[-2000:]
    x = lib.synth.read_kernel_block(out)
    N = M.ncols if right else M.nrows
    assert x.shape == (N, r) and (x < p).all()
    assert (Bm < 0).any() and np.array_equal(solve_oracle.reduce_rhs(Bm, p), b)
    assert np.array_equal(product(oracle, Mp, x, right, p), b)
    # the same numbers as the library and the CPU restatement
    A = solve_oracle.augmented(Mp, b, p, right)
    want = oracle.lanczos_run(A, n, p, right)
    Np = N + r
    rx, rf = solve_oracle.solve(Mp, b, want["v"][:Np * n], n, p, right)
    assert rf.all() and np.array_equal(x, rx)


def test_cli_rhs_inconsistent(driver, lib, oracle, tmp_path):
    """b non-zero on an empty row of M: exit status 1, the unsolved column named, no file."""
    p, n = 65537, 8
    M = lib.synth.uniform_rows(600, 600, 5, seed=2)
    keep = M.i != 11
    M = lib.SparseCOO(M.nrows, M.ncols, M.i[keep], M.j[keep], M.x[keep])
    Bm = planted_rhs(oracle, M.reduced(p), 2, p, True, seed=3)
    Bm[11, 1] = 5
    mtx, rhs, out = str(tmp_path / "m.mtx"), str(tmp_path / "b.mtx"), str(tmp_path / "x.mtx")
    lib.synth.write_mtx(mtx, M)
    write_array(rhs, Bm)
    res = cli(["--matrix", mtx, "--prime", str(p), "--n", str(n), "--right", "--rhs", rhs, "--output-file", out])
    assert res.returncode == 1, (res.stdout[-2000:], res.stderr[-2000:])
    assert "Solve: 1 of 2 right-hand sides solved" in res.stdout
    assert "right-hand side(s) 2" in res.stderr and "inconsistent" in res.stderr
    assert not os.path.exists(out)


def test_cli_rhs_usage_errors(driver, lib, tmp_path):
    M = lib.synth.uniform_rows(200, 180, 4, seed=1)
    mtx, rhs, out = str(tmp_path / "m.mtx"), str(tmp_path / "b.mtx"), str(tmp_path / "x.mtx")
    lib.synth.write_mtx(mtx, M)
    write_array(rhs, np.ones((180, 2), dtype=np.int64))          # --left: Mc = 180 rows
    base = ["--matrix", mtx, "--prime", "65537", "--n", "4"]
    for extra, msg in [([], "needs --output-file"),
                       (["--output-file", out, "--kernel-basis"], "cannot be combined"),
                       (["--stop-after", "3"], "needs --output-file"),
                       (["--output-file", out, "--stop-after", "3"], "cannot be combined"),
                       (["--output-file", out, "--checkpoint", "5"], "cannot be combined"),
                       (["--output-file", out, "--load-checkpoint"], "cannot be combined")]:
        res = cli(base + ["--rhs", rhs] + extra, cwd=str(tmp_path))
        assert res.returncode == 1 and msg in res.stderr, (extra, res.stdout[-500:], res.stderr[-500:])
    # wrong number of rows (--right needs 200), more right-hand sides than n
    res = cli(base + ["--right", "--rhs", rhs, "--output-file", out])
    assert res.returncode == 1 and "expected 200" in res.stderr, res.stderr[-500:]
    wide = str(tmp_path / "w.mtx")
    write_array(wide, np.ones((180, 5), dtype=np.int64))
    res = cli(base + ["--rhs", wide, "--output-file", out])
    assert res.returncode == 1 and "more than the blocking factor" in res.stderr, res.stderr[-500:]
    bad = str(tmp_path / "bad.mtx")
    with open(bad, "w") as f:
        f.write("%%MatrixMarket matrix coordinate integer general\n180 2 0\n")
    res = cli(base + ["--rhs", bad, "--output-file", out])
    assert res.returncode == 1 and "not supported" in res.stderr, res.stderr[-500:]
    assert not os.path.exists(out)


# ---- several GPUs --------------------------------------------------------------------------------
def _ngpus():
    import torch
    return torch.cuda.device_count()


def test_cli_rhs_several_gpus(driver, lib, oracle, tmp_path):
    if _ngpus() < 2:
        pytest.skip("needs 2 GPUs")
    p = 3
    M = lib.synth.powerlaw_rows(2800, 2600, mean=6, seed=21, with_empty_rows=7)
    mtx, rhs = str(tmp_path / "m.mtx"), str(tmp_path / "b.mtx")
    lib.synth.write_mtx(mtx, M)
    write_array(rhs, planted_rhs(oracle, M.reduced(p), 4, p, False, seed=1))
    files = {}
    for g in [1, 2] + ([4] if _ngpus() >= 4 else []) + ([8] if _ngpus() >= 8 else []):
        out = tmp_path / f"x{g}.mtx"
        res = cli(["--matrix", mtx, "--prime", str(p), "--n", "32", "--left", "--rhs", rhs, "--output-file", str(out)],
                  env=dict(os.environ, BLK_GPUS=str(g)), cwd=str(tmp_path))
        assert res.returncode == 0, (g, res.stdout[-2000:], res.stderr[-2000:])
        files[g] = out.read_bytes()
    assert len(set(files.values())) == 1


@pytest.mark.parametrize("world", [2, 4, 8])
def test_solve_one_process_per_gpu(lib, world):
    if _ngpus() < world:
        pytest.skip(f"needs {world} GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", str(29700 + world), os.path.join(ROOT, "tests", "solve_worker.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0 and f"SOLVE_OK world={world}" in res.stdout, (res.stdout[-3000:], res.stderr[-3000:])
