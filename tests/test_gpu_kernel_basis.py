"""GPU tests of the kernel-basis extraction (blk_kernel_basis, BlockLanczos.kernel_basis, --kernel-basis):
bit-identical to the CPU restatement (kbo_kernel_basis in tests/kb_oracle.c), k included, after whole loops at
small and large primes, on planted blocks large enough for many CTAs, with the state left untouched, through the driver and on
several GPUs.  Also runs complete loops at p = 2 and 3 against the oracle (the parity suite does not)."""
import os
import subprocess
import sys

import numpy as np
import pytest

import kb_oracle

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


def run_both(lib, oracle, M, n, p, right):
    Mp = M.reduced(p)
    N = M.ncols if right else M.nrows
    with lib.BlockLanczos(Mp, n=n, prime=p, right=right) as ctx:
        got = ctx.block_lanczos(oracle.start_block(N * n, p), batch=64)
        X = ctx.kernel_basis()
    want = oracle.lanczos_run(Mp, n, p, right)
    return Mp, N, got, want, X


@pytest.mark.parametrize("p", [2, 3])
@pytest.mark.parametrize("n", [1, 4, 16, 32, 64])
def test_loop_at_small_primes_matches_oracle(lib, oracle, p, n):
    for right in (False, True):
        for M in matrices(lib, right)[:2]:
            _, _, got, want, _ = run_both(lib, oracle, M, n, p, right)
            assert got["iters"] == want["iters"] and got["stopped"] == want["stopped"], (p, n, right)
            for k in ("v", "tmp", "Av", "p"):
                assert np.array_equal(got[k], want[k]), (p, n, right, k)


@pytest.mark.parametrize("right", [False, True])
@pytest.mark.parametrize("n", NS)
@pytest.mark.parametrize("p", PRIMES)
def test_kernel_basis_matches_oracle_after_the_loop(lib, oracle, p, n, right):
    for mi, M in enumerate(matrices(lib, right)):
        Mp, N, got, want, X = run_both(lib, oracle, M, n, p, right)
        assert np.array_equal(got["v"], want["v"]), (mi,)
        ref = kb_oracle.kernel_basis(Mp, want["v"][:N * n], n, p, right)
        assert X.shape == ref.shape and np.array_equal(X, ref), (mi, X.shape, ref.shape)
        if X.shape[1]:
            assert not oracle.sparse_matrix_vector_product(Mp, np.ascontiguousarray(X).ravel(), not right,
                                                           X.shape[1], p).any()


def planted(N, n, r, p, seed):
    rng = np.random.default_rng(seed)
    a = rng.integers(0, p, size=(N, r), dtype=np.uint64)
    b = rng.integers(0, p, size=(r, n), dtype=np.uint64)
    v = np.zeros((N, n), dtype=np.uint64)
    for i in range(r):                       # exact: every partial sum stays < 2^63
        v = (v + (a[:, i:i + 1] * b[i:i + 1, :]) % p) % p
    return v.astype(np.uint32)


@pytest.mark.parametrize("n,p,r,env", [
    (16, 65537, 11, {}),
    (16, 2147483647, 16, {"BLK_HOT_MIN_BYTES": "0", "BLK_HOT_BYTES": "8192"}),
    (13, 2, 9, {}),
    (4, 3, 3, {"BLK_BAND_BYTES": "8192"}),
    (3, 7, 3, {"BLK_BAND_BYTES": "8192"}),
])
def test_kernel_basis_many_ctas_planted(lib, oracle, monkeypatch, n, p, r, env):
    """A planted low-rank v on a tall matrix (Mc < n bounds the rank of T), T computed into scratch: the
    reductions run on hundreds of CTAs, which merge their bases."""
    for k, val in env.items():
        monkeypatch.setenv(k, val)
    N, Mc = 4_200_000, max(1, n // 2)
    M = lib.synth.uniform_rows(N, Mc, 2, seed=n).reduced(p)
    v = planted(N, n, r, p, seed=p % 97 + n)
    with lib.BlockLanczos(M, n=n, prime=p) as ctx:
        ctx.set_state(v.ravel())
        X = ctx.kernel_basis()
    ref = kb_oracle.kernel_basis(M, v.ravel(), n, p, False)
    assert X.shape == ref.shape and np.array_equal(X, ref)
    assert X.shape[1] > 0


@pytest.mark.parametrize("n,p,right", [(8, 65537, False), (16, 2147483647, True), (4, 2, False)])
def test_kernel_basis_leaves_the_state_untouched(lib, oracle, n, p, right):
    M = matrices(lib, right)[1].reduced(p)
    N = M.ncols if right else M.nrows
    with lib.BlockLanczos(M, n=n, prime=p, right=right) as ctx:
        ctx.set_state(oracle.start_block(N * n, p))
        X0 = ctx.kernel_basis()                      # nothing has run: T goes to scratch
        assert np.array_equal(X0, kb_oracle.kernel_basis(M, oracle.start_block(N * n, p), n, p, right))
        ctx.iterate(4)
        before = ctx.get_state()
        X = ctx.kernel_basis()
        after = ctx.get_state()
        for k in before:
            assert np.array_equal(before[k], after[k]), k
        want4 = oracle.lanczos_run(M, n, p, right, stop_after=4)
        assert np.array_equal(X, kb_oracle.kernel_basis(M, want4["v"][:N * n], n, p, right))
        it, _ = ctx.iterate(3)
        got = ctx.get_state()
        want = oracle.lanczos_run(M, n, p, right, stop_after=7)
        assert it == want["iters"]
        for k in ("v", "tmp", "Av", "p"):
            assert np.array_equal(got[k], want[k]), k


# ---- the driver ----------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def driver(lib):
    if not os.path.exists(DRIVER):
        import __graft_entry__
        __graft_entry__.build()
    return DRIVER


def cli(args, env=None, cwd=None):
    return subprocess.run([DRIVER, *args], capture_output=True, text=True, env=env, cwd=cwd)


def checker(oracle, lib, M, mtx, p, kernel, side):
    """checker_modp's verdict (as in test_gpu_cli.py): the CPU oracle, plus the reference's checker where built."""
    x = lib.synth.read_kernel_block(kernel)
    ok = bool(x.any()) and bool((x < p).all()) and \
        not oracle.sparse_matrix_vector_product(M.reduced(p), x.ravel(), side == "--left", x.shape[1], p).any()
    exe = os.path.join(ROOT, "oracle", "_ref", "checker_modp")
    if os.path.exists(exe):
        r = subprocess.run([exe, "--matrix", mtx, "--prime", str(p), "--kernel", kernel, side], capture_output=True, text=True)
        assert (r.returncode == 0 and r.stdout.strip().endswith("OK")) == ok, r.stdout[-2000:]
    return ok


def test_cli_kernel_basis(driver, lib, oracle, tmp_path):
    p, n = 2, 64
    M = lib.synth.uniform_rows(2000, 1900, 5, seed=1)
    mtx = str(tmp_path / "m.mtx")
    lib.synth.write_mtx(mtx, M)
    args = ["--matrix", mtx, "--prime", str(p), "--n", str(n), "--left"]
    plain, basis = str(tmp_path / "plain.mtx"), str(tmp_path / "basis.mtx")
    r = cli(args + ["--output-file", plain])
    assert r.returncode == 0, r.stderr[-2000:]
    r = cli(args + ["--kernel-basis", "--output-file", basis])
    assert r.returncode == 0, r.stderr[-2000:]
    want = oracle.lanczos_run(M.reduced(p), n, p, False)
    ref = kb_oracle.kernel_basis(M.reduced(p), want["v"][:M.nrows * n], n, p, False)
    k = ref.shape[1]
    assert k > 0 and f"Kernel basis: {k} independent vectors" in r.stdout and "OK: kernel basis * M == 0" in r.stdout
    x = lib.synth.read_kernel_block(basis)
    assert x.shape == (M.nrows, k) and np.array_equal(x, ref)
    assert checker(oracle, lib, M, mtx, p, basis, "--left")
    # without the option the file is the block v, as before
    assert np.array_equal(lib.synth.read_kernel_block(plain), want["v"][:M.nrows * n].reshape(M.nrows, n))
    # --kernel-basis alone: usage
    r = cli(["--matrix", mtx, "--prime", str(p), "--kernel-basis"])
    assert r.returncode == 0 and "--kernel-basis" in r.stdout and "Options:" in r.stdout


def test_cli_kernel_basis_none(driver, lib, tmp_path):
    """A non-singular matrix has no kernel vector: exit status 1 and no file."""
    N, p = 300, 65537
    rng = np.random.default_rng(2)
    i = np.concatenate([np.arange(N), rng.integers(0, N, 900)])
    j = np.concatenate([np.arange(N), rng.integers(0, N, 900)])
    keep = j >= i                                    # upper triangular with a non-zero diagonal
    x = rng.integers(1, 100, size=i.shape[0])
    M = lib.SparseCOO(N, N, i[keep].astype(np.int32), j[keep].astype(np.int32), x[keep].astype(np.uint32))
    mtx, out = str(tmp_path / "m.mtx"), str(tmp_path / "k.mtx")
    lib.synth.write_mtx(mtx, M)
    r = cli(["--matrix", mtx, "--prime", str(p), "--n", "4", "--kernel-basis", "--output-file", out])
    assert r.returncode == 1 and "Kernel basis: 0 independent vectors" in r.stdout, (r.stdout[-1000:], r.stderr[-1000:])
    assert not os.path.exists(out)


# ---- several GPUs --------------------------------------------------------------------------------
def _ngpus():
    import torch
    return torch.cuda.device_count()


def test_cli_kernel_basis_several_gpus(driver, lib, tmp_path):
    if _ngpus() < 2:
        pytest.skip("needs 2 GPUs")
    M = lib.synth.powerlaw_rows(2800, 2600, mean=6, seed=21, with_empty_rows=7)
    mtx = str(tmp_path / "m.mtx")
    lib.synth.write_mtx(mtx, M)
    files = {}
    for g in [1, 2] + ([4] if _ngpus() >= 4 else []) + ([8] if _ngpus() >= 8 else []):
        out = tmp_path / f"k{g}.mtx"
        r = cli(["--matrix", mtx, "--prime", "3", "--n", "32", "--left", "--kernel-basis", "--output-file", str(out)],
                env=dict(os.environ, BLK_GPUS=str(g)), cwd=str(tmp_path))
        assert r.returncode == 0, (g, r.stdout[-2000:], r.stderr[-2000:])
        files[g] = out.read_bytes()
    assert len(set(files.values())) == 1


@pytest.mark.parametrize("world", [2, 4, 8])
def test_kernel_basis_one_process_per_gpu(lib, world):
    if _ngpus() < world:
        pytest.skip(f"needs {world} GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", str(29600 + world), os.path.join(ROOT, "tests", "kb_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and f"KB_OK world={world}" in r.stdout, (r.stdout[-3000:], r.stderr[-3000:])
