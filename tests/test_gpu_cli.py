"""GPU tests of the drop-in driver: same command line and files as the reference program, output
files byte-identical to the reference's (golden sha256 made by running the unmodified reference),
accepted by checker_modp's test, checkpoint files interchangeable with the reference's.

The reference is not part of this repository.  Where its build exists (oracle/_ref), its checker and
its OpenMP program are run as well; every test also stands without them: checker_modp's verdict is
evaluated with the CPU oracle, and checkpoint files are compared with the oracle's state.
"""
import hashlib
import json
import os
import subprocess

import numpy as np
import pytest

from conftest import GOLDEN, ROOT, golden_cases, load_golden

pytestmark = pytest.mark.gpu

DRIVER = os.path.join(ROOT, "block-lanczos-algorithm-parallelization_b200", "driver", "lanczos_modp")
REF = os.path.join(ROOT, "oracle", "_ref")


@pytest.fixture(scope="module")
def driver(lib):
    if not os.path.exists(DRIVER):
        import __graft_entry__
        __graft_entry__.build()
    return DRIVER


def run(cmd, cwd=None, env=None):
    r = subprocess.run(cmd, capture_output=True, text=True, cwd=cwd, env=env)
    assert r.returncode == 0, (cmd, r.stdout[-2000:], r.stderr[-2000:])
    return r


def sha(path):
    return hashlib.sha256(open(path, "rb").read()).hexdigest()


def checker(oracle, lib, M, mtx, p, kernel, side):
    """checker_modp's verdict on a kernel file (checker_modp.c:146-204) for the matrix M written to mtx: every
    entry < p, the block not all zero, and x^T M == 0 (--left) or M x == 0 (--right), evaluated with the CPU
    oracle.  Where the reference's own checker has been built, it must give the same verdict."""
    x = lib.synth.read_kernel_block(kernel)
    ok = bool(x.any()) and bool((x < p).all()) and \
        not oracle.sparse_matrix_vector_product(M.reduced(p), x.ravel(), side == "--left", x.shape[1], p).any()
    exe = os.path.join(REF, "checker_modp")
    if os.path.exists(exe):
        r = subprocess.run([exe, "--matrix", mtx, "--prime", str(p), "--kernel", kernel, side], capture_output=True, text=True)
        assert (r.returncode == 0 and r.stdout.strip().endswith("OK")) == ok, r.stdout[-2000:]
    return ok


def assert_checkpoint_is_oracle_state(oracle, M, p, n, right, K, d):
    """The checkpoint files in d hold the four blocks of the reference's loop after K iterations, one residue
    per line, padded rows included (so tmp rows [N, Mc) keep M^T v of iteration K)."""
    want = oracle.lanczos_run(M.reduced(p), n, p, right, stop_after=K)
    assert want["iters"] == K and not want["stopped"]
    for f, k in (("v.txt", "v"), ("tmp.txt", "tmp"), ("Av.txt", "Av"), ("p.txt", "p")):
        assert (d / f).read_text() == "".join(f"{t}\n" for t in want[k]), f


@pytest.mark.parametrize("name", golden_cases("cli_"))
def test_cli_output_file_identical_to_reference(driver, lib, oracle, tmp_path, name):
    z, M = load_golden(name)
    p, n, right = int(z["p"]), int(z["n"]), bool(z["right"])
    mtx, out = str(tmp_path / "m.mtx"), str(tmp_path / "k.mtx")
    lib.synth.write_mtx(mtx, M)
    side = "--right" if right else "--left"
    r = run([driver, "--matrix", mtx, "--prime", str(p), "--n", str(n), side, "--output-file", out])
    assert f"after {int(z['iters'])} iterations" in r.stdout
    assert ("OK:    v != 0" in r.stdout) == bool(z["ok_v"]) and ("OK: vt*M == 0" in r.stdout) == bool(z["ok_vtM"])
    assert sha(out) == bytes(z["file_sha256"]).hex()
    assert checker(oracle, lib, M, mtx, p, out, side) == bool(z["checker_ok"])


@pytest.mark.parametrize("cfg", ["cfg1", "cfg2", "cfg3"])
def test_cli_full_baseline_config_identical_to_reference(driver, lib, oracle, tmp_path, cfg):
    """BASELINE.json configs[0], [1] and [2] at full size through the real CLI."""
    want = json.load(open(os.path.join(GOLDEN, "full_configs.json")))[cfg]
    M, a = lib.synth.baseline_config(int(cfg[3:]))
    mtx, out = str(tmp_path / "m.mtx"), str(tmp_path / "k.mtx")
    lib.synth.write_mtx(mtx, M)
    side = "--right" if a["right"] else "--left"
    r = run([driver, "--matrix", mtx, "--prime", str(a["p"]), "--n", str(a["n"]), side, "--output-file", out])
    assert f"after {want['iters']} iterations" in r.stdout
    assert sha(out) == want["kernel_file_sha256"]
    assert checker(oracle, lib, M, mtx, a["p"], out, side) == want["checker_ok"]


def test_cli_stop_after_and_usage(driver, lib, tmp_path):
    M = lib.synth.uniform_rows(300, 280, 5, seed=8)
    mtx = str(tmp_path / "m.mtx")
    lib.synth.write_mtx(mtx, M)
    r = run([driver, "--matrix", mtx, "--prime", "65537", "--n", "4", "--stop-after", "7"])
    assert "after 7 iterations" in r.stdout and "Final check" not in r.stdout
    assert "Not saving result" in r.stdout
    # usage() exits 0 (sequential/lanczos_modp.c:138), also when both exclusive options are given
    r = subprocess.run([driver, "--matrix", mtx, "--prime", "65537", "--stop-after", "3", "--output-file", "x"],
                       capture_output=True, text=True)
    assert r.returncode == 0 and "mutually exclusive" in r.stdout
    r = subprocess.run([driver, "--matrix", str(tmp_path / "missing.mtx"), "--prime", "65537"], capture_output=True, text=True)
    assert r.returncode == 1 and "impossible d'ouvrir" in r.stderr
    r = subprocess.run([driver, "--matrix", mtx, "--prime", "65537", "--bogus"], capture_output=True, text=True)
    assert r.returncode == 1


def test_cli_checkpoint_files_match_reference_and_resume(driver, lib, oracle, tmp_path):
    """--checkpoint 0 --stop-after K writes v/tmp/Av/p.txt after every iteration; they must hold the
    oracle's state and be byte-identical to the reference's OpenMP build run with one thread (SURVEY.md
    F3, F5), and a run resumed with --load-checkpoint must end in the same kernel file as an
    uninterrupted one."""
    p, n = 1073741789, 4
    M = lib.synth.uniform_nnz(420, 380, 2600, seed=13, order="col")       # N=420 > Mc=380: tmp keeps rows of v
    mtx = str(tmp_path / "m.mtx")
    lib.synth.write_mtx(mtx, M)
    ours, theirs = tmp_path / "ours", tmp_path / "ref"
    ours.mkdir(); theirs.mkdir()
    K = 9
    args = ["--matrix", mtx, "--prime", str(p), "--n", str(n), "--left"]
    run([driver, *args, "--checkpoint", "0", "--stop-after", str(K)], cwd=str(ours))
    for f in ("v.txt", "tmp.txt", "Av.txt", "p.txt", "verbosity.txt"):
        assert (ours / f).exists(), f
    assert open(ours / "verbosity.txt").read().split()[0] == str(K)
    assert_checkpoint_is_oracle_state(oracle, M, p, n, False, K, ours)
    ref_exe = os.path.join(REF, "lanczos_modp_omp")
    if os.path.exists(ref_exe):
        env = dict(os.environ, OMP_NUM_THREADS="1")
        run([ref_exe, *args, "--checkpoint", "0", "--stop-after", str(K)], cwd=str(theirs), env=env)
        for f in ("v.txt", "tmp.txt", "Av.txt", "p.txt"):
            assert sha(ours / f) == sha(theirs / f), f
    # resume from our checkpoint and compare with an uninterrupted run
    full, res = str(tmp_path / "full.mtx"), str(ours / "resumed.mtx")
    run([driver, *args, "--output-file", full])
    run([driver, *args, "--load-checkpoint", "--output-file", res], cwd=str(ours))
    assert sha(full) == sha(res)
    if os.path.exists(ref_exe):
        # the reference resumes from OUR files, and we resume from ITS files
        ref_res = str(theirs / "ref_resumed_from_ours.mtx")
        for f in ("v.txt", "tmp.txt", "Av.txt", "p.txt", "verbosity.txt"):
            (theirs / f).write_bytes((ours / f).read_bytes())
        run([ref_exe, *args, "--load-checkpoint", "--output-file", ref_res], cwd=str(theirs),
            env=dict(os.environ, OMP_NUM_THREADS="1"))
        assert sha(ref_res) == sha(full)


def test_cli_wide_matrix_tmp_tail(driver, lib, oracle, tmp_path):
    """Mc > N: tmp rows [N,Mc) keep M^T v of the previous iteration in the reference's checkpoint."""
    p, n, K = 65537, 2, 5
    M = lib.synth.uniform_nnz(150, 260, 1500, seed=19)
    mtx = str(tmp_path / "m.mtx")
    lib.synth.write_mtx(mtx, M)
    ours, theirs = tmp_path / "o", tmp_path / "r"
    ours.mkdir(); theirs.mkdir()
    args = ["--matrix", mtx, "--prime", str(p), "--n", str(n), "--left", "--checkpoint", "0", "--stop-after", str(K)]
    run([driver, *args], cwd=str(ours))
    assert_checkpoint_is_oracle_state(oracle, M, p, n, False, K, ours)
    ref_exe = os.path.join(REF, "lanczos_modp_omp")
    if os.path.exists(ref_exe):
        run([ref_exe, *args], cwd=str(theirs), env=dict(os.environ, OMP_NUM_THREADS="1"))
        for f in ("v.txt", "tmp.txt", "Av.txt", "p.txt"):
            assert sha(ours / f) == sha(theirs / f), f


@pytest.mark.parametrize("n", [16, 13])
def test_cli_dense_kernel_families_agree(driver, lib, oracle, tmp_path, n):
    """n_pad = 16 has two tensor-core implementations of the dense phases: tcgen05 + TMA (default) and
    mma.sync int8 (BLK_DENSE=mma).  Whole runs must end in byte-identical kernel files, accepted by the
    reference's checker (tools/umma_cli_check.sh additionally pins both to the reference's own output)."""
    p = 2147483647
    M = lib.synth.powerlaw_rows(2800, 3000, mean=9, seed=21, with_empty_rows=7)      # more columns than rows: a right kernel exists
    mtx = str(tmp_path / "m.mtx")
    lib.synth.write_mtx(mtx, M)
    hashes = {}
    for mode in ("", "mma"):
        out = str(tmp_path / f"k_{mode or 'default'}.mtx")
        env = dict(os.environ)
        env.pop("BLK_DENSE", None)
        if mode:
            env["BLK_DENSE"] = mode
        r = run([driver, "--matrix", mtx, "--prime", str(p), "--n", str(n), "--right", "--output-file", out], env=env)
        assert "OK:    v != 0" in r.stdout and "OK: vt*M == 0" in r.stdout
        hashes[mode or "default"] = sha(out)
    assert len(set(hashes.values())) == 1, hashes
    assert checker(oracle, lib, M, mtx, p, str(tmp_path / "k_default.mtx"), "--right")
