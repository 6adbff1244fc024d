"""bench.py --dump-outputs on the CPU-sized twin of the benchmark workload: the files, their type and size, the same
outputs from run to run with the same arguments, another state after one more step, and every file holding what
its name says -- the CPU oracle's blocks and n x n matrices after the same iterations on the same seeded inputs."""
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT
from oracle.oracle import block_pad

pytestmark = pytest.mark.gpu

WARMUP = 3


def run_bench(out, steps):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "cfg4_tiny", "--steps", str(steps),
                        "--warmup", str(WARMUP), "--no-extras", "--no-cpu-baseline", "--no-e2e", "--dump-outputs", str(out)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout
    return json.loads(lines[0]), {f[:-4]: np.load(out / f) for f in sorted(os.listdir(out))}


def test_bench_dump_outputs(lib, oracle, tmp_path):
    import torch
    spec = importlib.util.spec_from_file_location("_bench", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    w = bench.WORKLOADS["cfg4_tiny"]
    n, p, steps = w["n"], w["p"], 2

    a, da = run_bench(tmp_path / "a", steps)
    b, db = run_bench(tmp_path / "b", steps)
    c, dc = run_bench(tmp_path / "c", steps + 1)
    assert sorted(da) == ["Av", "d", "p", "tmp", "v", "vtAAv", "vtAv", "winv"]
    assert sum(x.nbytes for x in da.values()) <= 64 << 20
    assert da["v"].shape == (bench.DUMP_ROWS, n) and da["vtAv"].shape == (n, n) and da["d"].shape == (n,)
    for k, x in da.items():
        assert x.dtype == np.float64 and np.array_equal(x, db[k]), k
    assert a["state_sha256"] == b["state_sha256"] != c["state_sha256"]
    assert not np.array_equal(da["v"], dc["v"])

    # the same seeded matrix and start block as bench.py, through the oracle for warmup + steps iterations
    rows, cols, vals, _ = bench.gen_device_coo(torch, w, torch.device("cuda", 0))
    M = lib.SparseCOO(w["rows"], w["cols"], rows.cpu().numpy(), cols.cpu().numpy(), vals.cpu().numpy().astype(np.uint32))
    del rows, cols, vals
    N, K = M.nrows, WARMUP + steps
    v0 = torch.empty(N * n, dtype=torch.int32).random_(0, p, generator=torch.Generator().manual_seed(7)).numpy().view(np.uint32)
    pad = block_pad(M.nrows, M.ncols, n, False)
    st = dict(v=np.zeros(pad, np.uint32), tmp=np.zeros(pad, np.uint32), Av=np.zeros(pad, np.uint32),
              p=np.zeros(pad, np.uint32), iters=0)
    st["v"][:N * n] = v0
    want = oracle.lanczos_run(M, n, p, False, stop_after=K, state=st)
    assert want["iters"] == K
    sample = np.sort(np.random.default_rng(0).choice(pad // n, bench.DUMP_ROWS, replace=False))
    for k in ("v", "tmp", "Av", "p"):
        assert np.array_equal(da[k], want[k].reshape(pad // n, n)[sample]), k
    # the n x n matrices of iteration K, from the state after K - 1 iterations
    prev = oracle.lanczos_run(M, n, p, False, stop_after=K - 1, state=st)
    Av = oracle.sparse_matrix_vector_product(M, oracle.sparse_matrix_vector_product(M, prev["v"], True, n, p), False, n, p)
    vtAv, vtAAv = oracle.block_dot_products(N, Av, prev["v"], n, p)
    _, winv, d = oracle.semi_inverse(vtAv, n, p)
    for k, x in (("vtAv", vtAv), ("vtAAv", vtAAv), ("winv", winv), ("d", d)):
        assert np.array_equal(da[k].ravel(), x), k
