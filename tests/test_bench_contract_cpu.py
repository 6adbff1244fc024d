"""CPU suite, part 6: the reference arm of bench.py runs without a GPU (it times the reference's own
OpenMP build from oracle/_ref on the host cores) and prints the contract's JSON line."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    if not os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libref_omp.so")) and \
            not os.path.exists(os.path.join(ROOT, "oracle", "liboracle.so")):
        pytest.skip("no CPU implementation built")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout          # ONE JSON line
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "lanczos_iters_per_s" and d["unit"] == "iterations/s"
    assert d["higher_is_better"] is True and d["vs_baseline"] is None and d["value"] > 0
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and "twin" in cb["sample"] and cb["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]


def test_non_zero_ranks_of_the_reference_arm_do_nothing():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1"],
                       capture_output=True, text=True, timeout=60, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_reference_arm_rejects_dump_outputs(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                        "--dump-outputs", str(tmp_path / "d")], capture_output=True, text=True, timeout=60)
    assert r.returncode != 0 and "--dump-outputs" in r.stderr and r.stdout == ""
    assert not (tmp_path / "d").exists()


def test_dense_roofline_helper():
    import importlib.util
    spec = importlib.util.spec_from_file_location("_bench", os.path.join(ROOT, "bench.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    r = b.dense_roofline({"spmv1": 27.6, "dots": 0.92, "ortho": 2.63, "small": 0.0}, 50_000_000, 16, 6449.0)
    assert abs(r["dots"]["achieved"] - 2 * 3.2e9 / 0.92e-3 / 1e9) < 1e-6 and 1.0 < r["dots"]["frac"] < 1.2
    assert abs(r["ortho"]["bytes_per_launch"] - 16e9) < 1 and 0.9 < r["ortho"]["frac"] < 1.0
    assert b.dense_roofline({}, 10, 16, 6449.0) == {} and b.dense_roofline({"dots": 0.0}, 10, 16, 6449.0) == {}
