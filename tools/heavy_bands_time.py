"""Product 2 with its heavy row prefix run as column bands (SpOp::split, DESIGN.md section 4) on the bench.py config-4
matrix (50M x 50M power law, about 1.47G entries, p = 2^31-1, n = 16, --left), one GPU.

  1. the card's name, power limit and maximum SM clock;
  2. product 2 (blk_time_spmv, M x) unsplit (BLK_HEAVY=0), then for every minimum degree D x band slice of the sweep:
     H, K, the ms per product, and its device time split into the bands, the pass that adds their partials, and the
     light rows (torch.profiler, a separate call);
  3. whole iterations, alternating BLK_HEAVY=0 and the fastest sweep point, --runs times each: ms per iteration and
     per phase as bench.py measures them (profiling mode, CUDA events), and the sha256 of v after the run, which must
     be the same for both.

    python tools/heavy_bands_time.py --out profiles/r05_heavy_bands.json
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

P, NB, SIZE = 2147483647, 16, 50_000_000
MB = 1 << 20
KNOBS = ("BLK_HEAVY", "BLK_HEAVY_MIN_DEG", "BLK_HEAVY_BAND_BYTES")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def setenv(**kv):
    for k in KNOBS:
        os.environ.pop(k, None)
    os.environ.update({k: str(v) for k, v in kv.items()})


def create(B, coo, stream):
    return B.BlockLanczos(n=NB, prime=P, right=False, device=0, stream=stream.cuda_stream, device_coo=coo)


def breakdown(torch, ctx, reps=2):
    """Device ms of one product 2 split into bands / combine / light.  Per product the launches are, in order: k_spmv,
    k_spmv_fix of the K bands (one band-major operator), k_band_combine, then k_spmv, k_spmv_fix of the light rows."""
    from torch.profiler import ProfilerActivity, profile
    ctx.time_spmv(False, 1)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ctx.time_spmv(False, reps)
        torch.cuda.synchronize()
    kern = sorted((ev.time_range.start, ev.time_range.end, ev.name) for ev in prof.events()
                  if "CUDA" in str(getattr(ev, "device_type", "")) and ev.time_range.elapsed_us() > 0
                  and ("k_spmv" in ev.name or "k_band_combine" in ev.name))
    per = 5
    kern = kern[-per * reps:]
    out = dict(bands_ms=0.0, combine_ms=0.0, light_ms=0.0)
    for i, (s, e, nm) in enumerate(kern):
        j = i % per
        key = "bands_ms" if j < 2 else "combine_ms" if j == 2 else "light_ms"
        out[key] += (e - s) / 1e3 / reps
    out["launches_per_product"] = per
    out["kernels_seen"] = len(kern)
    return out


def whole_run(torch, B, coo, stream, v0, warmup, steps):
    ctx = create(B, coo, stream)
    inf = ctx.info()
    ctx.set_state(v0)
    ctx.iterate(warmup)
    ctx.set_profiling(True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    with torch.cuda.stream(stream):
        e0.record(stream)
        ctx.iterate(steps)
        e1.record(stream)
    e1.synchronize()
    ms = e0.elapsed_time(e1) / steps
    ph = {k: v["ms"] / steps for k, v in ctx.phase_times().items()}
    ctx.set_profiling(False)
    v = ctx.get_state(which=("v",))["v"]
    sha = hashlib.sha256(v[:SIZE * NB].tobytes()).hexdigest()
    ctx.close()
    torch.cuda.empty_cache()
    return dict(ms_per_step=ms, phases_ms_per_step=ph, heavy_rows=inf["heavy_rows"], heavy_bands=inf["heavy_bands"],
                state_sha256=sha)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--degrees", default="100,200,400,1000")
    ap.add_argument("--slices-mb", default="8,16,24,32,48")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--steps", type=int, default=10)
    a = ap.parse_args()
    import torch
    import bench
    import blk_lanczos_b200 as B
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this measurement needs the GPU")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    stream = torch.cuda.Stream(device=dev)
    res = {"card": card(), "matrix": "bench.py cfg4 (seed 1)", "p": P, "n": NB, "side": "--left",
           "unit": "ms (device time, CUDA events)"}
    print("card", res["card"], flush=True)
    rows, cols, vals, nnz = bench.gen_device_coo(torch, bench.WORKLOADS["cfg4"], dev, seed=1)
    torch.cuda.synchronize()
    coo = (SIZE, SIZE, nnz, rows.data_ptr(), cols.data_ptr(), vals.data_ptr())
    res["nnz"] = nnz

    setenv(BLK_HEAVY=0)
    ctx = create(B, coo, stream)
    res["unsplit_M_x_ms"] = ctx.time_spmv(False, a.reps)
    res["unsplit_Mt_x_ms"] = ctx.time_spmv(True, a.reps)
    ctx.close()
    torch.cuda.empty_cache()
    print("unsplit", res["unsplit_M_x_ms"], flush=True)

    sweep = []
    for d in [int(x) for x in a.degrees.split(",")]:
        for mb in [int(x) for x in a.slices_mb.split(",")]:
            setenv(BLK_HEAVY_MIN_DEG=d, BLK_HEAVY_BAND_BYTES=mb * MB)
            ctx = create(B, coo, stream)
            inf = ctx.info()
            rec = dict(min_deg=d, slice_mb=mb, H=inf["heavy_rows"], K=inf["heavy_bands"], device_gb=inf["device_bytes"] / 1e9)
            if rec["H"] > 0:
                rec["M_x_ms"] = ctx.time_spmv(False, a.reps)
                try:
                    rec.update(breakdown(torch, ctx))
                except Exception as exc:          # the breakdown is secondary: keep the point
                    rec["breakdown_error"] = f"{type(exc).__name__}: {exc}"
            ctx.close()
            torch.cuda.empty_cache()
            sweep.append(rec)
            print(json.dumps(rec), flush=True)
    res["sweep"] = sweep
    timed = [r for r in sweep if "M_x_ms" in r]
    best = min(timed, key=lambda r: r["M_x_ms"])
    res["best"] = dict(min_deg=best["min_deg"], slice_mb=best["slice_mb"], M_x_ms=best["M_x_ms"],
                       gain_ms=res["unsplit_M_x_ms"] - best["M_x_ms"])

    v0 = np.random.default_rng(7).integers(0, P, size=SIZE * NB).astype(np.uint32)
    runs = {"off": [], "split": []}
    for _ in range(a.runs):
        for key in ("off", "split"):
            if key == "off":
                setenv(BLK_HEAVY=0)
            else:
                setenv(BLK_HEAVY_MIN_DEG=best["min_deg"], BLK_HEAVY_BAND_BYTES=best["slice_mb"] * MB)
            r = whole_run(torch, B, coo, stream, v0, a.warmup, a.steps)
            runs[key].append(r)
            print(key, json.dumps(r), flush=True)
    setenv()
    summ = {}
    for key, rs in runs.items():
        ms = [r["ms_per_step"] for r in rs]
        summ[key] = dict(ms_per_step=ms, mean=float(np.mean(ms)), spread=float(max(ms) - min(ms)),
                         phases_mean={k: float(np.mean([r["phases_ms_per_step"][k] for r in rs])) for k in rs[0]["phases_ms_per_step"]})
    summ["gap_ms"] = summ["off"]["mean"] - summ["split"]["mean"]
    summ["gap_over_max_spread"] = summ["gap_ms"] / max(1e-9, summ["off"]["spread"], summ["split"]["spread"])
    summ["same_state"] = len({r["state_sha256"] for r in runs["off"] + runs["split"]}) == 1
    res["whole_iterations"] = dict(warmup=a.warmup, steps=a.steps, runs=runs, summary=summ)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    json.dump(res, open(a.out, "w"), indent=1)
    print(json.dumps(dict(best=res["best"], summary=summ)))


if __name__ == "__main__":
    main()
