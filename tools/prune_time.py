"""Time blk_create_pruned (the removal of empty and singleton constraints, DESIGN.md section 14) against blk_create on
the same device COO, for two matrices generated on the device:

  cfg4      the bench.py config-4 matrix (50M x 50M power law, about 1.47G entries): nothing is removed
  uniform3  50M x 50M, 3 entries per row, uniform columns, values in [1, 100): heavy pruning over many rounds

Both at p = 2^31-1, n = 16, --left.  For each: the whole call (host clock around the call, which ends in a device
synchronisation; best of --reps after a warm-up call), and the device time of the pruning kernels from torch.profiler
in a separate call, split into round 0 (k_prune_round0), the rounds (k_prune_classify, k_prune_decrement) and the
compaction (every other kernel up to the last k_prune_* kernel: k_prune_keep, the CUB scans, k_prune_index,
k_prune_count, k_prune_select).  For uniform3 also the ms per iteration (CUDA events around blk_iterate after a
warm-up) and the expected iteration count 1 + Mc/n, pruned against unpruned.  The card's name and power limit are
read in the same run.

    python tools/prune_time.py --out profiles/r04_prune_time.json [--reps 2] [--iters 8]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

P, NB = 2147483647, 16
SIZE = 50_000_000
ROUND0, ROUNDS = ("k_prune_round0",), ("k_prune_classify", "k_prune_decrement")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def gen(torch, bench, name, dev):
    if name == "cfg4":
        return bench.gen_device_coo(torch, dict(rows=SIZE, cols=SIZE, mean=30.0), dev, seed=1)
    g = torch.Generator(device=dev)
    g.manual_seed(3)
    rows = torch.repeat_interleave(torch.arange(SIZE, device=dev, dtype=torch.int32), 3)
    nnz = rows.numel()
    cols = torch.randint(0, SIZE, (nnz,), device=dev, generator=g, dtype=torch.int32)
    vals = torch.randint(1, 100, (nnz,), device=dev, generator=g, dtype=torch.int32)
    return rows, cols, vals, nnz


def create(B, coo, stream, prune):
    t0 = time.perf_counter()
    ctx = B.BlockLanczos(n=NB, prime=P, right=False, device=0, stream=stream.cuda_stream, device_coo=coo, prune=prune)
    return ctx, (time.perf_counter() - t0) * 1e3


def phases(torch, B, coo, stream):
    """Device ms of round 0, the rounds and the compaction of one blk_create_pruned call (torch.profiler)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ctx, _ = create(B, coo, stream, True)
        torch.cuda.synchronize()
    ctx.close()
    kern = []
    for ev in prof.events():
        if "CUDA" in str(getattr(ev, "device_type", "")) and ev.time_range.elapsed_us() > 0:
            kern.append((ev.time_range.start, ev.time_range.end, ev.name))
    kern.sort()
    last = max((i for i, k in enumerate(kern) if "k_prune_" in k[2]), default=-1)
    out = dict(round0_ms=0.0, rounds_ms=0.0, compaction_ms=0.0, kernels={})
    for s, e, nm in kern[:last + 1]:
        ms = (e - s) / 1e3
        key = "round0_ms" if any(t in nm for t in ROUND0) else "rounds_ms" if any(t in nm for t in ROUNDS) else "compaction_ms"
        out[key] += ms
        short = next((t for t in nm.split("(")[0].split() if t.startswith("k_prune_")), None) or \
            ("cub scan" if "Scan" in nm else nm[:40])
        out["kernels"][short] = out["kernels"].get(short, 0.0) + ms
    out["prune_kernels_ms"] = out["round0_ms"] + out["rounds_ms"] + out["compaction_ms"]
    return out


def per_iteration(torch, ctx, stream, iters):
    v = torch.randint(0, P, (ctx.N * ctx.n,), dtype=torch.int32, generator=torch.Generator().manual_seed(7))
    ctx.set_state(v.numpy().view(np.uint32))
    del v
    ctx.iterate(1)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    ctx.iterate(iters)
    e1.record(stream)
    e1.synchronize()
    return e0.elapsed_time(e1) / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--iters", type=int, default=8)
    ap.add_argument("--matrices", default="cfg4,uniform3")
    a = ap.parse_args()
    import torch
    import bench
    import blk_lanczos_b200 as B
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this measurement needs the GPU")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    stream = torch.cuda.Stream(device=dev)
    res = {"card": card(), "p": P, "n": NB, "side": "--left", "matrices": {}}
    print("card", res["card"], flush=True)
    for name in a.matrices.split(","):
        rows, cols, vals, nnz = gen(torch, bench, name, dev)
        torch.cuda.synchronize()
        coo = (SIZE, SIZE, nnz, rows.data_ptr(), cols.data_ptr(), vals.data_ptr())
        r = dict(N=SIZE, Mc=SIZE, nnz=nnz)
        for prune in (False, True):
            ctx, _ = create(B, coo, stream, prune)             # warm-up (module load, allocator)
            ctx.close()
            times = []
            for _ in range(a.reps):
                ctx, ms = create(B, coo, stream, prune)
                times.append(ms)
                if _ < a.reps - 1:
                    ctx.close()
            key = "pruned" if prune else "plain"
            r[key] = dict(create_ms=times, create_ms_best=min(times))
            if prune:
                r[key]["stats"] = ctx.prune_stats
            r[key]["device_bytes"] = ctx.info()["device_bytes"]
            r[key]["expected_iterations"] = 1 + ctx.Mc // NB
            if name == "uniform3":
                r[key]["ms_per_iteration"] = per_iteration(torch, ctx, stream, a.iters)
            ctx.close()
            torch.cuda.empty_cache()
            print(name, key, json.dumps(r[key]), flush=True)
        r["pruned"]["phases"] = phases(torch, B, coo, stream)
        r["create_ratio"] = r["pruned"]["create_ms_best"] / r["plain"]["create_ms_best"]
        if name == "uniform3":
            r["loop_time_ratio"] = (r["pruned"]["ms_per_iteration"] * r["pruned"]["expected_iterations"]) / \
                (r["plain"]["ms_per_iteration"] * r["plain"]["expected_iterations"])
        print(name, "phases", json.dumps(r["pruned"]["phases"]), flush=True)
        res["matrices"][name] = r
        del rows, cols, vals, coo
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    json.dump(res, open(a.out, "w"), indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
