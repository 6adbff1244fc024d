"""Time blk_solve (the inhomogeneous solve, DESIGN.md section 13) and the loop on the augmented matrix, on the
bench.py config-4 matrix (50M x 50M power law) with dense random right-hand sides (M^T x = b, --left):

  cfg4_r1   p = 2^31-1, n = 16, r = 1
  cfg4_r8   p = 2^31-1, n = 16, r = 8
  p2n64_r8  p = 2,      n = 64, r = 8

For each: ms per iteration of the loop on the augmented matrix against the plain matrix at the same n and p (CUDA
events around blk_iterate, after a warm-up), the whole blk_solve call (CUDA events, after a warm-up call; it includes
T = M^T v and the copy of x to the host), and the device time of its kernels from torch.profiler in a separate call.
k_block_apply is set against the copy-rate floor: the bytes it has to move (N n_pad 4 read, N r_pad 4 written) at the
device-to-device copy rate measured in the same run.  The card's name and power limit are read in the same run.

    python tools/solve_time.py --out /tmp/solve_time.json [--iters 8] [--reps 3]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

MATRIX = dict(rows=50_000_000, cols=50_000_000, mean=30.0)
STATES = {
    "cfg4_r1": dict(n=16, p=2147483647, r=1),
    "cfg4_r8": dict(n=16, p=2147483647, r=8),
    "p2n64_r8": dict(n=64, p=2, r=8),
}
TAGS = ("k_kb_reduce", "k_kb_small", "k_solve_tail", "k_solve_small", "k_block_apply")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def copy_rate(torch, dev, reps=10):
    """Device-to-device copy rate (bytes read + written per second) of a 4 GB buffer."""
    a = torch.empty(1 << 30, dtype=torch.int32, device=dev)
    b = torch.empty_like(a)
    b.copy_(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        b.copy_(a)
    e1.record()
    e1.synchronize()
    ms = e0.elapsed_time(e1) / reps
    del a, b
    torch.cuda.empty_cache()
    return 2 * (1 << 32) / (ms * 1e-3)


def make_ctx(torch, B, bench, dev, stream, n, p, r, seed=1):
    w = dict(MATRIX, n=n, p=p, right=False)
    rows, cols, vals, nnz = bench.gen_device_coo(torch, w, dev, seed=seed)
    torch.cuda.synchronize()
    coo = (w["rows"], w["cols"], nnz, rows.data_ptr(), cols.data_ptr(), vals.data_ptr())
    kw = {}
    rhs = None
    if r:
        g = torch.Generator(device=dev)
        g.manual_seed(11)
        rhs = torch.randint(0, p, (w["cols"], r), device=dev, generator=g, dtype=torch.int32)   # Mc x r, dense
        kw["rhs_device"] = (rhs.data_ptr(), r)
    torch.cuda.synchronize()
    ctx = B.BlockLanczos(n=n, prime=p, right=False, device=0, stream=stream.cuda_stream, device_coo=coo, **kw)
    del rows, cols, vals, rhs
    torch.cuda.empty_cache()
    return ctx, nnz


def per_iteration(torch, ctx, stream, iters, p):
    N, n = ctx.N, ctx.n
    v = torch.randint(0, p, (N * n,), dtype=torch.int32, generator=torch.Generator().manual_seed(7))
    ctx.set_state(v.numpy().view(np.uint32))
    del v
    ctx.iterate(1)                                          # warm-up (graph capture, first launches)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    done, _ = ctx.iterate(iters)
    e1.record(stream)
    e1.synchronize()
    return e0.elapsed_time(e1) / iters, done


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--iters", type=int, default=8)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--states", default="cfg4_r1,cfg4_r8,p2n64_r8")
    a = ap.parse_args()
    import torch
    import bench
    import blk_lanczos_b200 as B
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this measurement needs the GPU")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    stream = torch.cuda.Stream(device=dev)
    rate = copy_rate(torch, dev)
    res = {"card": card(), "copy_rate_bytes_per_s": rate, "plain": {}, "states": {}}
    print("card", res["card"], "copy rate %.1f GB/s" % (rate / 1e9), flush=True)
    for name in a.states.split(","):
        s = STATES[name]
        key = f"n{s['n']}_p{s['p']}"
        if key not in res["plain"]:
            ctx, nnz = make_ctx(torch, B, bench, dev, stream, s["n"], s["p"], 0)
            ms, _ = per_iteration(torch, ctx, stream, a.iters, s["p"])
            res["plain"][key] = dict(nnz=nnz, ms_per_iteration=ms)
            print("plain", key, json.dumps(res["plain"][key]), flush=True)
            ctx.close()
            torch.cuda.empty_cache()
        ctx, nnz = make_ctx(torch, B, bench, dev, stream, s["n"], s["p"], s["r"])
        info = ctx.info()
        ms_it, iters = per_iteration(torch, ctx, stream, a.iters, s["p"])
        N0, r, n, npad = ctx.N0, ctx.nrhs, info["n"], info["n_pad"]
        rp = 1 << (r - 1).bit_length()
        x = np.empty(N0 * r, dtype=np.uint32)
        found = np.zeros(r, dtype=np.int32)
        call = lambda: ctx._ck(ctx.L.blk_solve(ctx.h, C.c_void_p(x.ctypes.data), C.c_void_p(found.ctypes.data)))
        call()                                              # warm-up (module load, first-touch of x)
        times = []
        for _ in range(a.reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            call()
            e1.record(stream)
            e1.synchronize()
            times.append(e0.elapsed_time(e1))
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            call()
            torch.cuda.synchronize()
        kern = {}
        for ev in prof.key_averages():
            if ev.device_type is not None and "CUDA" in str(ev.device_type) and ev.self_device_time_total > 0:
                nm = ev.key
                tag = next((t for t in TAGS if t in nm), None) or ("spmv (T = M^T v)" if "spmv" in nm else
                                                                   "unpad (host layout)" if "unpad" in nm else "other")
                kern[tag] = kern.get(tag, 0.0) + ev.self_device_time_total / 1000.0
        solve_ms = sum(kern.get(t, 0.0) for t in TAGS)
        N = info["N"]
        apply_bytes = N * npad * 4 + N * rp * 4
        floor_ms = apply_bytes / rate * 1e3
        plain = res["plain"][key]
        res["states"][name] = dict(
            N=N, N0=N0, Mc=info["Mc"], n=n, n_pad=npad, r=r, r_pad=rp, p=s["p"], nnz_plain=plain["nnz"],
            nnz_augmented=int(info["nnz_local"][0]), iterations=iters, found=int(found.sum()),
            ms_per_iteration=ms_it, ms_per_iteration_plain=plain["ms_per_iteration"],
            iteration_ratio=ms_it / plain["ms_per_iteration"],
            call_ms=times, call_ms_best=min(times), device_kernels_ms=kern, solve_kernels_ms=solve_ms,
            apply_bytes=apply_bytes, apply_copy_floor_ms=floor_ms,
            apply_share_of_copy_floor=floor_ms / kern["k_block_apply"] if kern.get("k_block_apply") else None)
        print(name, json.dumps(res["states"][name]), flush=True)
        ctx.close()
        del x
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    json.dump(res, open(a.out, "w"), indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
