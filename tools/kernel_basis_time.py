"""Time blk_kernel_basis (the kernel-basis extraction) on two 50M-row states:

  cfg4   the bench.py config-4 workload (50M x 50M power law, p = 2^31-1, n = 16) after a few iterations
  p2n64  the same matrix generator at p = 2, n = 64, after a few iterations

For each: the whole call timed with CUDA events on the context's stream after a warm-up call (it includes the
copy of X to the host, and the product T = M^T v because a state in the middle of the loop has no T yet), and
the device time of its kernels from torch.profiler in a separate call.  Bytes: (N + Mc) n_pad 4 read by the
reductions, N n 4 written by X = v A_S.  The card's name and power limit are read in the same run.

    python tools/kernel_basis_time.py --out /tmp/kernel_basis_time.json [--iters 3] [--reps 3]
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

STATES = {
    "cfg4": dict(rows=50_000_000, cols=50_000_000, mean=30.0, n=16, p=2147483647),
    "p2n64": dict(rows=50_000_000, cols=50_000_000, mean=30.0, n=64, p=2),
}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--iters", type=int, default=3)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--states", default="cfg4,p2n64")
    a = ap.parse_args()
    import torch
    import bench
    import blk_lanczos_b200 as B
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this measurement needs the GPU")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    res = {"card": card(), "states": {}}
    for name in a.states.split(","):
        w = dict(STATES[name], right=False)
        rows, cols, vals, nnz = bench.gen_device_coo(torch, w, dev)
        torch.cuda.synchronize()
        stream = torch.cuda.Stream(device=dev)
        coo = (w["rows"], w["cols"], nnz, rows.data_ptr(), cols.data_ptr(), vals.data_ptr())
        ctx = B.BlockLanczos(n=w["n"], prime=w["p"], right=False, device=0, stream=stream.cuda_stream, device_coo=coo)
        del rows, cols, vals
        torch.cuda.empty_cache()
        info = ctx.info()
        N, Mc, n, npad = info["N"], info["Mc"], info["n"], info["n_pad"]
        v = torch.randint(0, w["p"], (N * n,), dtype=torch.int32, generator=torch.Generator().manual_seed(7))
        ctx.set_state(v.numpy().view(np.uint32))
        del v
        it, stopped = ctx.iterate(a.iters)
        x = np.empty(N * n, dtype=np.uint32)
        k = C.c_int32(0)
        call = lambda: ctx._ck(ctx.L.blk_kernel_basis(ctx.h, C.c_void_p(x.ctypes.data), C.byref(k)))
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
                tag = ("k_kb_reduce" if "k_kb_reduce" in nm else "k_kb_small" if "k_kb_small" in nm else
                       "k_block_apply" if "k_block_apply" in nm else "spmv (T = M^T v)" if "spmv" in nm else
                       "unpad (host layout)" if "unpad" in nm else "other")
                kern[tag] = kern.get(tag, 0.0) + ev.self_device_time_total / 1000.0
        kb_ms = sum(kern.get(t, 0.0) for t in ("k_kb_reduce", "k_kb_small", "k_block_apply"))
        rd, wr = (N + Mc) * npad * 4, N * n * 4
        best = min(times)
        res["states"][name] = dict(
            N=N, Mc=Mc, n=n, n_pad=npad, p=w["p"], nnz=nnz, iterations=it, stopped=stopped, k=k.value,
            call_ms=times, call_ms_best=best, device_kernels_ms=kern, kernel_basis_kernels_ms=kb_ms,
            bytes_read=rd, bytes_written=wr,
            gbs_kernels=(rd + wr) / (kb_ms * 1e6) if kb_ms > 0 else None,
            gbs_call=(rd + wr) / (best * 1e6))
        print(name, json.dumps(res["states"][name]), flush=True)
        ctx.close()
        del x
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    json.dump(res, open(a.out, "w"), indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
