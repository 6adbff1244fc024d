#!/usr/bin/env python
"""bench.py -- block-Lanczos mod-p hot path on B200: Lanczos iterations/s and SpMV G(nnz*n)/s.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload cfg4|cfg4_small|cfg4_tiny]
                    [--dump-outputs DIR]

A "step" is one block-Lanczos iteration (two n-wide sparse products, block dot products,
semi-inverse, orthogonalize) of the named workload.  Default workload (BASELINE.json configs[3],
the one the metric's 1/2/4/8-GPU scaling and HBM-roofline targets are quoted on; it fits one
GPU): synthetic 50M x 50M power-law matrix, ~1.5e9 non-zeros, p = 2^31-1, n = 16, generated on
the device with a seeded torch generator.  With N > 1 (torchrun) the same matrix is row-sharded
over the ranks ("strong" scaling); Av and tmp travel between the GPUs inside the library.

One JSON line on stdout (rank 0).  Its parts:

  value / ms_per_step   iterations/s with everything resident in HBM, device-timed with CUDA events on
                        the library's stream, max over ranks.
  state_sha256          sha256 of the block v after exactly warmup + steps iterations from the fixed start
                        block: the same digest for every N proves that sharding changes no bit.
  parity                the same library on a CPU-sized twin (cfg4_tiny), sharded the same way, compared
                        with the CPU oracle (oracle/ is only the checker here, outside every timed region).
  e2e                   the metric through the C ABI with HOST buffers: blk_set_state (each rank reads its
                        rows of the start block from pinned memory), K blk_iterate(1) calls (each returns
                        the iteration counter and stop flag to the host) and blk_get_state_local (each rank
                        writes its rows of v back), all inside the timed region; achieved PCIe rates stated.
  roofline              k_spmv against SURVEY.md 8(d)'s algorithmic bytes, the gather model and the DRAM
                        traffic ncu counted; roofline_dense the two dense kernels.
  spmv_sweep            BASELINE configs[4]: blk_time_spmv for n in {1,2,4,8,16,32} x p in {65537, 2^31-1},
                        both directions, on the cfg4 matrix (sharded when N > 1).
  small_configs         BASELINE configs[0..2] (N = 1): complete runs, us per iteration.
  cpu_baseline          the UNMODIFIED reference's builds (oracle/_ref, compiled from /root/reference) on
                        the host cores on a scaled-down twin: OpenMP (timing build), OpenMP at a prime where
                        its deferred modulo is exact, sequential, and its SpMV alone.

--dump-outputs DIR also writes the state after the last timed step as DIR/<name>.npy (see dump_outputs).  The
inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

P_MERSENNE = 2147483647
P_OMP_EXACT = 1073741789          # the reference's own cap (2^30 - 35): its OpenMP build is exact there (SURVEY F2)
WORKLOADS = {
    # name: rows, cols, mean nnz/row, n, p, right
    "cfg4": dict(rows=50_000_000, cols=50_000_000, mean=30.0, n=16, p=P_MERSENNE, right=False,
                 desc="BASELINE configs[3]: synthetic 50Mx50M power-law, ~1.5B nnz, p=2^31-1, n=16"),
    "cfg4_small": dict(rows=5_000_000, cols=5_000_000, mean=30.0, n=16, p=P_MERSENNE, right=False,
                       desc="1/10-scale twin of configs[3] (dev)"),
    "cfg4_tiny": dict(rows=200_000, cols=200_000, mean=30.0, n=16, p=P_MERSENNE, right=False,
                      desc="1/250-scale twin of configs[3] (CPU-sized)"),
}
METRIC = "lanczos_iters_per_s"
UNIT = "iterations/s"
CPU_TWIN = dict(rows=200_000, cols=200_000)          # bounded CPU sample of the same generator
SWEEP_NS = (1, 2, 4, 8, 16, 32)
SWEEP_PRIMES = (65537, P_MERSENNE)
DUMP_ROWS = 1 << 16          # rows per block kept by --dump-outputs: 4 blocks x 65536 x n=16 x 8 B = 32 MB


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------
def gen_device_coo(torch, w, dev, seed=1):
    """Power-law row degrees (Pareto shape 1.5, mean ~`mean`, cap 1e6), uniform columns, values in
    [1,100): SURVEY.md section 8(d).  Same generator family as synth.powerlaw_rows, on the device."""
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    N, Mc = w["rows"], w["cols"]
    u = torch.rand(N, device=dev, generator=g, dtype=torch.float64)
    dmin = max(1, round(w["mean"] / 3))
    d = torch.clamp((dmin * (1 - u) ** (-1 / 1.5)).floor().to(torch.int64), max=min(1_000_000, 8 * Mc))
    del u
    rows = torch.repeat_interleave(torch.arange(N, device=dev, dtype=torch.int32), d)
    del d
    nnz = rows.numel()
    cols = torch.randint(0, Mc, (nnz,), device=dev, generator=g, dtype=torch.int32)
    vals = torch.randint(1, 100, (nnz,), device=dev, generator=g, dtype=torch.int32)
    return rows, cols, vals, nnz


def bind_to_gpu_numa_node(index):
    """Run this process (and first-touch its pinned buffers) on the CPUs NVML reports as local to the GPU, so
    that the host side of every PCIe copy lives on the GPU's NUMA node.  Returns a short description."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {64 * i + b for i, wd in enumerate(mask) for b in range(64) if (wd >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return f"{len(cpus)} CPUs local to GPU {index} ({min(cpus)}-{max(cpus)})"
    except Exception as exc:          # affinity is an optimisation, never a requirement
        return f"unchanged ({type(exc).__name__})"
    return "unchanged"


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU with NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop_evt = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if not self.nv:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake_slowdown",
        }
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop_evt.wait(0.05)

    def finish(self):
        self._stop_evt.set()
        self.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# ------------------------------------------------------------------------------------------
def run_ref(lib, w, rows, cols, iters, warmup, threads, prime=None, spmv_reps=0, timeout=900):
    """One run of oracle/ref_runner.py (the reference's object code on a synthetic twin) in a subprocess."""
    env = dict(os.environ, OMP_NUM_THREADS=str(threads), OMP_STACKSIZE="1G", OMP_PROC_BIND="false")
    cmd = [sys.executable, os.path.join(ROOT, "oracle", "ref_runner.py"), "--lib", lib,
           "--rows", str(rows), "--cols", str(cols), "--mean", str(w["mean"]),
           "--n", str(w["n"]), "--prime", str(prime or w["p"]), "--right", str(int(w["right"])),
           "--iters", str(iters), "--warmup", str(warmup), "--spmv-reps", str(spmv_reps)]
    try:
        out = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=timeout)
        return json.loads(out.stdout.strip().splitlines()[-1])
    except Exception as e:                                   # pragma: no cover
        sys.stderr.write(f"[bench] CPU reference run ({lib}, {threads} threads) failed: {e}\n")
        return None


def run_cpu_reference(w, iters, warmup, threads=None, spmv_reps=0):
    """Reference OpenMP build on the host cores, on the CPU twin of workload w; the best thread count of
    {16 (where the authors found its peak), nproc} is kept."""
    cores = os.cpu_count() or 1
    cand = [threads] if threads else sorted({min(cores, 16), cores})
    best, tried = None, {}
    for t in cand:
        r = run_ref("omp", w, CPU_TWIN["rows"], CPU_TWIN["cols"], iters, warmup, t, spmv_reps=spmv_reps)
        if r is None:
            continue
        tried[str(t)] = r["iters_per_s"]
        if best is None or r["iters_per_s"] > best["iters_per_s"]:
            best = r
    if best is not None:
        best["tried_threads"] = tried
    return best


def cpu_baseline_obj(r, w, nnz_full):
    """Scale the twin's measured rate to the full workload by the work ratio (both the sparse
    products, ~nnz*n, and the dense phases, ~N*n^2, are linear in the twin's scale factor)."""
    scale = r["nnz"] / float(nnz_full)
    out = {
        "value": r["iters_per_s"] * scale, "unit": UNIT, "cores": r["threads"], "host_cores": r.get("host_cores"),
        "kind": r["kind"],
        "sample": (f"{r['lib']} build of the reference, {r['iters']} iterations on a {r['rows']}x{r['cols']} twin "
                   f"({r['nnz']} nnz, same generator, n={r['n']}, p={r['prime']}): {r['iters_per_s']:.3f} it/s "
                   f"= {r['gnnzn_per_s']:.3f} G(nnz*n)/s measured; value = that x nnz_twin/nnz_full ({scale:.3e}). "
                   "-DNDEBUG build: at p=2^31-1 the OpenMP variant's deferred modulo overflows u64 "
                   "(SURVEY F2), so it is a timing baseline only.  The OpenMP build cannot run the full size: "
                   "6.4 GB of stack per thread (openMP/lanczos_modp.c:336,352)."),
        "measured_iters_per_s_on_sample": r["iters_per_s"], "spmv_gnnzn_per_s": r["gnnzn_per_s"],
        "threads_tried": r.get("tried_threads"),
    }
    if r.get("spmv_gnnzn_per_s"):
        out["spmv_alone_gnnzn_per_s"] = r["spmv_gnnzn_per_s"]        # sparse_matrix_vector_product timed directly
    return out


def cpu_baseline_extras(w, threads):
    """BASELINE.md section 3's other two CPU figures (bounded): the OpenMP build at a prime where it is exact, and
    the sequential build on one core."""
    extra = {}
    r = run_ref("omp", w, CPU_TWIN["rows"], CPU_TWIN["cols"], 3, 1, threads, prime=P_OMP_EXACT)
    if r:
        extra["openmp_exact_prime"] = {"prime": P_OMP_EXACT, "threads": r["threads"], "iters_per_s_on_sample": r["iters_per_s"],
                                       "gnnzn_per_s": r["gnnzn_per_s"],
                                       "note": "same twin; p = 2^30-35 is the reference's own cap, where the deferred modulo cannot overflow"}
    rows = CPU_TWIN["rows"] // 4
    r = run_ref("seq", w, rows, rows, 2, 0, 1, spmv_reps=1)
    if r:
        extra["sequential_1_core"] = {"rows": rows, "nnz": r["nnz"], "iters_per_s_on_sample": r["iters_per_s"],
                                      "gnnzn_per_s": r["gnnzn_per_s"], "spmv_alone_gnnzn_per_s": r.get("spmv_gnnzn_per_s"),
                                      "note": f"sequential/lanczos_modp.c (the parity oracle's source) on a {rows}x{rows} twin, 1 core"}
    return extra


def expected_nnz(w):
    # mean of floor(10 * U^(-2/3)) capped at 1e6, measured on the generator: 29.33 per row
    return int(w["rows"] * 29.33 * (w["mean"] / 30.0))


# ------------------------------------------------------------------------------------------
def dense_roofline(phases_ms_per_step, rows_local, n_pad, peak):
    """Secondary kernels against the same HBM peak: algorithmic bytes of SURVEY 8(d) (block_dot_products reads v and
    Av: 2 blocks; orthogonalize reads v, Av, p and writes v, p: 5 blocks of rows x n_pad x 4 bytes) over the in-run
    phase times.  On one GPU the dots phase includes the fused n x n stage (one block, ~25 us)."""
    out = {}
    block = rows_local * n_pad * 4
    for key, blocks, kernel in (("dots", 2, "block_dot_products (+ n x n stage)"), ("ortho", 5, "orthogonalize")):
        ms = float(phases_ms_per_step.get(key, 0.0) or 0.0)
        if ms > 0 and block > 0:
            ach = blocks * block / (ms * 1e-3) / 1e9
            out[key] = {"kernel": kernel, "bound": "hbm", "bytes_per_launch": blocks * block, "ms_per_launch": ms,
                        "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak}
    return out


def spmv_bytes(nnz, rows_out, rows_in, n, n_pad=None):
    """SURVEY 8(d): algorithmic bytes (each x row once), gather model (a 4n-byte x row per non-zero) and line
    model (what B200's memory system moves: one 128-byte line per gathered row when 4*n_pad <= 128)."""
    n_pad = n_pad or n
    alg = 8 * nnz + 4 * (rows_out + 1) + 4 * n * rows_in + 4 * n * rows_out
    gather = nnz * (8 + 4 * n) + 4 * (rows_out + 1) + 4 * n * rows_out
    line = nnz * (8 + max(128, 4 * n_pad)) + 4 * (rows_out + 1) + 4 * n_pad * rows_out
    return alg, gather, line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=os.environ.get("BLK_BENCH_WORKLOAD", "cfg4"), choices=sorted(WORKLOADS))
    ap.add_argument("--chunk", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip spmv_sweep, small_configs and the tiny-twin parity check")
    ap.add_argument("--sweep-budget-s", type=float, default=100.0)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the state after the last timed step to DIR/<name>.npy (float64, sampled rows)")
    a = ap.parse_args()
    if a.dump_outputs and a.impl == "reference":
        # the reference arm times the CPU program on a scaled-down twin: it has no state of the workload to write
        ap.error("--dump-outputs is not available with --impl reference")
    a.warmup = max(a.warmup, 3) if a.impl == "ours" else a.warmup
    w = WORKLOADS[a.workload]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    config = {"workload": f"{a.workload}: {w['desc']}", "rows": w["rows"], "cols": w["cols"], "n": w["n"],
              "prime": w["p"], "side": "right" if w["right"] else "left", "sharding": f"row-blocks x{world}",
              "l2": "inputs (matrix 12 GB/operator, 3.2 GB blocks) far larger than the 126 MB L2; no flush needed"
                    if a.workload == "cfg4" else "working set exceeds L2"}

    # ---------------- reference arm: the reference's own CPU implementation --------------
    if a.impl == "reference":
        if rank != 0:
            return 0
        r = run_cpu_reference(w, max(1, a.steps), max(0, a.warmup), spmv_reps=2)
        nnz_full = expected_nnz(w)
        if r is None:
            print(json.dumps({"impl": "reference", "unavailable": "reference run failed on this host"}))
            return 0
        cb = cpu_baseline_obj(r, w, nnz_full)
        config["cpu_sample"] = {"rows": r["rows"], "cols": r["cols"], "nnz": r["nnz"],
                                "note": "timed on this twin of the workload and scaled by nnz (the reference cannot run the full size)"}
        line = {"metric": METRIC, "value": cb["value"], "unit": UNIT, "impl": "reference", "n_gpus": a.gpus,
                "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1e3 / cb["value"], "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "u32 (u64 accumulate)", "data": "synthetic",
                "config": config, "cpu_baseline": cb,
                "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return 0

    # ---------------- our arm ---------------------------------------------------------------
    numa = bind_to_gpu_numa_node(local_rank)
    import numpy as np
    import torch
    import blk_lanczos_b200 as B
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    def new_id():
        if world == 1:
            return None
        ident = [B.nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ident, src=0)
        return ident[0]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t)
        return float(t.item())

    t0 = time.time()
    rows, cols, vals, nnz = gen_device_coo(torch, w, dev)
    torch.cuda.synchronize()
    t_gen = time.time() - t0
    stream = torch.cuda.Stream(device=dev)
    coo = (w["rows"], w["cols"], nnz, rows.data_ptr(), cols.data_ptr(), vals.data_ptr())
    t0 = time.time()
    ctx = B.BlockLanczos(n=w["n"], prime=w["p"], right=w["right"], device=local_rank, rank=rank, world=world,
                         nccl_id=new_id(), stream=stream.cuda_stream, chunk_len=a.chunk, device_coo=coo)
    torch.cuda.synchronize()
    t_build = time.time() - t0
    info = ctx.info()
    n, p = w["n"], w["p"]
    N, Mc = info["N"], info["Mc"]

    # start block: pinned host memory, uniform residues (the reference's xoshiro start block is a
    # host-side sequential generator, sequential/lanczos_modp.c:624-625; for a throughput run any
    # full-rank start is equivalent)
    v_host = torch.empty(N * n, dtype=torch.int32, pin_memory=True)
    v_host.random_(0, p, generator=torch.Generator().manual_seed(7))
    v_np = v_host.numpy().view(np.uint32)
    out_host = torch.empty(ctx.pad, dtype=torch.int32, pin_memory=True)
    out_np = out_host.numpy().view(np.uint32)

    ctx.set_state(v_np)
    ctx.iterate(a.warmup)                       # warm-up steps (untimed)

    # -------- device-resident timed region: K steps, CUDA events on the library's stream
    sampler = ClockSampler(local_rank)
    ctx.set_profiling(True)
    launches0 = ctx.kernel_launches()
    barrier()
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(stream):
        e0.record(stream)
        it, stopped = ctx.iterate(a.steps)
        e1.record(stream)
    barrier()
    clocks = sampler.finish()
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    launches = ctx.kernel_launches() - launches0
    phases = ctx.phase_times()
    ctx.set_profiling(False)
    assert not stopped, "the synthetic run hit the termination condition inside the timed region"
    assert it == a.warmup + a.steps
    value = a.steps / (ms_total / 1e3)

    # -------- the state after warmup + steps iterations, hashed: identical for every number of GPUs
    # (blk_get_state is collective: every rank asks for v; rank 0 hashes it)
    ctx.L.blk_get_state(ctx.h, out_np.ctypes.data, None, None, None)
    state_sha256 = hashlib.sha256(out_np[:N * n].tobytes()).hexdigest() if rank == 0 else None
    if a.dump_outputs:
        dump_outputs(np, ctx, out_np, n, rank, a.dump_outputs)

    # -------- end to end through the C ABI with host buffers
    e2e = None
    if not a.no_e2e:
        lo, hi = info["local_N0"], info["local_N1"]
        moved = (hi - lo) * n * 4                              # bytes of this rank's rows, each way
        barrier()
        t0 = time.perf_counter()
        ctx.set_state(v_np)                                   # H2D of this rank's rows of the start block (pinned)
        t1 = time.perf_counter()
        for _ in range(a.steps):
            ctx.iterate(1)                                    # returns (n_iterations, stopped) to the host
        t2 = time.perf_counter()
        ctx.get_state_local(v=out_np)                         # D2H of this rank's rows of v
        t3 = time.perf_counter()
        barrier()
        t4 = time.perf_counter()
        dt = max_over_ranks(t4 - t0)
        # a plain pinned-memory copy of the same size next to it: what this box's PCIe path gives any program
        probe = torch.empty(moved // 4, dtype=torch.int32, device=dev)
        torch.cuda.synchronize()
        tp = time.perf_counter()
        probe.copy_(v_host[lo * n:hi * n], non_blocking=True)
        torch.cuda.synchronize()
        probe_h2d = moved / (time.perf_counter() - tp) / 1e9
        del probe
        total_moved = sum_over_ranks(float(moved))
        e2e = {"value": a.steps / dt, "unit": UNIT,
               "h2d_bytes_per_step": int(total_moved / a.steps + 32 * world), "d2h_bytes_per_step": int(total_moved / a.steps + 32 * world),
               "seconds": {"set_state": t1 - t0, "iterate": t2 - t1, "get_state": t3 - t2},
               "pcie": {"h2d_gbs_this_rank": moved / (t1 - t0) / 1e9, "d2h_gbs_this_rank": moved / (t3 - t2) / 1e9,
                        "plain_pinned_copy_h2d_gbs": probe_h2d, "bytes_this_rank_each_way": moved, "cpu_affinity": numa,
                        "note": "set_state also all-gathers v over NVLink and (N > 1) runs one sparse product to set up the loop"},
               "note": "blk_set_state + K x blk_iterate(1) + blk_get_state_local(v); every rank moves only its own rows "
                       "over PCIe; state copies amortised over K"}

    # -------- roofline of the SpMV kernel (both products), SURVEY 8(d) algorithmic bytes
    peak, peak_src = peaks()
    nnz1, nnz2 = info["nnz_local"]
    r1, r2 = info["local_M1"] - info["local_M0"], info["local_N1"] - info["local_N0"]
    b1, g1, l1 = spmv_bytes(nnz1, r1, N, n, info["n_pad"])
    b2, g2, l2 = spmv_bytes(nnz2, r2, Mc, n, info["n_pad"])
    t_spmv = (phases["spmv1"]["ms"] + phases["spmv2"]["ms"]) / a.steps          # ms per iteration, this rank
    achieved = (b1 + b2) / (t_spmv * 1e-3) / 1e9
    achieved_g = (g1 + g2) / (t_spmv * 1e-3) / 1e9
    achieved_l = (l1 + l2) / (t_spmv * 1e-3) / 1e9
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "spmv_traffic.json")
    tnote = ""
    if os.path.exists(tpath):
        tj = json.load(open(tpath))
        if tj.get("workload") == a.workload and tj.get("n_gpus", 1) == world:
            traffic = tj.get("dram_bytes_per_launch")
            tnote = tj.get("source", "")
    dram = None
    if traffic:
        # both products move the same bytes to within a few %; `traffic` is one launch
        dram = {"bytes_per_launch": traffic, "achieved": 2 * traffic / (t_spmv * 1e-3) / 1e9,
                "frac": 2 * traffic / (t_spmv * 1e-3) / 1e9 / peak,
                "note": "ncu dram__bytes_read+write of one k_spmv launch (" + tnote + "): every L2 miss fills a 128 B line, "
                        "so a 64 B x-row gather costs 128 B of HBM traffic (profiles/r01_gather_granularity.txt)"}
    roofline = {"kernel": "k_spmv (both products of one iteration)", "bound": "hbm", "achieved": achieved,
                "peak": peak, "peak_source": peak_src, "unit": "GB/s", "frac": achieved / peak,
                "algorithmic_bytes_per_iteration": b1 + b2, "traffic": traffic, "dram": dram,
                "gather_model": {"bytes_per_iteration": g1 + g2, "achieved": achieved_g, "frac": achieved_g / peak,
                                 "note": "x block (3.2 GB) >> L2: every non-zero gathers its own 4n-byte x row"},
                "line_model": {"bytes_per_iteration": l1 + l2, "achieved": achieved_l, "frac": achieved_l / peak,
                               "note": "what the memory system must move for a gather formulation: a whole 128-byte line "
                                       "per gathered x row (profiles/r01_gather_granularity.txt, profiles/r02_band_probe.txt)"},
                "ms_per_launch_pair": t_spmv, "frac_of_nominal_8TBs": achieved / 8000.0}
    spmv_rate = sum_over_ranks((nnz1 + nnz2) * n / (t_spmv * 1e-3) / 1e9)

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": ms_total / a.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "u32 (u64 accumulate)", "data": "synthetic", "config": dict(config, nnz=nnz),
            "state_sha256": state_sha256, "state_iterations": a.warmup + a.steps,
            "spmv_gnnzn_per_s": spmv_rate, "clocks": clocks, "gpu_launches": int(launches), "roofline": roofline,
            "phases_ms_per_step": {k: v["ms"] / a.steps for k, v in phases.items()},
            "setup_s": {"generate": t_gen, "build_layout": t_build}, "device_bytes": info["device_bytes"]}
    try:
        line["roofline_dense"] = dense_roofline(line["phases_ms_per_step"], info["local_N1"] - info["local_N0"], info["n_pad"], peak)
    except Exception as exc:          # secondary information must never cost the bench line
        line["roofline_dense"] = {"error": str(exc)}
    if e2e:
        line["e2e"] = e2e
    ctx.close()
    del v_host, out_host, v_np, out_np

    if not a.no_extras:
        # -------- BASELINE configs[4]: the SpMV-only sweep on the same matrix (sharded over the ranks)
        try:
            line["spmv_sweep"] = spmv_sweep(B, torch, w, coo, nnz, local_rank, rank, world, new_id, max_over_ranks, stream, peak,
                                            a.sweep_budget_s)
        except Exception as exc:
            line["spmv_sweep"] = {"error": f"{type(exc).__name__}: {exc}"}
    del rows, cols, vals
    torch.cuda.empty_cache()
    if not a.no_extras:
        # -------- parity: the library on a CPU-sized twin, sharded like this run, against the oracle
        try:
            line["parity"] = parity_check(B, torch, np, local_rank, rank, world, new_id)
        except Exception as exc:
            line["parity"] = {"ok": False, "error": f"{type(exc).__name__}: {exc}"}
        # -------- BASELINE configs[0..2]: complete runs (latency-bound; one GPU)
        if world == 1:
            try:
                line["small_configs"] = small_configs(B, np)
            except Exception as exc:
                line["small_configs"] = {"error": f"{type(exc).__name__}: {exc}"}

    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        r = run_cpu_reference(w, 3, 1, spmv_reps=2)
        if r:
            line["cpu_baseline"] = cpu_baseline_obj(r, w, nnz)
            try:
                line["cpu_baseline"].update(cpu_baseline_extras(w, r["threads"]))
            except Exception as exc:
                line["cpu_baseline"]["extras_error"] = str(exc)
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


def dump_outputs(np, ctx, buf, n, rank, out_dir):
    """--dump-outputs: what a caller of the timed path receives after its last step, as DIR/<name>.npy in float64
    (exact for residues < 2^32).  v, tmp, Av, p: the blocks of blk_get_state, as rows x n -- every padded row, or
    DUMP_ROWS rows drawn with a fixed seed (sorted) when there are more.  vtAv, vtAAv, winv, d: the n x n matrices
    of that step (blk_get_small).  blk_get_state is collective, so every rank takes part; rank 0 writes.  `buf` is
    a host buffer of ctx.pad residues."""
    R = ctx.pad // n
    rows = np.arange(R) if R <= DUMP_ROWS else np.sort(np.random.default_rng(0).choice(R, DUMP_ROWS, replace=False))
    out = {}
    for k, name in enumerate(("v", "tmp", "Av", "p")):
        ptrs = [None] * 4
        ptrs[k] = buf.ctypes.data
        ctx._ck(ctx.L.blk_get_state(ctx.h, *ptrs))
        out[name] = buf.reshape(R, n)[rows]
    small = ctx.get_small()
    out.update(vtAv=small["vtAv"].reshape(n, n), vtAAv=small["vtAAv"].reshape(n, n), winv=small["winv"].reshape(n, n),
               d=small["d"])
    if rank == 0:
        os.makedirs(out_dir, exist_ok=True)
        for name, arr in out.items():
            np.save(os.path.join(out_dir, name + ".npy"), arr.astype(np.float64))


def spmv_sweep(B, torch, w, coo, nnz, local_rank, rank, world, new_id, max_over_ranks, stream, peak, budget_s):
    """blk_time_spmv for every (n, p) of BASELINE configs[4] on the resident COO of the workload; both directions;
    time = the slowest rank's; fractions of the measured HBM peak for the three byte models."""
    out = {"matrix": "the workload's matrix", "nnz": nnz, "reps": 3, "unit_ms": "ms per product (max over ranks)", "points": []}
    t_start = time.time()
    N, Mc = (w["cols"], w["rows"]) if w["right"] else (w["rows"], w["cols"])
    for n in SWEEP_NS:
        for p in SWEEP_PRIMES:
            over = max_over_ranks(1.0 if time.time() - t_start > budget_s else 0.0)      # all ranks stop together
            if over:
                out["truncated"] = f"time box of {budget_s:.0f} s reached"
                return out
            ctx = B.BlockLanczos(n=n, prime=p, right=w["right"], device=local_rank, rank=rank, world=world,
                                 nccl_id=new_id(), stream=stream.cuda_stream, device_coo=coo)
            inf = ctx.info()
            rec = {"n": n, "p": p, "column_bands": inf.get("bands")}
            for tr in (False, True):
                ms = max_over_ranks(ctx.time_spmv(tr, 3))
                rows_out, rows_in = (w["cols"], w["rows"]) if tr else (w["rows"], w["cols"])
                alg, gather, linem = spmv_bytes(nnz, rows_out, rows_in, n, inf["n_pad"])
                rec["Mt_x" if tr else "M_x"] = {
                    "ms": ms, "gnnzn_per_s": nnz * n / (ms * 1e-3) / 1e9,
                    "frac_algorithmic": alg / (ms * 1e-3) / 1e9 / peak / world,
                    "frac_gather_model": gather / (ms * 1e-3) / 1e9 / peak / world,
                    "frac_line_model": linem / (ms * 1e-3) / 1e9 / peak / world}
            out["points"].append(rec)
            ctx.close()
    out["seconds"] = time.time() - t_start
    out["note"] = ("fractions are of the measured copy bandwidth x number of GPUs; algorithmic = each x row once (SURVEY 8d), "
                   "gather = 4n bytes per non-zero, line = one 128-byte line per non-zero (what a gather must move on B200 when x "
                   "misses L2).  n <= 4: the operators run as column bands whose x slice is L2-resident (column_bands = bands of "
                   "S1, S2), so their line-model fraction exceeds 1 -- those lines are no longer fetched from HBM")
    return out


def parity_check(B, torch, np, local_rank, rank, world, new_id):
    """cfg4_tiny through the same library and the same sharding, 4 iterations, every block against the CPU oracle
    (rank 0 compares; the oracle is the checker, never on a timed path)."""
    w = WORKLOADS["cfg4_tiny"]
    M = B.synth.powerlaw_rows(w["rows"], w["cols"], mean=w["mean"], seed=1).reduced(w["p"])
    n, p, iters = w["n"], w["p"], 4
    ctx = B.BlockLanczos(M, n=n, prime=p, right=w["right"], device=local_rank, rank=rank, world=world, nccl_id=new_id())
    v0 = np.random.default_rng(11).integers(0, p, size=M.nrows * n).astype(np.uint32)
    got = ctx.block_lanczos(v0, stop_after=iters, batch=iters)
    ctx.close()
    if rank != 0:
        return None
    from oracle.oracle import Oracle
    O = Oracle()
    pad = got["v"].size
    st = dict(v=np.zeros(pad, np.uint32), tmp=np.zeros(pad, np.uint32), Av=np.zeros(pad, np.uint32), p=np.zeros(pad, np.uint32), iters=0)
    st["v"][:v0.size] = v0
    t0 = time.time()
    want = O.lanczos_run(M, n, p, w["right"], stop_after=iters, state=st)
    same = {k: bool(np.array_equal(got[k], want[k])) for k in ("v", "tmp", "Av", "p")}
    return {"workload": "cfg4_tiny", "rows": M.nrows, "nnz": M.nnz, "n": n, "prime": p, "iterations": iters, "n_gpus": world,
            "blocks_identical_to_oracle": same, "ok": all(same.values()) and got["iters"] == want["iters"],
            "oracle": O.kind, "oracle_seconds": time.time() - t0}


def small_configs(B, np):
    """BASELINE configs[0..2] run to termination on one GPU: us per iteration, total seconds, kernel property."""
    out = []
    for k in (1, 2, 3):
        M, a = B.synth.baseline_config(k)
        p, n, right = a["p"], a["n"], a["right"]
        N = M.ncols if right else M.nrows
        ctx = B.BlockLanczos(M.reduced(p), n=n, prime=p, right=right)
        v0 = np.random.default_rng(5 + k).integers(0, p, size=N * n).astype(np.uint32)
        ctx.set_state(v0)
        ctx.iterate(64)                                # warm-up (graph capture / kernel load)
        ctx.set_state(v0)
        t0 = time.perf_counter()
        it, stopped = 0, False
        while not stopped:
            it, stopped = ctx.iterate(4096)
        dt = time.perf_counter() - t0
        ok = ctx.final_check() == (True, True)
        out.append(dict(config=k, rows=M.nrows, cols=M.ncols, nnz=M.nnz, n=n, p=p, right=right, iterations=it,
                        seconds=dt, us_per_iter=dt / it * 1e6, kernel_ok=bool(ok), launches=ctx.kernel_launches()))
        ctx.close()
    return out


if __name__ == "__main__":
    sys.exit(main())
