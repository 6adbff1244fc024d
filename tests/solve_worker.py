"""Worker for tests/test_gpu_solve.py: one process per GPU (torchrun).  Every rank builds the augmented system
(blk_create_system), runs the loop to the end, solves (the tail rows of v meet in one NCCL all-reduce inside the
library) and checks x and found against the CPU restatement."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import blk_lanczos_b200 as B          # noqa: E402
from oracle.oracle import Oracle      # noqa: E402
import solve_oracle                   # noqa: E402


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    O = Oracle()
    s = B.synth
    cases = [(s.powerlaw_rows(2800, 2600, mean=6, seed=21, with_empty_rows=7), 32, 4, 3, False),
             (s.uniform_rows(1900, 2000, 5, seed=2), 16, 8, 65537, True),
             (s.uniform_rows(1500, 1400, 5, seed=4), 8, 1, 2147483647, False)]
    for ci, (M, n, r, p, right) in enumerate(cases):
        Mp = M.reduced(p)
        N = M.ncols if right else M.nrows
        X0 = np.random.default_rng(ci).integers(0, p, size=(N, r), dtype=np.int64).astype(np.uint32)
        Bm = O.sparse_matrix_vector_product(Mp, X0.ravel(), not right, r, p).reshape(-1, r)
        ident = [B.nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ident, src=0)
        with B.BlockLanczos(Mp, n=n, prime=p, right=right, device=local, rank=rank, world=world, nccl_id=ident[0],
                            rhs=Bm) as ctx:
            got = ctx.block_lanczos(O.start_block((N + r) * n, p), batch=32)
            x, found = ctx.solve()
        A = solve_oracle.augmented(Mp, Bm, p, right)
        want = O.lanczos_run(A, n, p, right)
        assert np.array_equal(got["v"], want["v"]), (ci, rank)
        rx, rf = solve_oracle.solve(Mp, Bm, want["v"][:(N + r) * n], n, p, right)
        assert np.array_equal(found, rf) and np.array_equal(x, rx), (ci, rank)
        dist.barrier()
    if rank == 0:
        print("SOLVE_OK world=%d" % world)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
