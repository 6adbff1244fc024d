"""Worker for tests/test_gpu_prune.py: one process per GPU (torchrun).  Every rank prunes the whole COO itself
(blk_create_pruned), runs the loop on M' to the end and checks the kept indices, the stats and the state against the
CPU restatement and the oracle's loop on M'."""
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
import prune_oracle                   # noqa: E402


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    O = Oracle()
    s = B.synth
    cases = [(s.powerlaw_rows(2800, 2600, mean=6, seed=21, with_empty_rows=7), 32, 3, False),
             (s.uniform_rows(3000, 3000, 3, seed=2), 16, 65537, True),
             (s.uniform_rows(2000, 1900, 3, seed=4), 8, 2147483647, False)]
    for ci, (M, n, p, right) in enumerate(cases):
        ref = prune_oracle.prune(M, p, right)
        ident = [B.nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ident, src=0)
        with B.BlockLanczos(M, n=n, prime=p, right=right, device=local, rank=rank, world=world, nccl_id=ident[0],
                            prune=True) as ctx:
            assert ctx.prune_stats == ref["stats"], (ci, rank)
            u, c = ctx.pruned_index()
            assert np.array_equal(u, ref["unknowns"]) and np.array_equal(c, ref["constraints"]), (ci, rank)
            got = ctx.block_lanczos(O.start_block(ctx.N * n, p), batch=32)
        want = O.lanczos_run(ref["M"], n, p, right)
        assert got["iters"] == want["iters"] and np.array_equal(got["v"], want["v"]), (ci, rank)
        dist.barrier()
    if rank == 0:
        print("PRUNE_OK world=%d" % world)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
