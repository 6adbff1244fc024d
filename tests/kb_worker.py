"""Worker for tests/test_gpu_kernel_basis.py: one process per GPU (torchrun).  Every rank runs the loop to the
end, extracts the kernel basis (one NCCL all-gather of the ranks' bases inside the library) and checks the
block and k against the CPU oracle; the single-process group context (BLK_RANK_ALL) must agree."""
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
import kb_oracle                      # noqa: E402


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    O = Oracle()
    s = B.synth
    cases = [(s.powerlaw_rows(2800, 2600, mean=6, seed=21, with_empty_rows=7), 32, 3, False),
             (s.uniform_rows(1900, 2000, 5, seed=2), 16, 2, True),
             (s.uniform_rows(1500, 1400, 5, seed=4), 8, 65537, False)]
    for ci, (M, n, p, right) in enumerate(cases):
        Mp = M.reduced(p)
        N = M.ncols if right else M.nrows
        ident = [B.nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ident, src=0)
        with B.BlockLanczos(Mp, n=n, prime=p, right=right, device=local, rank=rank, world=world, nccl_id=ident[0]) as ctx:
            got = ctx.block_lanczos(O.start_block(N * n, p), batch=32)
            X = ctx.kernel_basis()
        want = O.lanczos_run(Mp, n, p, right)
        assert np.array_equal(got["v"], want["v"]), (ci, rank)
        ref = kb_oracle.kernel_basis(Mp, want["v"][:N * n], n, p, right)
        assert X.shape == ref.shape and np.array_equal(X, ref), (ci, rank, X.shape, ref.shape)
        dist.barrier()
    if rank == 0:
        print("KB_OK world=%d" % world)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
