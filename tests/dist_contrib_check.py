"""Multi-GPU check of sharded contribution scores (run under torchrun on a GPU box):

  python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 tests/dist_contrib_check.py [config]

Every rank scores its contiguous block of the view's sub-frames (deblurgs_b200.dist.render_blurry_sharded with
`contrib=`), then dist.all_reduce_contribution combines them over NCCL.  Every rank compares the result with the
scores of the unsharded view computed on its own GPU: they must be the same bits.
"""
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402
from deblurgs_b200 import dist as dd  # noqa: E402
from deblurgs_b200.rasterizer import ContributionScores  # noqa: E402


def main():
    cfg = sys.argv[1] if len(sys.argv) > 1 else "small"
    rank, world, local = bench.dist_setup(0)
    dev = torch.device("cuda", local)
    w = bench.build_workload(cfg, 0, dev)          # same store and view on every rank
    cmm, P = w["cmm"], w["P"]
    with torch.no_grad():
        full = cmm.accumulate_contribution(w["bg"])
        sharded = ContributionScores(P, dev)
        _, _, (a, b) = dd.render_blurry_sharded(cmm, 0, w["bg"], contrib=sharded)
        local_sum = int(sharded.wsum.sum())
        dd.all_reduce_contribution(sharded)
    torch.cuda.synchronize()
    ok = torch.equal(full.wsum, sharded.wsum) and torch.equal(full.wmax, sharded.wmax) and int(full.wsum.sum()) > 0
    print("rank %d/%d: sub-frames [%d, %d), local weight sum %.3f, combined %.3f, unsharded %.3f: %s"
          % (rank, world, a, b, local_sum / 2 ** 26, int(sharded.wsum.sum()) / 2 ** 26, int(full.wsum.sum()) / 2 ** 26,
             "equal" if ok else "DIFFERENT"), flush=True)
    flags = torch.tensor([int(ok)], device=dev)
    if world > 1:
        dist.all_reduce(flags, op=dist.ReduceOp.MIN)
    if rank == 0:
        print("contrib sharding OK" if int(flags.item()) else "contrib sharding FAILED", flush=True)
    if dist.is_initialized():
        dist.destroy_process_group()
    sys.exit(0 if int(flags.item()) else 1)


if __name__ == "__main__":
    main()
