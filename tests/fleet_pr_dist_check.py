#!/usr/bin/env python
"""Fleet precision-recall across ranks (run under torchrun with the nccl backend, one rank per GPU):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 \
        --master-port 29512 tests/fleet_pr_dist_check.py

Streams are sharded contiguously; every rank's precision_recall(reduce=True) must equal, in every mode, what one
rank computes alone for the whole fleet (the thresholds span all ranks), and reduce=False must give the rank's own
curve.  Run by tests/test_gpu_fleet_pr.py when the box has >= 2 GPUs.
"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from lens_b200 import synth  # noqa: E402
from lens_b200.pipeline import InferencePipeline, shard_range  # noqa: E402


def same(a, b):
    return all(np.array_equal(np.array(a[k], np.float64), np.array(b[k], np.float64), equal_nan=True)
               for k in ("P", "R", "tp", "fp")) and a["gtp"] == b["gtp"]


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    B, Q, P, L = 9, 8, 300, 3
    rng = np.random.default_rng(11)
    S = rng.poisson(1.3, size=(B, Q, P)).astype(np.float32)
    S[: B // 2] *= 2                                   # ranks see different value ranges
    c = rng.integers(-1, P - L + 1, size=(B, Q - L + 1)).astype(np.int32)
    Wf, Wo = synth.weights(4, 8, 3, seed=1)
    pipe = InferencePipeline(torch.from_numpy(Wf), torch.from_numpy(Wo), roi=2, k=1, T=1, L=L, device=dev)
    lo, hi = shard_range(B, rank, world)
    mine = dict(S=torch.from_numpy(S[lo:hi]).to(dev), gt_center=torch.from_numpy(c[lo:hi]).to(dev))
    whole = dict(S=torch.from_numpy(S).to(dev), gt_center=torch.from_numpy(c).to(dev))
    ok = True
    for matching, best in (("single", "place"), ("single", "query"), ("multi", "place")):
        kw = dict(gt_tol=1, matching=matching, best=best, n_thresh=64)
        got = pipe.precision_recall(mine["S"], gt_center=mine["gt_center"], **kw)
        alone = pipe.precision_recall(whole["S"], gt_center=whole["gt_center"], reduce=False, **kw)
        own = pipe.precision_recall(mine["S"], gt_center=mine["gt_center"], reduce=False, **kw)
        ok &= same(got, alone) and not same(own, alone)
    print(f"fleet_pr_dist_check rank={rank} world={world}: {'OK' if ok else 'MISMATCH'}")
    dist.barrier()
    dist.destroy_process_group()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
