#!/usr/bin/env python
"""Subset pushes of a live fleet across ranks (run under torchrun with the nccl backend, one rank per GPU):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 \\
        --master-port 29514 tests/stream_subset_dist_check.py

Streams are sharded contiguously and every push names streams of the rank's own shard; a rank with nothing to push
calls push(streams=[]) so that it takes part in the all-reduce.  The all-reduced Recall@N counters of every push and
the session precision-recall (reduce=True) must equal what one process computes alone for the whole fleet over the
same schedule.  Run by tests/test_gpu_stream_subsets.py when the box has >= 2 GPUs.
"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from lens_b200 import synth  # noqa: E402
from lens_b200.pipeline import StreamingPipeline, shard_range  # noqa: E402


def same(a, b):
    return all(np.array_equal(np.array(a[k], np.float64), np.array(b[k], np.float64), equal_nan=True)
               for k in ("P", "R", "tp", "fp")) and a["gtp"] == b["gtp"]


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    B, P, L, tol = 10, 300, 3, 1
    Wf, Wo = synth.weights(100, 96, P, seed=3)
    W = (torch.from_numpy(Wf), torch.from_numpy(Wo))
    pooled = torch.from_numpy(synth.pixel_counts((B, 40, 100), 7)).to(dev)
    rng = np.random.default_rng(11)
    shards = [shard_range(B, r, world) for r in range(world)]
    lo, hi = shards[rank]
    mk = lambda n: StreamingPipeline(*W, roi=80, k=8, T=30, L=L, n_streams=n, device=dev,   # noqa: E731
                                     track_pr=("place", "query", "multi"))
    mine, alone = mk(hi - lo), mk(B)
    cursor = np.zeros(B, np.int64)
    ok = True
    for k in range(10):
        Q = int(rng.integers(1, 3))
        pushed = []                                    # fleet indices, every rank's own subset in random order
        for r, (a, b) in enumerate(shards):
            take = rng.permutation(np.arange(a, b))[:int(rng.integers(0, b - a + 1))]
            if r == 1 and k % 3 == 0:
                take = take[:0]                        # this rank has nothing to push
            pushed.append(take.tolist())
        every = [b for p in pushed for b in p]
        win = torch.stack([pooled[b, cursor[b]:cursor[b] + Q] for b in every]) if every else None
        gt = torch.from_numpy(rng.integers(-1, P - L + 1, size=(len(every), Q)).astype(np.int32)).to(dev)
        cursor[every] += Q
        o0 = sum(len(p) for p in pushed[:rank])
        own = pushed[rank]
        got = mine.push(pooled=None if not own else win[o0:o0 + len(own)].contiguous(),
                        gt_center=gt[o0:o0 + len(own)].contiguous(), gt_tol=tol, streams=[b - lo for b in own])
        want = alone.push(pooled=win, gt_center=gt, gt_tol=tol, streams=every, reduce=False)
        ok &= torch.equal(got["hits"], want["hits"]) and torch.equal(got["n_valid"], want["n_valid"])
    for matching, best in (("single", "place"), ("single", "query"), ("multi", "place")):
        kw = dict(matching=matching, best=best, n_thresh=64)
        ok &= same(mine.session_precision_recall(**kw), alone.session_precision_recall(reduce=False, **kw))
    print(f"stream_subset_dist_check rank={rank} world={world}: {'OK' if ok else 'MISMATCH'}")
    dist.barrier()
    dist.destroy_process_group()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
