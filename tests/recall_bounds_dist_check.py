#!/usr/bin/env python
"""Tie-aware Recall@N bounds across ranks (run under torchrun with the nccl backend, one rank per GPU):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 \\
        --master-port 29514 tests/recall_bounds_dist_check.py

Streams are sharded contiguously; a batch step and a session of pushes (one of them empty on the last rank) with
bounds=True must give, on every rank, the hits / hits_lo / hits_hi / n_valid that one process computes alone for
the whole fleet.  Run by tests/test_gpu_fleet_recall_bounds.py when the box has >= 2 GPUs.
"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from lens_b200 import synth  # noqa: E402
from lens_b200.pipeline import InferencePipeline, StreamingPipeline, shard_range  # noqa: E402

KEYS = ("hits", "hits_lo", "hits_hi", "n_valid")


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    B, Q, P, L, tol = 10, 9, 300, 3, 1
    Wf, Wo = synth.weights(100, 96, P, seed=3)
    W = (torch.from_numpy(Wf), torch.from_numpy(Wo))
    pooled = synth.pixel_counts((B, Q, 100), 7)
    c = np.random.default_rng(11).integers(-1, P - L + 1, size=(B, Q)).astype(np.int32)
    lo, hi = shard_range(B, rank, world)
    on = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)    # noqa: E731
    ok = True
    # batch steps
    mk = lambda n: InferencePipeline(*W, roi=80, k=8, T=30, L=L, max_streams=n, device=dev)   # noqa: E731
    got = mk(hi - lo).step(pooled=on(pooled[lo:hi]), gt_center=on(c[lo:hi, L - 1:]), gt_tol=tol, bounds=True)
    want = mk(B).step(pooled=on(pooled), gt_center=on(c[:, L - 1:]), gt_tol=tol, bounds=True, reduce=False)
    ok &= all(torch.equal(got[k], want[k]) for k in KEYS)
    # a session of pushes; the last rank pushes nothing in the second push
    mine = StreamingPipeline(*W, roi=80, k=8, T=30, L=L, n_streams=hi - lo, device=dev)
    alone = StreamingPipeline(*W, roi=80, k=8, T=30, L=L, n_streams=B, device=dev)
    for q0, n in ((0, 2), (2, 1), (3, 6)):
        sl = slice(q0, q0 + n)
        empty = (q0 == 2 and rank == world - 1)
        streams = [] if empty else list(range(hi - lo))
        r_lo = hi if empty else lo
        g = mine.push(pooled=on(pooled[r_lo:hi, sl]), gt_center=on(c[r_lo:hi, sl]), gt_tol=tol, streams=streams,
                      bounds=True)
        a_streams = [b for b in range(B) if not (q0 == 2 and b >= shard_range(B, world - 1, world)[0])]
        w = alone.push(pooled=on(pooled[a_streams][:, sl]), gt_center=on(c[a_streams][:, sl]), gt_tol=tol,
                       streams=a_streams, bounds=True, reduce=False)
        ok &= all(torch.equal(g[k], w[k]) for k in KEYS)
    print(f"recall_bounds_dist_check rank={rank} world={world}: {'OK' if ok else 'MISMATCH'}")
    dist.barrier()
    dist.destroy_process_group()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
