#!/usr/bin/env python
"""Session precision-recall of a live fleet across ranks (run under torchrun with the nccl backend, one rank per GPU):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 \\
        --master-port 29513 tests/stream_pr_dist_check.py

Streams are sharded contiguously; every rank's session_precision_recall(reduce=True) must equal, in every mode, what
one process computes alone for the whole fleet (the thresholds span all ranks), and reduce=False must give the rank's
own curve.  Run by tests/test_gpu_stream_pr.py when the box has >= 2 GPUs.
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
    B, Q, P, L, tol = 10, 9, 300, 3, 1
    Wf, Wo = synth.weights(100, 96, P, seed=3)
    W = (torch.from_numpy(Wf), torch.from_numpy(Wo))
    pooled = synth.pixel_counts((B, Q, 100), 7)
    c = np.random.default_rng(11).integers(-1, P - L + 1, size=(B, Q)).astype(np.int32)
    lo, hi = shard_range(B, rank, world)
    mk = lambda n: StreamingPipeline(*W, roi=80, k=8, T=30, L=L, n_streams=n, device=dev,   # noqa: E731
                                     track_pr=("place", "query", "multi"))
    mine, alone = mk(hi - lo), mk(B)
    for q0, n in ((0, 2), (2, 1), (3, 6)):
        sl = slice(q0, q0 + n)
        mine.push(pooled=torch.from_numpy(pooled[lo:hi, sl].copy()).to(dev),
                  gt_center=torch.from_numpy(c[lo:hi, sl].copy()).to(dev), gt_tol=tol)
        alone.push(pooled=torch.from_numpy(pooled[:, sl].copy()).to(dev),
                   gt_center=torch.from_numpy(c[:, sl].copy()).to(dev), gt_tol=tol, reduce=False)
    ok = True
    for matching, best in (("single", "place"), ("single", "query"), ("multi", "place")):
        kw = dict(matching=matching, best=best, n_thresh=64)
        got = mine.session_precision_recall(**kw)
        whole = alone.session_precision_recall(reduce=False, **kw)
        own = mine.session_precision_recall(reduce=False, **kw)
        ok &= same(got, whole) and not same(own, whole)
    print(f"stream_pr_dist_check rank={rank} world={world}: {'OK' if ok else 'MISMATCH'}")
    dist.barrier()
    dist.destroy_process_group()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
