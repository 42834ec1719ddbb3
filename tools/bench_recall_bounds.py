#!/usr/bin/env python
"""Tie-aware Recall@N bounds straight from the spike counts: what bounds=True costs a step and a push, on one GPU.

    python tools/bench_recall_bounds.py [--steps K] [--warmup W] [--shapes fleet3,large_map] [--streams B]

Workload as tools/bench_pr.py (LENS I=100 -> F=200 -> P, synth.weights, T=250, 80x80 count frames, k=8, band
tolerance 2).  Per shape:
  batch  one real step's S (fleet3: 65 536 streams x Q=10 x P=10 000, L=10, S is 26.2 GB; large_map: 1 stream x
         Q=300 x P=100 000).  ops.seq_recall_bounds timed with CUDA events, with two ground truths: centres at K4's own
         top-1 (every column is scanned to the end: the worst case) and random centres (synth.gt_centers), beside K4
         (ops.seqmatch_topk, top-25) and the step.  Bytes counted: S once.
  push   a StreamingPipeline of the same fleet, one window per stream and push: push end to end with bounds off and
         on (random centres), and the bounds call alone on a fixed state for both ground truths.  Bytes counted: S
         once plus the L - 1 ring rows of every stream.
early_exit_fraction: valid rows with A >= max(ns) (A = places ranked strictly above the best positive), whose scan
stops as soon as that is reached.  Checked in the same run: 4 sampled streams' bounds against the oracle
(O.recall_bounds on O.seqmatch), and lo <= hits <= hi with n_valid equal to the step's.  One JSON line on stdout with
the card's name and power limit; nothing is written.
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench import load_peaks   # noqa: E402
from bench_stream import gpu_info, timed   # noqa: E402

I_DIMS, FEATURE, ROI, K_POOL, T_STEPS, N_TOP, TOL = 10, 200, 80, 8, 250, 25, 2
NS = (1, 5, 10, 15, 20, 25)
SHAPES = {"fleet3": dict(streams=65536, places=10000, queries=10, seq_len=10),
          "large_map": dict(streams=1, places=100000, queries=300, seq_len=10)}


def oracle_sample(torch, S, gt, L, sample):
    """seq_recall_bounds on each sampled stream == O.recall_bounds on the oracle's own sequence-matched matrix."""
    from lens_b200 import ops
    from oracle import oracle as O
    ok = True
    for b in sample:
        lo, hi, nv = ops.seq_recall_bounds(S[b:b + 1].contiguous(), L, gt_center=gt[b:b + 1].contiguous(), gt_tol=TOL,
                                           ns=NS)
        D = O.seqmatch(S[b].cpu().numpy(), L)
        c = gt[b].cpu().numpy()
        G = (c[None, :] >= 0) & (np.abs(np.arange(D.shape[0])[:, None] - c[None, :]) <= TOL)
        n = int(G.any(0).sum())
        for i, K in enumerate(NS):
            fl, fh = O.recall_bounds(D, G, K) if n else (0.0, 0.0)
            ok &= int(lo[i]) == round(fl * n) and int(hi[i]) == round(fh * n)
        ok &= int(nv.item()) == int((c >= 0).sum())
    return dict(streams=list(sample), equal=bool(ok))


def run_shape(torch, args, peaks, c):
    from lens_b200 import ops, synth
    from lens_b200.pipeline import InferencePipeline, StreamingPipeline
    B, P, Q, L = args.streams or c["streams"], c["places"], c["queries"], c["seq_len"]
    Po, Qo = P - L + 1, Q - L + 1
    Wf, Wo = synth.weights(I_DIMS * I_DIMS, FEATURE, P, seed=1)
    W = (torch.from_numpy(Wf), torch.from_numpy(Wo))
    peak = peaks["hbm_gbs"]

    def rate(nbytes, ms, whole_ms, k4_ms):
        gbs = nbytes / (ms / 1e3) / 1e9
        return dict(ms=ms, bytes=int(nbytes), achieved_GBps=gbs, frac_of_hbm_peak=gbs / peak,
                    frac_of_whole=ms / whole_ms, k4_ms=k4_ms)

    def early(lo_hi_nv):
        _, hi, nv = lo_hi_nv
        nv = int(nv.item())
        return (nv - int(hi[-1].item())) / nv if nv else None

    # ---- batch
    pipe = InferencePipeline(*W, roi=ROI, k=K_POOL, T=T_STEPS, L=L, n_top=N_TOP, ns=NS, max_streams=B)
    frames = synth.frames_device(B, Q, roi=ROI, seed=2)
    gt_rand = torch.from_numpy(synth.gt_centers(B, Qo, Po, seed=7)).cuda()
    pipe.step(frames=frames)
    ms_step = timed(torch, lambda i: pipe.step(frames=frames), 1)
    out_step = pipe.step(frames=frames, gt_center=gt_rand, gt_tol=TOL, bounds=True)
    S = out_step["S"]
    del frames
    torch.cuda.empty_cache()
    lo, hi, h = (out_step[k].cpu() for k in ("hits_lo", "hits_hi", "hits"))
    invariants = bool((lo <= h).all() and (h <= hi).all())
    k4 = lambda i: ops.seqmatch_topk(S, L, N_TOP)     # noqa: E731
    for i in range(args.warmup):
        k4(i)
    ms_k4 = timed(torch, k4, args.steps)
    gt_top1 = k4(0)[1][..., 0].contiguous()
    out = dict(streams=B, places=P, queries=Q, seq_len=L, S_bytes=int(4 * B * Q * P), step_ms=ms_step, batch={},
               push={})
    for name, gt in (("top1", gt_top1), ("random", gt_rand)):
        call = lambda i: ops.seq_recall_bounds(S, L, gt_center=gt, gt_tol=TOL, ns=NS)    # noqa: E731
        for i in range(args.warmup):
            call(i)
        ms = timed(torch, call, args.steps)
        res = call(0)
        if name == "random":
            invariants &= torch.equal(res[2], out_step["n_valid"])
        out["batch"][name] = dict(**rate(4.0 * B * Q * P, ms, ms_step, ms_k4), early_exit_fraction=early(res))
    sample = sorted(set([0, B - 1]) | set(np.random.default_rng(3).choice(B, min(4, B), replace=False).tolist()))[:4]
    out["oracle_sample"] = oracle_sample(torch, S, gt_rand, L, sample)
    out["invariants_ok"] = invariants
    del pipe, S, out_step, gt_top1
    torch.cuda.empty_cache()

    # ---- push: one window per stream
    sp = StreamingPipeline(*W, roi=ROI, k=K_POOL, T=T_STEPS, L=L, n_streams=B, n_top=N_TOP, ns=NS)
    n_frames = 4
    frames = synth.frames_device(B, n_frames, roi=ROI, seed=2)
    pushes = [frames[:, i:i + 1].contiguous() for i in range(n_frames)]
    del frames
    gt = torch.from_numpy(synth.gt_centers(B, 1, Po, seed=7)).cuda()
    for bounds in (False, True):
        push = lambda i: sp.push(frames=pushes[i % n_frames], gt_center=gt, gt_tol=TOL, bounds=bounds)   # noqa: E731
        for i in range(max(args.warmup, L)):
            push(i)
        out["push"]["push_ms_bounds_" + ("on" if bounds else "off")] = timed(torch, push, args.steps)
    S = push(0)["S"]
    ring, seen = sp.ring.clone(), sp.seen.clone()
    match = lambda i: ops.seqmatch_topk_stream(S, L, N_TOP, ring, seen, sp.t)     # noqa: E731 (on a copy of the state)
    ms_match = timed(torch, match, 1)
    ring.copy_(sp.ring)
    seen.copy_(sp.seen)
    gt_top1 = match(0)[1][..., 0].contiguous()
    del ring, seen
    nbytes = 4.0 * B * (L - 1 + 1) * P
    for name, g in (("top1", gt_top1), ("random", gt)):
        call = lambda i: ops.seq_recall_bounds_stream(S, L, sp.ring, sp.seen, sp.t, g, TOL, ns=NS)   # noqa: E731
        for i in range(args.warmup):
            call(i)
        ms = timed(torch, call, args.steps)
        out["push"][name] = dict(**rate(nbytes, ms, out["push"]["push_ms_bounds_off"], ms_match),
                                 early_exit_fraction=early(call(0)))
    out["ok"] = out["invariants_ok"] and out["oracle_sample"]["equal"]
    del sp, S, pushes
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--shapes", default="fleet3,large_map")
    ap.add_argument("--streams", type=int, default=None, help="override the stream count (rehearsals)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_recall_bounds.py needs a CUDA device")
    peaks = load_peaks()
    out = dict(metric="recall_bounds", **gpu_info(), peaks_source=peaks["source"], hbm_peak_GBps=peaks["hbm_gbs"],
               roi="80x80", k=K_POOL, timesteps=T_STEPS, feature=FEATURE, gt_tol=TOL, ns=list(NS), steps=args.steps)
    for s in args.shapes.split(","):
        out[s] = run_shape(torch, args, peaks, SHAPES[s])
    out["ok"] = all(out[s]["ok"] for s in args.shapes.split(","))
    print(json.dumps(out))
    if not out["ok"]:
        sys.exit(1)


if __name__ == "__main__":
    main()
