#!/usr/bin/env python
"""Live fleets whose pushes carry any subset of the streams: StreamingPipeline.push(..., streams=...) on one GPU.

    python tools/bench_stream_subsets.py [--steps K] [--warmup W] [--shapes fleet2,fleet3] [--streams B]

Workload as tools/bench_stream.py (LENS I=100 -> F=200 -> P, synth.weights, T=250, 80x80 count frames, k=8, top-25,
one window per push):
  fleet2     1 000 streams,  P = 1 000,   L = 2
  fleet3    65 536 streams,  P = 10 000,  L = 10 (its "1 camera" subset is one camera of the config-3 fleet)
Reported per shape, each as ms per push from CUDA events over --steps pushes after --warmup:
  lockstep        push() of every stream on the lockstep kernels (a session that never pushed a subset)
  permuted_all    push(streams=<all, permuted>) on the indexed kernels (SNN state gathered / scattered)
  subsets         push(streams=<random subset>) of 1/2, 1/8 and 1/64 of the fleet and of one camera, with the cost per
                  pushed stream against the lockstep push's
  match           lens_seqmatch_topk_stream (lockstep) against lens_seqmatch_topk_stream_ids over every stream in
                  permuted order, alone
  gather_scatter  the SNN state gather + scatter kernels of the permuted push (torch.profiler, a run of its own) and
                  their bytes, 2 * 2 * n * (I + F + P) * 4
Before timing, an exactness sample: a fleet of 6 streams at the shape's P and L is driven through a seeded random
schedule of subset, permuted, empty and lockstep pushes; every stream's spike counts and top-N rows must equal a
batch step over its own windows, bit for bit, with warm-up rows -inf / -1.  One JSON line on stdout; nothing is
written.
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_stream import FEATURE, I_DIMS, K_POOL, N_TOP, ROI, SHAPES, T_STEPS, gpu_info, timed   # noqa: E402

FRACTIONS = (("1/2", 2), ("1/8", 8), ("1/64", 64))


def exactness_sample(torch, W, L, seed=5, B=6, n_push=14):
    from lens_b200 import ops, synth
    from lens_b200.pipeline import InferencePipeline, StreamingPipeline
    rng = np.random.default_rng(seed)
    sp = StreamingPipeline(*W, roi=ROI, k=K_POOL, T=T_STEPS, L=L, n_streams=B, n_top=N_TOP)
    frames = synth.frames_device(B, 3 * n_push, roi=ROI, seed=seed)
    cursor = [0] * B
    got = [dict(win=[], S=[], tv=[], ti=[]) for _ in range(B)]
    for k in range(n_push):
        Q = int(rng.integers(1, 4))
        kind = ("none", "subset", "all", "subset", "empty")[k % 5]
        streams = None if kind == "none" else [] if kind == "empty" else rng.permutation(B).tolist() \
            if kind == "all" else rng.choice(B, size=int(rng.integers(1, B)), replace=False).tolist()
        ids = list(range(B)) if streams is None else streams
        win = torch.stack([frames[b, cursor[b]:cursor[b] + Q] for b in ids]) if ids else None
        out = sp.push(frames=win, streams=streams)
        for i, b in enumerate(ids):
            got[b]["win"].append(win[i])
            got[b]["S"].append(out["S"][i])
            got[b]["tv"].append(out["top_val"][i])
            got[b]["ti"].append(out["top_idx"][i])
            cursor[b] += Q
    bp = InferencePipeline(*W, roi=ROI, k=K_POOL, T=T_STEPS, L=L, n_top=N_TOP, max_streams=1)
    ok, nonzero, checked = True, False, 0
    for g in got:
        if not g["win"]:
            continue
        bp.net.reset_states()
        S = bp.similarity(frames=torch.cat(g["win"])[None].contiguous())
        mine = {k: torch.cat(g[k])[None] for k in ("S", "tv", "ti")}
        ok &= torch.equal(mine["S"], S)
        nonzero |= float(S.sum()) > 0
        warm = min(L - 1, S.shape[1])
        ok &= bool((mine["tv"][:, :warm] == float("-inf")).all()) and bool((mine["ti"][:, :warm] == -1).all())
        if S.shape[1] >= L:
            tv, ti, _ = ops.seqmatch_topk(S, L, N_TOP)
            ok &= torch.equal(mine["tv"][:, L - 1:], tv) and torch.equal(mine["ti"][:, L - 1:], ti)
            checked += S.shape[1] - L + 1
    return dict(streams=B, pushes=n_push, valid_rows_checked=checked, bit_exact=bool(ok), nonzero_counts=nonzero)


def kernel_ms(torch, fn, names):
    """Device ms of the kernels whose name contains one of `names`, in one profiled call of fn."""
    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return sum(e.device_time_total for e in prof.key_averages() if any(n in e.key for n in names)) / 1e3


def run_shape(torch, args, name, c):
    from lens_b200 import ops, synth
    from lens_b200.pipeline import StreamingPipeline
    B, P, L = args.streams or c["streams"], c["places"], c["seq_len"]
    Wf, Wo = synth.weights(I_DIMS * I_DIMS, FEATURE, P, seed=1)
    W = (torch.from_numpy(Wf), torch.from_numpy(Wo))
    exact = exactness_sample(torch, W, L)
    torch.cuda.empty_cache()

    rng = np.random.default_rng(11)
    n_frames = 4
    frames = synth.frames_device(B, n_frames, roi=ROI, seed=2)
    pushes = [frames[:, i:i + 1].contiguous() for i in range(n_frames)]
    del frames
    sp = StreamingPipeline(*W, roi=ROI, k=K_POOL, T=T_STEPS, L=L, n_streams=B, n_top=N_TOP)
    lock = lambda i: sp.push(frames=pushes[i % n_frames])   # noqa: E731
    for i in range(max(args.warmup, L)):
        lock(i)
    ms_lock = timed(torch, lock, args.steps)
    S = lock(0)["S"]
    match_lock = lambda i: ops.seqmatch_topk_stream(S, L, N_TOP, sp.ring, sp.seen, sp.t + i)   # noqa: E731
    for i in range(args.warmup):
        match_lock(i)
    ms_match_lock = timed(torch, match_lock, args.steps)

    # the same session goes indexed: every stream in a permuted order
    perm = rng.permutation(B).tolist()
    perm_dev = torch.tensor(perm, device="cuda")
    perm_frames = [p[perm_dev].contiguous() for p in pushes]
    full = lambda i: sp.push(frames=perm_frames[i % n_frames], streams=perm)   # noqa: E731
    for i in range(args.warmup + 1):
        full(i)
    ms_full = timed(torch, full, args.steps)
    ids = perm_dev.int()
    S_perm = full(0)["S"]
    match_ids = lambda i: ops.seqmatch_topk_stream_ids(S_perm, L, N_TOP, ids, sp.ring, sp.seen, sp._rows)  # noqa: E731
    for i in range(args.warmup):
        match_ids(i)
    ms_match_ids = timed(torch, match_ids, args.steps)
    del S, S_perm
    ms_gs = kernel_ms(torch, lambda: full(1), ["state_rows_kernel"])
    ms_full_kernels = kernel_ms(torch, lambda: full(2), ["kernel"])
    gs_bytes = 2 * 2 * B * (I_DIMS * I_DIMS + FEATURE + P) * 4

    subsets = {}
    for label, n in [(lbl, max(1, B // d)) for lbl, d in FRACTIONS] + [("1 camera", 1)]:
        sub = [sorted(rng.choice(B, size=n, replace=False).tolist()) for _ in range(n_frames)]
        sub = [rng.permutation(s).tolist() for s in sub]
        fr = [pushes[i][torch.tensor(s, device="cuda")].contiguous() for i, s in enumerate(sub)]
        push = lambda i: sp.push(frames=fr[i % n_frames], streams=sub[i % n_frames])   # noqa: E731
        for i in range(args.warmup + 1):
            push(i)
        ms = timed(torch, push, args.steps)
        subsets[label] = dict(streams=n, ms=ms, ms_per_stream=ms / n,
                              per_stream_over_lockstep=(ms / n) / (ms_lock / B))
        del fr
    del sp, pushes, perm_frames
    torch.cuda.empty_cache()
    return dict(streams=B, places=P, seq_len=L, queries_per_push=1, exactness_sample=exact,
                lockstep=dict(ms=ms_lock, ms_per_stream=ms_lock / B),
                permuted_all=dict(ms=ms_full, over_lockstep=ms_full / ms_lock),
                subsets=subsets,
                match=dict(lockstep_ms=ms_match_lock, indexed_permuted_ms=ms_match_ids,
                           indexed_over_lockstep=ms_match_ids / ms_match_lock),
                gather_scatter=dict(ms=ms_gs, bytes=gs_bytes, achieved_GBps=gs_bytes / (ms_gs / 1e3) / 1e9 if ms_gs
                                    else None, share_of_push_kernels=ms_gs / ms_full_kernels if ms_full_kernels else None,
                                    share_of_push=ms_gs / ms_full))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--shapes", default="fleet2,fleet3")
    ap.add_argument("--streams", type=int, default=None, help="override the stream count (rehearsals)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_stream_subsets.py needs a CUDA device")
    out = dict(metric="streaming_subset_push", **gpu_info(), roi="80x80", k=K_POOL, timesteps=T_STEPS,
               feature=FEATURE, top_n=N_TOP, steps=args.steps)
    shapes = args.shapes.split(",")
    for s in shapes:
        out[s] = run_shape(torch, args, s, SHAPES[s])
    out["bit_exact"] = all(out[s]["exactness_sample"]["bit_exact"] for s in shapes)
    print(json.dumps(out))
    if not out["bit_exact"]:
        sys.exit(1)


if __name__ == "__main__":
    main()
