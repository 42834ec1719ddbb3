#!/usr/bin/env python
"""Live fleets: StreamingPipeline.push with one new query window per stream and push, on one GPU.

    python tools/bench_stream.py [--steps K] [--warmup W] [--shapes fleet2,fleet3,large_map] [--streams B]

Workload: LENS I=100 -> F=200 -> P, random-init weights with trained statistics (synth.weights), T=250, count
frames of the 80x80 roi (synth.frames_device), k=8, top-25.
  fleet2     1 000 streams,  P = 1 000,   L = 2,  Q = 1 per push (the BASELINE config-2 fleet, live)
  fleet3    65 536 streams,  P = 10 000,  L = 10, Q = 1 per push (config 3, live: ring of 23.6 GB)
  large_map      1 stream,   P = 100 000, L = 10, Q = 1 per push (one camera, large map: segmented matching)
Reported per shape and push: the push end to end (CUDA events over --steps pushes after --warmup), the
lens_seqmatch_topk_stream call alone (CUDA events), that call's GB/s and share of HBM on the bytes it must move
(B (L - 1 + Q) P 4 read, the min(Q, L - 1) appended rows read and written, B Q N 8 for the top-N), and, for
comparison, ms per query of a batch step(frames=...) of --batch-queries windows with the same model.  The fleet2
ring (4 MB) and S rows fit in L2; the fleet3 ring does not.
Before timing, a sample of streams is checked bit for bit: a fresh pipeline pushes L + 2 windows one at a time, and
its spike counts and valid top-N rows must equal a batch step over the same windows.  One JSON line on stdout;
nothing is written.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bench import load_peaks   # noqa: E402  (MEASURED_PEAKS.json, else the fallback figures)

I_DIMS, FEATURE, ROI, K_POOL, T_STEPS, N_TOP = 10, 200, 80, 8, 250, 25
SHAPES = {"fleet2": dict(streams=1000, places=1000, seq_len=2, batch_queries=16),
          "fleet3": dict(streams=65536, places=10000, seq_len=10, batch_queries=10),
          "large_map": dict(streams=1, places=100000, seq_len=10, batch_queries=16)}


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        name, power = (s.strip() for s in r.stdout.strip().splitlines()[0].split(","))
        return dict(gpu=name, power_limit=power)
    except (OSError, IndexError, ValueError, subprocess.SubprocessError):
        return dict(gpu=None, power_limit=None)


def timed(torch, fn, steps):
    """ms per call from CUDA events on the current stream (synchronised at the end)."""
    evs = []
    for i in range(steps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(i); b.record()
        evs.append((a, b))
    torch.cuda.synchronize()
    return float(np.mean([a.elapsed_time(b) for a, b in evs]))


def check_sample(torch, W, L, frames, sample):
    """Push frames [B, L + 2, ...] one window at a time through a fresh pipeline over all B streams; the sampled
    streams' S and valid rows must equal a batch step over the same windows (streams are independent, so the
    batch runs on the sample only)."""
    from lens_b200.pipeline import InferencePipeline, StreamingPipeline
    B, Qc = frames.shape[:2]
    sp = StreamingPipeline(*W, roi=ROI, k=K_POOL, T=T_STEPS, L=L, n_streams=B, n_top=N_TOP)
    idx = torch.tensor(sample, device=frames.device)
    rows = []
    for q in range(Qc):
        r = sp.push(frames=frames[:, q:q + 1].contiguous())
        rows.append({k: r[k][idx] for k in ("S", "top_val", "top_idx")})
    got = {k: torch.cat([r[k] for r in rows], dim=1) for k in ("S", "top_val", "top_idx")}
    del sp, rows, r
    bp = InferencePipeline(*W, roi=ROI, k=K_POOL, T=T_STEPS, L=L, n_top=N_TOP, max_streams=len(sample))
    want = bp.step(frames=frames[idx].contiguous())
    ok = (torch.equal(got["S"], want["S"]) and torch.equal(got["top_val"][:, L - 1:], want["top_val"])
          and torch.equal(got["top_idx"][:, L - 1:], want["top_idx"])
          and bool((got["top_idx"][:, :L - 1] == -1).all()))
    return dict(streams=len(sample), pushes=Qc, bit_exact=bool(ok), nonzero_counts=bool(float(want["S"].sum()) > 0))


def run_shape(torch, args, peaks, name, c):
    from lens_b200 import ops, synth
    from lens_b200.pipeline import InferencePipeline, StreamingPipeline
    B, P, L, Qb = args.streams or c["streams"], c["places"], c["seq_len"], c["batch_queries"]
    Wf, Wo = synth.weights(I_DIMS * I_DIMS, FEATURE, P, seed=1)
    W = (torch.from_numpy(Wf), torch.from_numpy(Wo))
    sample = sorted(set([0, B - 1]) | set(np.random.default_rng(3).choice(B, min(6, B), replace=False).tolist()))
    exact = check_sample(torch, W, L, synth.frames_device(B, L + 2, roi=ROI, seed=5), sample)
    torch.cuda.empty_cache()

    # the timed session: a distinct frame per push (n_frames of them, reused in turn), all rows past warm-up
    n_frames = 4
    frames = synth.frames_device(B, n_frames, roi=ROI, seed=2)
    pushes = [frames[:, i:i + 1].contiguous() for i in range(n_frames)]
    del frames
    sp = StreamingPipeline(*W, roi=ROI, k=K_POOL, T=T_STEPS, L=L, n_streams=B, n_top=N_TOP)
    gt = torch.from_numpy(synth.gt_centers(B, 1, P - L + 1, seed=7)).cuda()
    push = lambda i: sp.push(frames=pushes[i % n_frames], gt_center=gt, gt_tol=2)   # noqa: E731
    for i in range(max(args.warmup, L)):
        push(i)
    ms_push = timed(torch, push, args.steps)
    S = push(0)["S"]
    match = lambda i: ops.seqmatch_topk_stream(S, L, N_TOP, sp.ring, sp.seen, sp.t + i)   # noqa: E731
    for i in range(args.warmup):
        match(i)
    ms_match = timed(torch, match, args.steps)
    del sp, S, pushes
    torch.cuda.empty_cache()

    bframes = synth.frames_device(B, Qb, roi=ROI, seed=4)
    bp = InferencePipeline(*W, roi=ROI, k=K_POOL, T=T_STEPS, L=L, n_top=N_TOP, max_streams=B)
    bgt = torch.from_numpy(synth.gt_centers(B, Qb - L + 1, P - L + 1, seed=7)).cuda()
    step = lambda i: bp.step(frames=bframes, gt_center=bgt, gt_tol=2)   # noqa: E731
    for i in range(args.warmup):
        step(i)
    ms_step = timed(torch, step, max(1, min(args.steps, args.batch_steps)))
    del bp, bframes
    torch.cuda.empty_cache()

    Q = 1
    n_app = min(Q, L - 1)
    bytes_match = 4.0 * B * (L - 1 + Q) * P + 2 * 4.0 * B * n_app * P + 8.0 * B * Q * N_TOP
    gbs = bytes_match / (ms_match / 1e3) / 1e9
    return dict(streams=B, places=P, seq_len=L, queries_per_push=Q, ring_bytes=4 * B * max(L - 1, 0) * P,
                exactness_sample=exact,
                push=dict(ms=ms_push, query_timesteps_per_s=B * Q * T_STEPS / (ms_push / 1e3)),
                seqmatch_topk_stream=dict(ms=ms_match, bytes=int(bytes_match), achieved_GBps=gbs,
                                          hbm_peak_GBps=peaks["hbm_gbs"], frac_of_hbm_peak=gbs / peaks["hbm_gbs"],
                                          bytes_counted="B(L-1+Q)P*4 read + appended rows read and written + "
                                                        "B*Q*N*8 top-N"),
                batch_step=dict(queries=Qb, ms=ms_step, ms_per_query=ms_step / Qb,
                                query_timesteps_per_s=B * Qb * T_STEPS / (ms_step / 1e3)),
                push_over_batch_per_query=ms_push / (ms_step / Qb))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--batch-steps", type=int, default=3, help="timed batch steps (capped by --steps)")
    ap.add_argument("--shapes", default="fleet2,fleet3,large_map")
    ap.add_argument("--streams", type=int, default=None, help="override the stream count (rehearsals)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_stream.py needs a CUDA device")
    peaks = load_peaks()
    out = dict(metric="streaming_push", **gpu_info(), peaks_source=peaks["source"], hbm_peak_GBps=peaks["hbm_gbs"],
               roi="80x80", k=K_POOL, timesteps=T_STEPS, feature=FEATURE, top_n=N_TOP, steps=args.steps)
    for s in args.shapes.split(","):
        out[s] = run_shape(torch, args, peaks, s, SHAPES[s])
    out["bit_exact"] = all(out[s]["exactness_sample"]["bit_exact"] for s in args.shapes.split(","))
    print(json.dumps(out))
    if not out["bit_exact"]:
        sys.exit(1)


if __name__ == "__main__":
    main()
