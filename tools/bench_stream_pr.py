#!/usr/bin/env python
"""Session precision-recall of live fleets: what track_pr costs StreamingPipeline.push, on one GPU.

    python tools/bench_stream_pr.py [--steps K] [--warmup W] [--shapes fleet2,fleet3,large_map] [--streams B]

Workload and shapes as tools/bench_stream.py (one new window per stream and push).  Reported per shape:
  push_ms           the push end to end (CUDA events over --steps pushes after the warm-up) with tracking off, with
                    each mode alone and with all three
  accumulate        the lens_seqpr_stream_accumulate call alone (CUDA events) for each of those, its GB/s and share of
                    HBM on the bytes it must move: B (L - 1 + Q) P 4 read, plus 2 * 4 B Po of place records (read and
                    written) when the place mode is tracked
  session_ms        session_precision_recall per mode (host clock; the call ends in a device synchronise)
Before timing, a sample of streams is pushed one window at a time through a tracking pipeline of its own, and each
mode's session curve must equal InferencePipeline.precision_recall over the same spike counts ("ok").  One JSON line
on stdout, with the card's name and power limit; nothing is written.
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench import load_peaks   # noqa: E402
from bench_stream import FEATURE, I_DIMS, K_POOL, N_TOP, ROI, SHAPES, T_STEPS, gpu_info, timed   # noqa: E402

MODES = ("place", "query", "multi")
KW = {"place": dict(matching="single", best="place"), "query": dict(matching="single", best="query"),
      "multi": dict(matching="multi")}
TOL = 2


def check_sample(torch, W, L, P, frames, gt, sample):
    """Sampled streams pushed one window at a time with every mode tracked, against the batch method over the
    concatenated spike counts (streams are independent, so the sample is a fleet of its own)."""
    from lens_b200.pipeline import InferencePipeline, StreamingPipeline
    idx = torch.tensor(sample, device=frames.device)
    f, g = frames[idx].contiguous(), gt[idx].contiguous()
    Qc = f.shape[1]
    sp = StreamingPipeline(*W, roi=ROI, k=K_POOL, T=T_STEPS, L=L, n_streams=len(sample), n_top=N_TOP,
                           track_pr=MODES)
    S = torch.cat([sp.push(frames=f[:, q:q + 1].contiguous(), gt_center=g[:, q:q + 1].contiguous(),
                           gt_tol=TOL)["S"] for q in range(Qc)], dim=1)
    bp = InferencePipeline(*W, roi=ROI, k=K_POOL, T=T_STEPS, L=L, n_top=N_TOP, max_streams=len(sample))
    ok = True
    for m in MODES:
        got = sp.session_precision_recall(**KW[m])
        want = bp.precision_recall(S, gt_center=g[:, L - 1:].contiguous(), gt_tol=TOL, **KW[m])
        ok &= all(np.array_equal(np.array(got[k], np.float64), np.array(want[k], np.float64), equal_nan=True)
                  for k in ("P", "R", "tp", "fp")) and got["gtp"] == want["gtp"]
    return dict(streams=len(sample), pushes=Qc, exact=bool(ok), nonzero_counts=bool(float(S.sum()) > 0))


def run_shape(torch, args, peaks, name, c):
    from lens_b200 import ops, synth
    from lens_b200.pipeline import StreamingPipeline
    B, P, L = args.streams or c["streams"], c["places"], c["seq_len"]
    Po, Q = P - L + 1, 1
    Wf, Wo = synth.weights(I_DIMS * I_DIMS, FEATURE, P, seed=1)
    W = (torch.from_numpy(Wf), torch.from_numpy(Wo))
    sample = sorted(set([0, B - 1]) | set(np.random.default_rng(3).choice(B, min(6, B), replace=False).tolist()))
    Qc = L + 2
    gt_all = torch.from_numpy(synth.gt_centers(B, Qc, Po, seed=7)).cuda()
    exact = check_sample(torch, W, L, P, synth.frames_device(B, Qc, roi=ROI, seed=5), gt_all, sample)
    del gt_all
    torch.cuda.empty_cache()

    n_frames = 4
    frames = synth.frames_device(B, n_frames, roi=ROI, seed=2)
    pushes = [frames[:, i:i + 1].contiguous() for i in range(n_frames)]
    del frames
    gt = torch.from_numpy(synth.gt_centers(B, 1, Po, seed=7)).cuda()
    out = dict(streams=B, places=P, seq_len=L, queries_per_push=Q, exactness_sample=exact,
               place_records_bytes=ops.seqpr_stream_bytes(B, P, L, 0), push_ms={}, accumulate={}, session_ms={})
    for track in [(), ("place",), ("query",), ("multi",), MODES]:
        key = "+".join(track) or "off"
        sp = StreamingPipeline(*W, roi=ROI, k=K_POOL, T=T_STEPS, L=L, n_streams=B, n_top=N_TOP, track_pr=track)
        push = lambda i: sp.push(frames=pushes[i % n_frames], gt_center=gt, gt_tol=TOL)   # noqa: E731
        for i in range(max(args.warmup, L)):
            push(i)
        out["push_ms"][key] = timed(torch, push, args.steps)
        if track:
            S = push(0)["S"]
            accs = {"acc_" + m: a for m, a in sp._pr_acc.items()}
            acc = lambda i: ops.seqpr_stream_accumulate(S, L, sp.ring, sp.seen, sp.t, gt, TOL, **accs)   # noqa: E731
            for i in range(args.warmup):
                acc(i)
            ms = timed(torch, acc, args.steps)
            nbytes = 4.0 * B * (L - 1 + Q) * P + (2 * 4.0 * B * Po if "place" in track else 0.0)
            gbs = nbytes / (ms / 1e3) / 1e9
            out["accumulate"][key] = dict(ms=ms, bytes=int(nbytes), achieved_GBps=gbs,
                                          frac_of_hbm_peak=gbs / peaks["hbm_gbs"])
            del S
        if track == MODES:
            for m in MODES:
                sp.session_precision_recall(**KW[m])
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for _ in range(args.steps):
                    sp.session_precision_recall(**KW[m])
                out["session_ms"][m] = (time.perf_counter() - t0) * 1e3 / args.steps
        del sp
        torch.cuda.empty_cache()
    out["tracking_all_over_off"] = out["push_ms"]["+".join(MODES)] / out["push_ms"]["off"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--shapes", default="fleet2,fleet3,large_map")
    ap.add_argument("--streams", type=int, default=None, help="override the stream count (rehearsals)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_stream_pr.py needs a CUDA device")
    peaks = load_peaks()
    out = dict(metric="streaming_session_pr", **gpu_info(), peaks_source=peaks["source"],
               hbm_peak_GBps=peaks["hbm_gbs"], roi="80x80", k=K_POOL, timesteps=T_STEPS, feature=FEATURE,
               top_n=N_TOP, gt_tol=TOL, steps=args.steps)
    for s in args.shapes.split(","):
        out[s] = run_shape(torch, args, peaks, s, SHAPES[s])
    out["ok"] = all(out[s]["exactness_sample"]["exact"] for s in args.shapes.split(","))
    print(json.dumps(out))
    if not out["ok"]:
        sys.exit(1)


if __name__ == "__main__":
    main()
