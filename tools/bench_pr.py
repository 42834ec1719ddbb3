#!/usr/bin/env python
"""Fleet precision-recall: InferencePipeline.precision_recall's two passes on the spike counts of a real step.

    python tools/bench_pr.py [--steps K] [--warmup W] [--shapes fleet3,large_map] [--streams B] [--n-thresh N]

Workload: LENS I=100 -> F=200 -> P, random-init weights with trained statistics (synth.weights), T=250, count
frames of the 80x80 roi (synth.frames_device), k=8, band ground truth (synth.gt_centers, tolerance 2).
  fleet3     65 536 streams, P = 10 000,  Q = 10,  L = 10 (BASELINE config 3: S is 26.2 GB, Qo = 1)
  large_map      1 stream,   P = 100 000, Q = 300, L = 10 (one camera against a large map)
One step produces S; on that S every mode (per place, per query, multi) is timed pass by pass with CUDA events
over --steps calls after --warmup, and so is K4 (ops.seqmatch_topk, top-25) for comparison.  Bytes counted per
pass: S once (B Q P 4), the band centres, the records written (scan) or read (count), and the per-query records'
second read by the extremes kernel; the shared-memory tables and the 16 B per threshold of histogram are not
counted.  Checked in the same run: tp[-1] + fp[-1] = the number of columns (entries in multi mode); in per-query
mode the maximum of the records equals the maximum of K4's top-1 values; and 4 sampled streams against the oracle
(O.create_pr over the concatenation of O.seqmatch).  One JSON line on stdout; nothing is written.
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bench import load_peaks   # noqa: E402  (MEASURED_PEAKS.json, else the fallback figures)
from bench_stream import gpu_info, timed   # noqa: E402  (same directory)

I_DIMS, FEATURE, ROI, K_POOL, T_STEPS, N_TOP, TOL = 10, 200, 80, 8, 250, 25, 2
SHAPES = {"fleet3": dict(streams=65536, places=10000, queries=10, seq_len=10),
          "large_map": dict(streams=1, places=100000, queries=300, seq_len=10)}
MODES = {"place": ("single", "place"), "query": ("single", "query"), "multi": ("multi", None)}


def key_to_float(k):
    """Inverse of the kernels' order-preserving float key (f32_orderable)."""
    u = int(k) & 0xffffffff
    bits = (u & 0x7fffffff) if u & 0x80000000 else (~u & 0xffffffff)
    return float(np.array([bits], np.uint32).view(np.float32)[0])


def oracle_sample(torch, pipe, S, gt, L, sample, n_thresh):
    """precision_recall on the sampled streams alone == O.create_pr over their concatenated matrices."""
    from oracle import oracle as O
    idx = torch.tensor(sample, device=S.device)
    Ss, gs = S[idx].contiguous(), gt[idx].contiguous()
    Sh, gh = Ss.cpu().numpy(), gs.cpu().numpy()
    B, Q, P = Sh.shape
    Po, Qo = P - L + 1, Q - L + 1
    Ds = [O.seqmatch(Sh[b], L) for b in range(B)]
    p = np.arange(Po)[:, None]
    Gs = [(gh[b][None, :] >= 0) & (np.abs(p - gh[b][None, :]) <= TOL) for b in range(B)]
    ok = {}
    for name, (matching, best) in MODES.items():
        got = pipe.precision_recall(Ss, gt_center=gs, gt_tol=TOL, matching=matching, best=best, n_thresh=n_thresh)
        if best == "place":
            M, G = np.concatenate([D.T for D in Ds], axis=1), np.concatenate([g.T for g in Gs], axis=1)
        else:
            M, G = np.concatenate(Ds, axis=1), np.concatenate(Gs, axis=1)
        Pw, Rw = O.create_pr(M, G, n_thresh=n_thresh, matching=matching)
        ok[name] = bool(np.array_equal(np.array(got["P"], np.float64), np.array(Pw, np.float64), equal_nan=True)
                        and np.array_equal(np.array(got["R"], np.float64), np.array(Rw, np.float64), equal_nan=True))
    return dict(streams=sample, equal=ok)


def run_shape(torch, args, peaks, c):
    from lens_b200 import ops, synth
    from lens_b200.pipeline import InferencePipeline
    B, P, Q, L = args.streams or c["streams"], c["places"], c["queries"], c["seq_len"]
    Po, Qo, n = P - L + 1, Q - L + 1, args.n_thresh
    Wf, Wo = synth.weights(I_DIMS * I_DIMS, FEATURE, P, seed=1)
    pipe = InferencePipeline(torch.from_numpy(Wf), torch.from_numpy(Wo), roi=ROI, k=K_POOL, T=T_STEPS, L=L,
                             n_top=N_TOP, max_streams=B)
    frames = synth.frames_device(B, Q, roi=ROI, seed=2)
    gt = torch.from_numpy(synth.gt_centers(B, Qo, Po, seed=7)).cuda()
    pipe.step(frames=frames)
    ms_step = timed(torch, lambda i: pipe.step(frames=frames), 1)
    S = pipe.step(frames=frames)["S"]
    del frames
    torch.cuda.empty_cache()
    peak = peaks["hbm_gbs"]

    def rate(nbytes, ms):
        gbs = nbytes / (ms / 1e3) / 1e9
        return dict(ms=ms, bytes=int(nbytes), achieved_GBps=gbs, frac_of_hbm_peak=gbs / peak)

    s_bytes, gt_bytes = 4.0 * B * Q * P, 4.0 * B * Qo
    rec_bytes = {"place": 5.0 * B * Po, "query": 9.0 * B * Qo, "multi": 0.0}
    scan_bytes = {"place": s_bytes + gt_bytes + rec_bytes["place"],
                  "query": s_bytes + gt_bytes + 2 * rec_bytes["query"] + rec_bytes["query"],   # memset, atomics, read
                  "multi": s_bytes + gt_bytes}
    count_bytes = {"place": rec_bytes["place"], "query": 8.0 * B * Qo + gt_bytes, "multi": s_bytes + gt_bytes}
    n_cols = {"place": B * Po, "query": B * Qo, "multi": B * Po * Qo}
    out = dict(streams=B, places=P, queries=Q, seq_len=L, n_thresh=n, S_bytes=int(s_bytes), step_ms=ms_step,
               modes={}, invariants={})
    gtk = dict(gt_center=gt, gt_tol=TOL)
    for name, (matching, best) in MODES.items():
        m = ops.seqpr_mode(matching, best)
        scan = lambda i: ops.seqpr_scan(S, L, m, **gtk)        # noqa: E731
        for i in range(args.warmup):
            scan(i)
        ms_scan = timed(torch, scan, args.steps)
        records, ext, gtp = scan(0)
        count = lambda i: ops.seqpr_counts(S, L, m, records, ext, n, **gtk)     # noqa: E731
        for i in range(args.warmup):
            count(i)
        ms_count = timed(torch, count, args.steps)
        tp, fp = count(0)
        total = int(tp[-1].item() + fp[-1].item())
        out["invariants"][name] = dict(last_threshold_counts=total, columns=n_cols[name], ok=total == n_cols[name])
        out["modes"][name] = dict(ms=ms_scan + ms_count, frac_of_step=(ms_scan + ms_count) / ms_step,
                                  records_bytes=int(rec_bytes[name]),
                                  scan=rate(scan_bytes[name], ms_scan), count=rate(count_bytes[name], ms_count))
        if name == "query":
            rec_max = key_to_float(ext[0].item())
            k4_max = float(ops.seqmatch_topk(S, L, 1)[0].max().item())
            out["invariants"]["query_max_equals_k4_top1"] = dict(records=rec_max, k4=k4_max, ok=rec_max == k4_max)
        del records, ext, gtp, tp, fp
        torch.cuda.empty_cache()
    k4 = lambda i: ops.seqmatch_topk(S, L, N_TOP)     # noqa: E731
    for i in range(args.warmup):
        k4(i)
    out["seqmatch_topk"] = rate(s_bytes + 8.0 * B * Qo * N_TOP, timed(torch, k4, args.steps))
    sample = sorted(set([0, B - 1]) | set(np.random.default_rng(3).choice(B, min(4, B), replace=False).tolist()))[:4]
    out["oracle_sample"] = oracle_sample(torch, pipe, S, gt, L, sample, n)
    out["ok"] = all(v["ok"] for v in out["invariants"].values()) and all(out["oracle_sample"]["equal"].values())
    del pipe, S
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--shapes", default="fleet3,large_map")
    ap.add_argument("--streams", type=int, default=None, help="override the stream count (rehearsals)")
    ap.add_argument("--n-thresh", type=int, default=100)
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_pr.py needs a CUDA device")
    peaks = load_peaks()
    out = dict(metric="fleet_pr", **gpu_info(), peaks_source=peaks["source"], hbm_peak_GBps=peaks["hbm_gbs"],
               roi="80x80", k=K_POOL, timesteps=T_STEPS, feature=FEATURE, gt_tol=TOL, steps=args.steps)
    for s in args.shapes.split(","):
        out[s] = run_shape(torch, args, peaks, SHAPES[s])
    out["ok"] = all(out[s]["ok"] for s in args.shapes.split(","))
    print(json.dumps(out))
    if not out["ok"]:
        sys.exit(1)


if __name__ == "__main__":
    main()
