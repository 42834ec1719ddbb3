#!/usr/bin/env python
"""Raw DVS event streams -> Recall@N on one GPU: the BASELINE config-2 and config-3 shapes fed from events.

    python tools/bench_events.py [--steps K] [--warmup W] [--shapes 2,3] [--group-streams G]

Workload: LENS I=100 -> F=200 -> P, random-init weights with trained statistics (synth.weights), T=250,
80x80 roi cropped at (23, 0) from the 128x128 sensor, k=8; synthetic Speck-density streams
(synth.event_streams_device: 250 ms windows of ~131 072 events, 8 per sensor pixel).
  config 2: 1 000 streams x 16 queries, P = 1 000, L = 2; all events resident (~2.1e9), one step_events call.
  config 3: 65 536 streams x 10 queries, P = 10 000, L = 10 via step_event_groups: the fleet's ~8.6e10
            events do not fit in HBM, so groups of --group-streams streams are fed from --buffers distinct
            device event buffers (generated before timing) used in turn.
Reported per shape: the events step (ms, events/s, query timesteps/s), the binning call alone (CUDA events;
GB/s on the streamed bytes, 4 B/event of x / y + I B per window, and its share of HBM peak), and in the same
run step(pooled=...) and step(frames=...) on what the binning produced, so the events path's cost over them
is the difference.  Before timing, a sample of streams is checked bit for bit: the step's spike counts and
window event counts against run_streams on per-stream ops.bin_events output.  One JSON line on stdout.
Everything stays on the device; nothing is written.
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
ROI_X0, ROI_Y0, WINDOW_US, EVENTS_PER_WINDOW = 23, 0, 250_000, 131_072
SHAPES = {2: dict(streams=1000, queries=16, places=1000, seq_len=2),
          3: dict(streams=65536, queries=10, places=10000, seq_len=10)}


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
    for _ in range(steps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record()
        evs.append((a, b))
    torch.cuda.synchronize()
    return float(np.mean([a.elapsed_time(b) for a, b in evs]))


def check_sample(torch, Wf, Wo, S, n_ev, stream_events, sample, Q):
    """S / n_ev rows of `sample` (from the first step of a fresh pipeline) against a fresh network run on
    per-stream ops.bin_events output.  stream_events(b) -> (t, x, y, t0) of stream b (aligned copies)."""
    from lens_b200 import ops
    from lens_b200.network import B200Network
    pooled, counts = [], []
    for b in sample:
        t, x, y, t0 = stream_events(b)
        _, p, c = ops.bin_events(t, x, y, t0, WINDOW_US, Q, ROI, K_POOL, roi_x0=ROI_X0, roi_y0=ROI_Y0,
                                 want_frames=False)
        pooled.append(p); counts.append(c)
    net = B200Network(torch.from_numpy(Wf), torch.from_numpy(Wo), roi=ROI, k=K_POOL, num_timesteps=T_STEPS,
                      max_streams=len(sample))
    S_ref = net.run_streams(pooled=torch.stack(pooled))
    idx = torch.tensor(sample, device=S.device)
    ok = torch.equal(S[idx], S_ref) and torch.equal(n_ev[idx], torch.stack(counts))
    return dict(streams=len(sample), bit_exact=bool(ok), nonzero_counts=bool(float(S_ref.sum()) > 0))


def shape_result(c, B, Q, n_events, ms_step, ms_bin, ms_pooled, ms_frames, peaks):
    I = I_DIMS * I_DIMS
    streamed = 4.0 * n_events + I * B * Q
    gbs = streamed / (ms_bin / 1e3) / 1e9
    return dict(streams=B, queries=Q, places=c["places"], seq_len=c["seq_len"], events_per_step=int(n_events),
                step_events=dict(ms=ms_step, events_per_s=n_events / (ms_step / 1e3),
                                 query_timesteps_per_s=B * Q * T_STEPS / (ms_step / 1e3)),
                binning=dict(ms=ms_bin, streamed_bytes=int(streamed), achieved_GBps=gbs, hbm_peak_GBps=peaks["hbm_gbs"],
                             frac_of_hbm_peak=gbs / peaks["hbm_gbs"], kernel="bin_kernel (80x80 crop)",
                             bytes="4 B/event (x, y) + I B per window (pooled)"),
                step_pooled=dict(ms=ms_pooled, query_timesteps_per_s=B * Q * T_STEPS / (ms_pooled / 1e3)),
                step_frames=dict(ms=ms_frames, query_timesteps_per_s=B * Q * T_STEPS / (ms_frames / 1e3)),
                events_cost_over_pooled_ms=ms_step - ms_pooled, events_cost_over_frames_ms=ms_step - ms_frames)


def run_config2(torch, args, peaks, c):
    from lens_b200 import ops, synth
    from lens_b200.pipeline import InferencePipeline
    B, Q, P, L = args.streams or c["streams"], c["queries"], c["places"], c["seq_len"]
    I = I_DIMS * I_DIMS
    Wf, Wo = synth.weights(I, FEATURE, P, seed=1)
    t, x, y, off, t0 = synth.event_streams_device(B, Q, WINDOW_US, EVENTS_PER_WINDOW, seed=11)
    n = t.numel()
    gt = torch.from_numpy(synth.gt_centers(B, Q - L + 1, P - L + 1, seed=7)).cuda()
    pipe = InferencePipeline(torch.from_numpy(Wf), torch.from_numpy(Wo), roi=ROI, k=K_POOL, T=T_STEPS, L=L,
                             n_top=N_TOP, max_streams=B)
    step = lambda: pipe.step_events(t, x, y, off, t0, WINDOW_US, Q, roi_x0=ROI_X0, roi_y0=ROI_Y0,  # noqa: E731
                                    gt_center=gt, gt_tol=2)
    first = step()
    oh, t0h = off.cpu().numpy(), t0.cpu().numpy()

    def stream_events(b):
        s = slice(int(oh[b]), int(oh[b + 1]))
        return t[s].clone(), x[s].clone(), y[s].clone(), int(t0h[b])
    sample = sorted(np.random.default_rng(3).choice(B, size=min(8, B), replace=False).tolist())
    exact = check_sample(torch, Wf, Wo, first["S"], first["events_per_window"], stream_events, sample, Q)
    del first
    binning = lambda: ops.bin_event_streams(t, x, y, off, t0, WINDOW_US, Q, ROI, K_POOL,  # noqa: E731
                                            roi_x0=ROI_X0, roi_y0=ROI_Y0)
    frames, pooled, _ = ops.bin_event_streams(t, x, y, off, t0, WINDOW_US, Q, ROI, K_POOL, roi_x0=ROI_X0,
                                              roi_y0=ROI_Y0, want_frames=True)
    for _ in range(args.warmup):
        step(); binning(); pipe.step(pooled=pooled, gt_center=gt, gt_tol=2); pipe.step(frames=frames, gt_center=gt,
                                                                                      gt_tol=2)
    ms_step = timed(torch, step, args.steps)
    ms_bin = timed(torch, binning, args.steps)
    ms_pooled = timed(torch, lambda: pipe.step(pooled=pooled, gt_center=gt, gt_tol=2), args.steps)
    ms_frames = timed(torch, lambda: pipe.step(frames=frames, gt_center=gt, gt_tol=2), args.steps)
    res = shape_result(c, B, Q, n, ms_step, ms_bin, ms_pooled, ms_frames, peaks)
    res["exactness_sample"] = exact
    del pipe, t, x, y, off, t0, frames, pooled
    torch.cuda.empty_cache()
    return res


def run_config3(torch, args, peaks, c):
    from lens_b200 import ops, synth
    from lens_b200.pipeline import InferencePipeline
    B, Q, P, L = args.streams or c["streams"], c["queries"], c["places"], c["seq_len"]
    G = min(args.group_streams, B)
    assert G % 2 == 0 and B % G == 0, "--group-streams must be even and divide the stream count"
    I = I_DIMS * I_DIMS
    Wf, Wo = synth.weights(I, FEATURE, P, seed=1)
    bufs = [synth.event_streams_device(G, Q, WINDOW_US, EVENTS_PER_WINDOW, seed=31 + i) for i in range(args.buffers)]
    n_groups = B // G
    n = sum(bufs[g % len(bufs)][0].numel() for g in range(n_groups))
    gt = torch.from_numpy(synth.gt_centers(B, Q - L + 1, P - L + 1, seed=7)).cuda()
    pipe = InferencePipeline(torch.from_numpy(Wf), torch.from_numpy(Wo), roi=ROI, k=K_POOL, T=T_STEPS, L=L,
                             n_top=N_TOP, max_streams=B)

    def groups():
        for g in range(n_groups):
            t, x, y, off, t0 = bufs[g % len(bufs)]
            yield g * G, t, x, y, off, t0
    step = lambda: pipe.step_event_groups(groups(), B, Q, WINDOW_US, roi_x0=ROI_X0, roi_y0=ROI_Y0,  # noqa: E731
                                          gt_center=gt, gt_tol=2)
    first = step()
    host = [(off.cpu().numpy(), t0.cpu().numpy()) for _, _, _, off, t0 in bufs]

    def stream_events(b):
        i = (b // G) % len(bufs)
        t, x, y = bufs[i][:3]
        oh, t0h = host[i]
        s = slice(int(oh[b % G]), int(oh[b % G + 1]))
        return t[s].clone(), x[s].clone(), y[s].clone(), int(t0h[b % G])
    sample = sorted(set([0, 1, G - 1, G, B - 1]) | set(np.random.default_rng(3).choice(B, 3, replace=False).tolist()))
    exact = check_sample(torch, Wf, Wo, first["S"], first["events_per_window"], stream_events, sample, Q)
    del first

    def binning():
        for _, t, x, y, off, t0 in groups():
            ops.bin_event_streams(t, x, y, off, t0, WINDOW_US, Q, ROI, K_POOL, roi_x0=ROI_X0, roi_y0=ROI_Y0)
    binned = [ops.bin_event_streams(t, x, y, off, t0, WINDOW_US, Q, ROI, K_POOL, roi_x0=ROI_X0, roi_y0=ROI_Y0,
                                    want_frames=True)[:2] for t, x, y, off, t0 in bufs]
    frames = torch.cat([binned[g % len(bufs)][0] for g in range(n_groups)])
    pooled = torch.cat([binned[g % len(bufs)][1] for g in range(n_groups)])
    del binned
    for _ in range(args.warmup):
        step(); binning()
    pipe.step(pooled=pooled, gt_center=gt, gt_tol=2); pipe.step(frames=frames, gt_center=gt, gt_tol=2)
    ms_step = timed(torch, step, args.steps)
    ms_bin = timed(torch, binning, args.steps)
    ms_pooled = timed(torch, lambda: pipe.step(pooled=pooled, gt_center=gt, gt_tol=2), args.steps)
    ms_frames = timed(torch, lambda: pipe.step(frames=frames, gt_center=gt, gt_tol=2), args.steps)
    res = shape_result(c, B, Q, n, ms_step, ms_bin, ms_pooled, ms_frames, peaks)
    res.update(exactness_sample=exact, group_streams=G, groups_per_step=n_groups, event_buffers=len(bufs),
               recycling="group g reads event buffer g %% %d (%d distinct buffers of %d streams, generated before "
                         "timing)" % (len(bufs), len(bufs), G))
    del pipe, bufs, frames, pooled
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--shapes", default="2,3", help="which BASELINE shapes to run (2, 3)")
    ap.add_argument("--streams", type=int, default=None, help="override the stream count (rehearsals)")
    ap.add_argument("--group-streams", type=int, default=2048, help="config 3: streams per step_event_groups group")
    ap.add_argument("--buffers", type=int, default=2, help="config 3: distinct device event buffers")
    args = ap.parse_args()
    if args.steps < 1 or args.buffers < 2:
        ap.error("--steps must be >= 1 and --buffers >= 2")
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_events.py needs a CUDA device")
    peaks = load_peaks()
    out = dict(metric="events_to_recall", **gpu_info(), peaks_source=peaks["source"], hbm_peak_GBps=peaks["hbm_gbs"],
               roi="80x80 at (23, 0) of 128x128", k=K_POOL, timesteps=T_STEPS, feature=FEATURE,
               window_us=WINDOW_US, events_per_window=EVENTS_PER_WINDOW, steps=args.steps)
    for s in (int(v) for v in args.shapes.split(",")):
        out["config%d" % s] = (run_config2 if s == 2 else run_config3)(torch, args, peaks, SHAPES[s])
    out["bit_exact"] = all(out[k]["exactness_sample"]["bit_exact"] for k in out if k.startswith("config"))
    print(json.dumps(out))
    if not out["bit_exact"]:
        sys.exit(1)


if __name__ == "__main__":
    main()
