#!/usr/bin/env python
"""Benchmark of the LENS inference hot path on B200 (contract: see DESIGN.md "Measurement").

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # CPU arm (oracle port, host cores)
    python bench.py --config {1,2,3,4,5} ...                 # pick the BASELINE.json configuration
    python bench.py ... --dump-outputs DIR                   # also save the main line's last timed step (.npy)

Default workload = BASELINE.json configs[2] ("config3", the largest single-GPU configuration):
LENS architecture I=100 -> F=200 -> P=10 000 places, random-init weights with trained statistics,
65 536 query streams IN TOTAL (strong scaling: 65 536 / N per GPU) of 10 queries x T=250 timesteps,
sequence length 10, synthetic Speck-resolution count frames.  A step = one pass of the hot path over
the whole batch:
    u8 frames [B,Q,80,80] -> pooling -> SNN (feature + output layers) -> spike counts
    -> diagonal sequence matching + top-25 -> Recall@N counters (all-reduced when N > 1).
`value`     : query timesteps / s with the frames already resident in HBM.
`e2e`       : the same through the public API with HOST (pinned) frames: H2D of the frames and D2H
              of the recall counters + top-N indices inside the timed region.
`roofline`  : the dominant kernel (output-layer contraction); `rooflines` lists every kernel of the
              path (K1 binning, K2 hidden layer, K3 output layer, K4 matching).
`extras`    : the other configurations measured in the same run (bounded): config 1 latency (one
              stream, serial chain), config 2, config 4 (1e9 events / N per GPU, window-aligned
              shards), config 5 (P=100 000, W_out row shards all-gathered over NCCL, top-N gathered).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

I_DIMS, ROI, K_POOL, T_STEPS = 10, 80, 8, 250
N_TOP, NS = 25, (1, 5, 10, 15, 20, 25)
FEATURE = 200

# BASELINE.json configs[k-1]; streams are per GPU for weak scaling and in total for strong scaling
CONFIGS = {
    1: dict(name="config1", places=100, streams=1, queries=100, seq_len=2, scaling="replicas",
            what="bundled-model shape, one stream of 100 queries (serial 25 000-step chain)"),
    2: dict(name="config2", places=1000, streams=1000, queries=16, seq_len=2, scaling="weak",
            what="1k places x 1k query streams per GPU"),
    3: dict(name="config3", places=10000, streams=65536, queries=10, seq_len=10, scaling="strong",
            what="10k-place database, 64k batched query streams in total, sequence length 10"),
    4: dict(name="config4", events=1_000_000_000, scaling="strong",
            what="1e9 DVS events at 128x128 into frames, window-aligned shards"),
    5: dict(name="config5", places=100000, streams=1024, queries=10, seq_len=10, scaling="weak",
            what="100k-place database arriving as row shards (NCCL all-gather), 1 024 query streams per GPU"),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=3, choices=sorted(CONFIGS))
    ap.add_argument("--streams", type=int, default=None, help="override: query streams (see CONFIGS)")
    ap.add_argument("--queries", type=int, default=None, help="override: queries per stream")
    ap.add_argument("--places", type=int, default=None, help="override: database places")
    ap.add_argument("--seq-len", type=int, default=None)
    ap.add_argument("--mode", type=int, default=0, help="0 auto, 1 CUDA-core, 2 tensor-core output layer")
    ap.add_argument("--events", type=int, default=None, help="override: total events of the binning measurement")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="main configuration only")
    ap.add_argument("--extras", default="1,2,4,5", help="configurations measured beside the main one")
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the main line's last timed step returned as DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200 (the reference arm times a bounded sample on the host)")
    return args


def resolve(args, config=None, world=1):
    """Configuration dict with overrides applied and the per-GPU stream count filled in."""
    c = dict(CONFIGS[config if config is not None else args.config])
    if config is None or config == args.config:
        for k, a in (("streams", args.streams), ("queries", args.queries), ("places", args.places),
                     ("seq_len", args.seq_len), ("events", args.events)):
            if a is not None and k in c:
                c[k] = a
        c["overridden"] = any(a is not None for a in (args.streams, args.queries, args.places, args.seq_len,
                                                      args.events))
    if "streams" in c:
        if c["scaling"] == "strong":
            c["streams_per_gpu"] = max(2, c["streams"] // world)
            c["streams_total"] = c["streams_per_gpu"] * world
        else:
            c["streams_per_gpu"] = c["streams"]
            c["streams_total"] = c["streams"] * world
    return c


def workload_config(c, world):
    if "events" in c and "places" not in c:
        return dict(workload="%s: %s; %d events in total, 250 ms windows, 128x128 sensor, %d events per GPU" %
                             (c["name"], c["what"], c["events"], c["events"] // world),
                    events_total=c["events"], parallelism="window-sharded x%d" % world,
                    l2="inputs (8 B/event) far larger than L2")
    label = c["name"] + (" (overridden sizes)" if c.get("overridden") else "")
    return dict(workload="%s: %s; LENS I=100 F=%d P=%d random-init (trained statistics), %d streams/GPU x %d "
                         "queries x T=%d, L=%d, synthetic 80x80 Speck count frames" %
                         (label, c["what"], FEATURE, c["places"], c["streams_per_gpu"], c["queries"], T_STEPS,
                          c["seq_len"]),
                streams_per_gpu=c["streams_per_gpu"], streams_total=c["streams_total"],
                queries_per_stream=c["queries"], timesteps=T_STEPS, places=c["places"],
                sequence_length=c["seq_len"], parallelism="stream-sharded x%d" % world,
                l2="flushed between timed iterations (256 MiB memset)")


def load_traffic(kernel, workload):
    """DRAM bytes per launch of `kernel` from the committed ncu capture of this workload (else None)."""
    for name in ("r02_traffic.json", "r01_traffic.json"):
        try:
            t = json.load(open(os.path.join(ROOT, "profiles", name))).get(kernel)
        except (OSError, ValueError):
            continue
        if isinstance(t, dict):
            t = [t]
        for e in t or []:
            if e.get("workload") == workload:
                return e["dram_bytes_per_launch"]
    return None


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(hbm_gbs=p["hbm_gbs"], bf16_burst=p["bf16_tflops"],
                    bf16_sustained=p.get("bf16_tflops_sustained", p["bf16_tflops"]), source="measured")
    return dict(hbm_gbs=6650.0, bf16_burst=1590.0, bf16_sustained=1400.0, source="fallback")


def tensor_peak(peaks, timed_region_s):
    """Burst figure for a kernel timed in a short region, sustained one inside a long step."""
    if timed_region_s >= 2.0:
        return peaks["bf16_sustained"], peaks["source"] + " bf16 sustained (timed region %.1f s)" % timed_region_s
    return peaks["bf16_burst"], peaks["source"] + " bf16 burst (timed region %.2f s)" % timed_region_s


# ------------------------------------------------------------------------------------------------
# clocks
class ClockSampler:
    """nvidia-smi sampled every 200 ms while the timed regions run (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def mark(self):
        return len(self.rows)

    def stop(self, lo=0, hi=None):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.proc.terminate()
        sm, mx, pw, reasons = [], [], [], set()
        for r in self.rows[lo:hi]:
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); pw.append(float(r[3]))
            except (ValueError, IndexError):
                continue
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6),
                              ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                if len(r) > col and r[col].lower() == "active":
                    reasons.add(name)
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_mhz_min=min(sm) if sm else None,
                    sm_max_mhz=max(mx) if mx else None, power_w_max=max(pw) if pw else None,
                    reasons=sorted(reasons), samples=len(sm))


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle port on the host cores
def cpu_arm(c, seconds, steps=1, warmup=0):
    """Times oracle/ (C restatement of the reference's path) on a bounded sample of the workload.

    One python thread per host core, each with its own oracle network and its own streams (ctypes
    releases the GIL); a sample step = `cores` x n streams x Q queries x T timesteps through
    pooling -> SNN -> sequence matching -> top-N.
    """
    from lens_b200 import synth
    from oracle import oracle as O
    cores = os.cpu_count() or 1
    I, F, P, Q, L = I_DIMS * I_DIMS, FEATURE, c["places"], c["queries"], c["seq_len"]
    Wf, Wo = synth.weights(I, F, P, seed=1)
    U = O.raster_uniforms(T_STEPS, ROI, K_POOL)
    # calibrate: one stream, one query
    net = O.OracleSNN(Wf, Wo, U, T_STEPS)
    fr = synth.frames(1, 1, ROI, seed=99)
    t0 = time.perf_counter()
    net.run_streams(O.pool(fr[0], K_POOL)[None])
    per_query = time.perf_counter() - t0
    streams_per_thread = max(1, int(seconds / max(steps + warmup, 1) / (per_query * Q)))
    if c["streams_total"] < cores * streams_per_thread:          # config 1: a single serial stream
        cores, streams_per_thread = max(1, min(cores, c["streams_total"])), 1
    nets = [O.OracleSNN(Wf, Wo, U, T_STEPS, n_streams=streams_per_thread) for _ in range(cores)]
    frames = [synth.frames(streams_per_thread, Q, ROI, seed=100 + k) for k in range(cores)]

    def work(k):
        pooled = O.pool(frames[k].reshape(-1, ROI, ROI), K_POOL).reshape(streams_per_thread, Q, I)
        S = nets[k].run_streams(pooled)
        for b in range(streams_per_thread):
            O.topk(O.seqmatch(S[b], L), N_TOP)

    times = []
    for s in range(warmup + steps):
        th = [threading.Thread(target=work, args=(k,)) for k in range(cores)]
        t0 = time.perf_counter()
        [t.start() for t in th]
        [t.join() for t in th]
        if s >= warmup:
            times.append(time.perf_counter() - t0)
    units = cores * streams_per_thread * Q * T_STEPS
    sample = (f"{cores} threads x {streams_per_thread} streams x {Q} queries x {T_STEPS} steps per step "
              f"(P={P}, L={L}), C oracle port: pool + SNN + seq-match + top-{N_TOP}")
    return dict(value=units * len(times) / sum(times), unit="query_timesteps/s", cores=cores, kind="port",
                sample=sample), float(np.mean(times)) * 1e3


def cpu_binning(seconds):
    """C oracle port of the event binning (collect_data.py:193-202) on one host core."""
    from lens_b200 import synth
    from oracle import oracle as O
    n = 1 << 22
    t, x, y, n_win = synth.events(n, sensor=128, seed=5)
    t0 = time.perf_counter()
    reps = 0
    while reps < 1 or time.perf_counter() - t0 < seconds:
        O.bin_events(t, x, y, 0, 250_000, n_win, 128, 8)
        reps += 1
    return dict(value=n * reps / (time.perf_counter() - t0), unit="events/s", cores=1, kind="port",
                sample="%d x %d events, 128x128, C oracle port" % (reps, n))


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    c = resolve(args, world=world)
    budget = float(os.environ.get("LENS_BENCH_CPU_SECONDS", max(20.0, 4.0 * (args.steps + args.warmup))))
    if "places" not in c:                                           # config 4: events/s
        cb = cpu_binning(budget)
        line = dict(metric="events_per_sec", value=cb["value"], unit="events/s", n_gpus=args.gpus,
                    steps=args.steps, warmup=args.warmup, ms_per_step=None, higher_is_better=True,
                    scaling=c["scaling"], vs_baseline=None, dtype="u8+int32", data="synthetic", impl="reference",
                    config=workload_config(c, world), cpu_baseline=cb,
                    e2e=dict(value=cb["value"], unit="events/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))
        return emit(line)
    cb, ms = cpu_arm(c, seconds=budget, steps=args.steps, warmup=args.warmup)
    line = dict(metric="query_timesteps_per_sec", value=cb["value"], unit="query_timesteps/s",
                n_gpus=args.gpus, steps=args.steps, warmup=args.warmup, ms_per_step=ms,
                higher_is_better=True, scaling=c["scaling"], vs_baseline=None, dtype="i8->i64+f32", data="synthetic",
                impl="reference", config=workload_config(c, world), cpu_baseline=cb,
                e2e=dict(value=cb["value"], unit="query_timesteps/s", h2d_bytes_per_step=0,
                         d2h_bytes_per_step=0),
                note="reference = Python/sinabs (not installable offline); timed: the C oracle port of its "
                     "path on all host cores, each step a bounded sample of the workload")
    emit(line)


# ------------------------------------------------------------------------------------------------
_REAL_STDOUT = None


def quiet_stdout():
    """Route everything libraries print to stdout (e.g. NCCL's version banner) to stderr so that the
    ONE JSON line is the only thing on stdout."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


DUMP_BYTES = 60 << 20          # array data of --dump-outputs: with the .npy headers the files stay under 64 MB


def dump_outputs(directory, arrays, budget=DUMP_BYTES):
    """Write the tensors one step of the timed path returned (name -> tensor) as DIR/<name>.npy, so that two
    builds run with the same arguments can be compared output for output.

    Values are float32 where that is exact (float32, integers of up to 16 bits, bool) and float64 otherwise.
    Arrays of two or more dimensions share their leading dimension (streams, or event windows); when they do
    not fit in `budget` bytes, the same fixed, seeded sample of those rows is written for each of them.
    DIR/sample_rows.npy lists the rows written."""
    import math
    import torch
    exact32 = (torch.float32, torch.uint8, torch.int8, torch.int16, torch.bool)

    def dtype(t):
        return np.dtype(np.float32 if t.dtype in exact32 else np.float64)
    whole = {k: t for k, t in arrays.items() if t.dim() < 2}
    rowed = {k: t for k, t in arrays.items() if t.dim() >= 2}
    lead = {t.shape[0] for t in rowed.values()}
    assert len(lead) <= 1, "arrays of two or more dimensions must share their leading dimension"
    n = lead.pop() if lead else 0
    fixed = sum(t.numel() * dtype(t).itemsize for t in whole.values())
    per_row = 8 + sum(math.prod(t.shape[1:]) * dtype(t).itemsize for t in rowed.values())
    keep = min(n, (budget - fixed) // per_row)
    rows = np.arange(n) if keep == n else np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
    os.makedirs(directory, exist_ok=True)
    for k, t in whole.items():
        np.save(os.path.join(directory, k + ".npy"), t.cpu().numpy().astype(dtype(t)))
    for k, t in rowed.items():
        picked = t.index_select(0, torch.from_numpy(rows).to(t.device))
        np.save(os.path.join(directory, k + ".npy"), picked.cpu().numpy().astype(dtype(t)))
    np.save(os.path.join(directory, "sample_rows.npy"), rows.astype(np.float64))


# ------------------------------------------------------------------------------------------------
class Ctx:
    """torch / distributed state shared by the measurements."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            import datetime
            # a desynchronised collective should abort the run within minutes, not after NCCL's default 10
            dist.init_process_group("nccl", device_id=self.dev, timeout=datetime.timedelta(seconds=180))
        self.peaks = load_peaks()
        self.flush = torch.empty(256 << 20, dtype=torch.uint8, device=self.dev)
        self.args = args

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def timed(self, fn, steps):
        """CUDA events on the launching (current) stream around every call; L2 flushed in between.
        -> (ms per call, what the last call returned)."""
        torch = self.torch
        evs, out = [], None
        for _ in range(steps):
            out = None                  # free the previous call's outputs before this call allocates its own
            self.flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); out = fn(); b.record()
            evs.append((a, b))
        torch.cuda.synchronize()
        return [a.elapsed_time(b) for a, b in evs], out

    def max_over_ranks(self, *vals):
        t = self.torch.tensor(list(vals), dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return t.tolist()


def measure_snn(ctx, c, steps, warmup, W_out_sharded=False, want_e2e=True, dump=None):
    """One SNN + matching configuration: resident and host-fed throughput, per-kernel rooflines.
    `dump`: directory for what the last timed resident step returned (this rank's streams)."""
    torch, dist = ctx.torch, ctx.dist
    from lens_b200 import synth, _lib
    from lens_b200.pipeline import InferencePipeline
    dev, world, rank, peaks = ctx.dev, ctx.world, ctx.rank, ctx.peaks
    B, Q, L, P = c["streams_per_gpu"], c["queries"], c["seq_len"], c["places"]
    I, F = I_DIMS * I_DIMS, FEATURE
    res = {}
    if W_out_sharded and world > 1:
        # the database arrives as row shards (P / world places per rank): one NCCL all-gather over NVLink
        rows = P // world
        Wf, Wo_shard = synth.weights(I, F, rows, seed=6 + rank)
        Wf, _ = synth.weights(I, F, 1, seed=6)                      # the feature layer is replicated
        shard = torch.from_numpy(Wo_shard).to(dev)
        full = torch.empty((rows * world, F), dtype=torch.float32, device=dev)
        for _ in range(2):
            dist.all_gather_into_tensor(full, shard)
        ctx.barrier()
        ag, _ = ctx.timed(lambda: dist.all_gather_into_tensor(full, shard), 5)
        ag_ms, = ctx.max_over_ranks(float(np.mean(ag)))
        res["all_gather"] = dict(bytes=int(full.numel() * 4), ms=ag_ms,
                                 algbw_GBps=full.numel() * 4 / (ag_ms / 1e3) / 1e9, collective="ncclAllGather (W_out rows)")
        Wo_t, P = full, rows * world
    else:
        Wf, Wo = synth.weights(I, F, P, seed=6 if W_out_sharded else 1)
        Wo_t = torch.from_numpy(Wo)
    pipe = InferencePipeline(torch.from_numpy(Wf), Wo_t, roi=ROI, k=K_POOL, T=T_STEPS,
                             L=L, n_top=N_TOP, ns=NS, max_streams=B, device=dev, mode=ctx.args.mode)
    frames_dev = synth.frames_device(B, Q, ROI, seed=2 + rank, device=dev)
    frames_host = None
    if want_e2e:
        frames_host = torch.empty(frames_dev.shape, dtype=torch.uint8, pin_memory=True)
        frames_host.copy_(frames_dev)
    gt_center = torch.from_numpy(synth.gt_centers(B, Q - L + 1, P - L + 1, seed=7 + rank)).to(dev)
    units_per_step = B * Q * T_STEPS

    def step_resident():
        out = pipe.step(frames=frames_dev, gt_center=gt_center, gt_tol=2)
        return out

    def step_e2e():
        # public API fed from pinned host memory: H2D of this step's frames (side stream; the copy for the
        # following step is started behind this step's kernels) ... D2H of the step's result
        out = pipe.step_host(frames_host, gt_center=gt_center, gt_tol=2, next_frames=frames_host)
        r = torch.cat([out["hits"], out["n_valid"]]).cpu()
        idx = out["top_idx"].cpu()
        return r, idx

    for _ in range(max(warmup, 3)):
        step_resident()
    if want_e2e:
        for _ in range(2):
            step_e2e()
    ctx.barrier()
    pipe.net.set_timing(True)
    pipe.stage_timing = True
    launches0 = _lib.launch_count()
    ctx.barrier()
    ms, out = ctx.timed(step_resident, steps)
    ctx.barrier()
    launches = _lib.launch_count() - launches0
    ktime = pipe.net.get_timing()
    stage = pipe.pop_stage_timing()
    pipe.net.set_timing(False)
    pipe.stage_timing = False
    if dump:
        dump_outputs(dump, {k: v for k, v in out.items() if v is not None})
    del out
    ms_e2e = [0.0]
    if want_e2e:
        ctx.barrier()
        ms_e2e, _ = ctx.timed(step_e2e, steps)
        ctx.barrier()
    last = step_resident()
    recall = pipe.recall(last["hits"], last["n_valid"])
    overflow = pipe.net.overflow()
    if W_out_sharded and world > 1:
        # final merge of the query shards' top-N lists on every rank (config 5)
        ti = last["top_idx"].contiguous()
        allti = torch.empty((world,) + tuple(ti.shape), dtype=ti.dtype, device=dev)
        dist.all_gather_into_tensor(allti, ti)
        ctx.barrier()
        tg, _ = ctx.timed(lambda: dist.all_gather_into_tensor(allti, ti), 5)
        tg_ms, = ctx.max_over_ranks(float(np.mean(tg)))
        res["topn_gather"] = dict(bytes=int(allti.numel() * 4), ms=tg_ms, collective="ncclAllGather (top-N indices)")
    del last

    tot_ms, tot_e2e_ms = ctx.max_over_ranks(sum(ms), sum(ms_e2e))
    value = world * units_per_step * steps / (tot_ms / 1e3)
    region_s = sum(ms) / 1e3
    tpeak, tsrc = tensor_peak(peaks, region_s)
    # one launch covers at most `group` streams (the hidden-spike scratch is bounded to 6 GiB, csrc/snn.cu): the
    # committed ncu traffic figures are per launch of a full group
    chunks = Q * (-(-T_STEPS // 32))
    group = 2 * ((6 << 30) // (chunks * 64 * (-(-F // 32) * 32)))
    wl = "streams=%d,queries=%d,places=%d,feature=%d" % (min(B, group), Q, P, F)

    # ---- per-kernel rooflines (CUDA events on the launch stream, recorded by the library / the pipeline)
    def tensor_roof(kernel, flops_per_unit, total_ms, n_launch, traffic_key, algorithmic):
        ach = flops_per_unit * units_per_step * steps / (total_ms / 1e3) / 1e12 if total_ms > 0 else 0.0
        return dict(kernel=kernel, bound="tensor", achieved=ach, peak=tpeak, unit="TFLOP/s", frac=ach / tpeak,
                    traffic=load_traffic(traffic_key, wl), peak_source=tsrc,
                    kernel_ms=total_ms / max(n_launch, 1), launches_per_step=n_launch / steps,
                    ms_per_step=total_ms / steps, share_of_step=total_ms / sum(ms), algorithmic=algorithmic)
    k3 = tensor_roof("K3 snn output layer (F->P contraction + IAF#2 + spike counts)", 2.0 * F * P,
                     ktime["output_ms"], ktime["n_output"], "output_tc_kernel",
                     "2*F*P FLOP per query timestep")
    k2 = tensor_roof("K2 snn hidden layer (raster + I->F contraction + IAF#1)", 2.0 * I * F,
                     ktime["feature_ms"], ktime["n_feature"], "hidden_tc_kernel",
                     "2*I*F FLOP per query timestep")
    match_ms = stage["match_ms"]
    k4_bytes = (4.0 * B * Q * P + 8.0 * B * (Q - L + 1) * N_TOP) * steps
    k4_ach = k4_bytes / (match_ms / 1e3) / 1e9 if match_ms > 0 else 0.0
    k4 = dict(kernel="K4 sequence matching + top-%d + recall counters" % N_TOP, bound="hbm", achieved=k4_ach,
              peak=peaks["hbm_gbs"], unit="GB/s", frac=k4_ach / peaks["hbm_gbs"],
              traffic=load_traffic("seqmatch_topk_kernel", "streams=%d,queries=%d,places=%d,feature=%d" % (B, Q, P, F)),
              peak_source=peaks["source"],
              ms_per_step=match_ms / steps, share_of_step=match_ms / sum(ms),
              algorithmic="4 B per similarity entry read once + 8 B per top-N entry")
    res.update(value=value, ms_per_step=tot_ms / steps, units_per_step_per_gpu=units_per_step,
               gpu_launches=int(launches), recall_at_n=dict(zip(map(str, NS), recall)), spike_overflow=overflow,
               roofline=k3, rooflines=[k2, k3, k4],
               stage_ms_per_step=dict(pool_plus_snn=stage["similarity_ms"] / steps, match=match_ms / steps,
                                      hidden_kernels=ktime["feature_ms"] / steps,
                                      output_kernels=ktime["output_ms"] / steps))
    if want_e2e:
        res["e2e"] = dict(value=world * units_per_step * steps / (tot_e2e_ms / 1e3), unit="query_timesteps/s",
                          h2d_bytes_per_step=int(frames_host.numel()),
                          d2h_bytes_per_step=int(7 * 8 + B * (Q - L + 1) * N_TOP * 4),
                          ms_per_step=tot_e2e_ms / steps)
    del pipe, frames_dev, frames_host
    torch.cuda.empty_cache()
    return res


def measure_place_sharded(ctx, c, steps):
    """Config 5 the other way round: the DATABASE is sharded (P / N places + L - 1 halo per rank), every rank
    runs all streams of the job against its shard, the per-rank top-N lists are all-gathered over NCCL and
    merged on the GPU (lens_topn_merge).  Reports the whole step and the collective + merge part alone."""
    torch, dist = ctx.torch, ctx.dist
    from lens_b200 import synth, ops
    from lens_b200.pipeline import PlaceShardedPipeline
    dev, world, rank = ctx.dev, ctx.world, ctx.rank
    B, Q, L, P = c["streams_total"], c["queries"], c["seq_len"], c["places"]
    I, F = I_DIMS * I_DIMS, FEATURE
    Wf, Wo = synth.weights(I, F, P, seed=6)
    pipe = PlaceShardedPipeline(torch.from_numpy(Wf), torch.from_numpy(Wo), roi=ROI, k=K_POOL, T=T_STEPS, L=L,
                                n_top=N_TOP, ns=NS, max_streams=B, device=dev, mode=ctx.args.mode)
    frames = synth.frames_device(B, Q, ROI, seed=2, device=dev)           # every rank sees every stream
    gt = torch.from_numpy(synth.gt_centers(B, Q - L + 1, P - L + 1, seed=7)).to(dev)
    for _ in range(3):
        out = pipe.step(frames=frames, gt_center=gt, gt_tol=2)
    ctx.barrier()
    ms, _ = ctx.timed(lambda: pipe.step(frames=frames, gt_center=gt, gt_tol=2), steps)
    ctx.barrier()
    # the exchange alone: all-gather of (value, index) lists + merge
    tv, ti = out["top_val"].contiguous(), out["top_idx"].contiguous()
    allv = torch.empty((world,) + tuple(tv.shape), dtype=tv.dtype, device=dev)
    alli = torch.empty((world,) + tuple(ti.shape), dtype=ti.dtype, device=dev)

    def exchange():
        if world > 1:
            dist.all_gather_into_tensor(allv, tv)
            dist.all_gather_into_tensor(alli, ti)
        return ops.topn_merge(allv, alli)
    if world == 1:
        allv.copy_(tv[None]); alli.copy_(ti[None])
    for _ in range(3):
        exchange()
    ctx.barrier()
    xms, _ = ctx.timed(exchange, 5)
    tot, xt = ctx.max_over_ranks(sum(ms), float(np.mean(xms)))
    del pipe, frames
    torch.cuda.empty_cache()
    return dict(workload="%s, database sharded: %d places/GPU (+%d halo), all %d streams on every GPU" %
                         (c["name"], P // world, L - 1, B),
                value=B * Q * T_STEPS * steps / (tot / 1e3), unit="query_timesteps/s", ms_per_step=tot / steps,
                topn_exchange=dict(ms=xt, bytes_gathered=int(allv.numel() * 8),
                                   collective="2 x ncclAllGather (top-N values, indices) + lens_topn_merge"),
                recall_at_n=dict(zip(map(str, NS), (out["hits"].double() / max(int(out["n_valid"].item()), 1)).tolist())))


def measure_latency(ctx, c, reps=5, dump=None):
    """Config 1: ONE stream, serial chain of Q*T steps through the public batched call; us per step.
    `dump`: directory for what the last timed pass returned."""
    torch = ctx.torch
    from lens_b200 import synth
    from lens_b200.pipeline import InferencePipeline
    I, F, P, Q, L = I_DIMS * I_DIMS, FEATURE, c["places"], c["queries"], c["seq_len"]
    Wf, Wo = synth.weights(I, F, P, seed=1)
    pipe = InferencePipeline(torch.from_numpy(Wf), torch.from_numpy(Wo), roi=ROI, k=K_POOL, T=T_STEPS, L=L,
                             n_top=N_TOP, ns=NS, max_streams=1, device=ctx.dev, mode=ctx.args.mode)
    frames = torch.from_numpy(synth.frames(1, Q, ROI, seed=2)).to(ctx.dev)
    gt = torch.from_numpy(synth.gt_centers(1, Q - L + 1, P - L + 1, seed=7)).to(ctx.dev)
    # reduce=False: a single stream is "replicas only" (no collective; other ranks may not even be here)
    for _ in range(3):
        pipe.step(frames=frames, gt_center=gt, gt_tol=2, reduce=False)
    ms, out = ctx.timed(lambda: pipe.step(frames=frames, gt_center=gt, gt_tol=2, reduce=False), reps)
    if dump:
        dump_outputs(dump, {k: v for k, v in out.items() if v is not None})
    best = float(np.min(ms))
    return dict(workload="%s: %s" % (c["name"], c["what"]), ms_per_pass=float(np.mean(ms)), ms_best=best,
                serial_steps=Q * T_STEPS, us_per_step=float(np.mean(ms)) * 1e3 / (Q * T_STEPS),
                value=Q * T_STEPS / (float(np.mean(ms)) / 1e3), unit="query_timesteps/s")


def measure_binning(ctx, c, steps, dump=None):
    """Config 4: this rank's window-aligned shard of the event stream -> frames + pooled (K1).
    `dump`: directory for what the last timed call returned."""
    torch = ctx.torch
    from lens_b200 import synth, ops
    world, dev, peaks = ctx.world, ctx.dev, ctx.peaks
    n_local = c["events"] // world
    t_dev, x_dev, y_dev, n_win = synth.events_device(n_local, sensor=128, seed=5 + ctx.rank, device=dev)
    I = (128 // K_POOL) ** 2

    def bin_step():
        return ops.bin_events(t_dev, x_dev, y_dev, 0, 250_000, n_win, 128, K_POOL)
    for _ in range(3):
        bin_step()
    ctx.barrier()
    bms, out = ctx.timed(bin_step, steps)
    ctx.barrier()
    if dump:
        dump_outputs(dump, dict(zip(("frames", "pooled", "counts"), out)))
    del out
    bsec, = ctx.max_over_ranks(float(np.mean(bms)))
    bsec /= 1e3
    out_bytes = n_win * (128 * 128 + I)
    alg_bytes = 8.0 * n_local + out_bytes            # SURVEY 8d: t, x, y read once
    act_bytes = 4.0 * n_local + out_bytes            # what this kernel streams: x, y (t only by binary search)
    del t_dev, x_dev, y_dev
    torch.cuda.empty_cache()
    return dict(metric="events_per_sec", value=world * n_local / bsec, unit="events/s", events_per_gpu=n_local,
                events_total=n_local * world, windows_per_gpu=n_win, ms=bsec * 1e3,
                roofline=dict(kernel="K1 event binning + pooling (bin_pow2_kernel)", bound="hbm",
                              achieved=act_bytes / bsec / 1e9, peak=peaks["hbm_gbs"], unit="GB/s",
                              frac=act_bytes / bsec / 1e9 / peaks["hbm_gbs"],
                              achieved_survey_8d=alg_bytes / bsec / 1e9,
                              frac_survey_8d=alg_bytes / bsec / 1e9 / peaks["hbm_gbs"],
                              traffic=load_traffic("bin_pow2_kernel", "events=%d" % n_local),
                              peak_source=peaks["source"],
                              algorithmic="streamed: 4 B/event (x, y; the sorted time array is only probed by "
                                          "the per-window binary search) + 1 B per frame pixel + I B per frame; "
                                          "SURVEY 8d figure (8 B/event) reported as *_survey_8d"))


def main():
    args = parse()
    quiet_stdout()
    if args.impl == "reference":
        return run_reference(args)

    ctx = Ctx(args)
    torch, dist = ctx.torch, ctx.dist
    rank, world = ctx.rank, ctx.world
    c = resolve(args, world=world)
    sampler = ClockSampler(ctx.local)
    if rank == 0:
        sampler.start()                      # samples through warm-up and the timed regions

    dump = args.dump_outputs if rank == 0 else None
    if "places" not in c:                    # --config 4: binning is the main line
        b = measure_binning(ctx, c, args.steps, dump=dump)
        line = dict(metric="events_per_sec", value=b["value"], unit="events/s", n_gpus=world, steps=args.steps,
                    warmup=max(args.warmup, 3), ms_per_step=b["ms"], higher_is_better=True, scaling=c["scaling"],
                    vs_baseline=None, dtype="u8+int32", data="synthetic", config=workload_config(c, world),
                    roofline=b["roofline"], binning=b, gpu_launches=2 * args.steps)
    elif c["name"] == "config1":
        lat = measure_latency(ctx, c, reps=args.steps, dump=dump)
        line = dict(metric="query_timesteps_per_sec", value=lat["value"], unit="query_timesteps/s", n_gpus=world,
                    steps=args.steps, warmup=max(args.warmup, 3), ms_per_step=lat["ms_per_pass"],
                    higher_is_better=True, scaling="replicas", vs_baseline=None, dtype="i8->i64+f32",
                    data="synthetic", config=workload_config(c, world), latency=lat)
    else:
        m = measure_snn(ctx, c, args.steps, args.warmup, W_out_sharded=(c["name"] == "config5"), dump=dump)
        line = dict(metric="query_timesteps_per_sec", value=m.pop("value"), unit="query_timesteps/s", n_gpus=world,
                    steps=args.steps, warmup=max(args.warmup, 3), ms_per_step=m.pop("ms_per_step"),
                    higher_is_better=True, scaling=c["scaling"], vs_baseline=None, dtype="i8->i64+f32",
                    data="synthetic", config=workload_config(c, world), e2e=m.pop("e2e"),
                    gpu_launches=m.pop("gpu_launches"), roofline=m.pop("roofline"), **m)
    main_rows = sampler.mark()

    # ---- the other configurations, bounded (a few steps each)
    extras = {}
    if not args.no_extras:
        want = [int(k) for k in args.extras.split(",") if k.strip()]
        ksteps = max(3, min(args.steps, 5))
        for k in want:
            if k == args.config:
                continue
            ck = resolve(args, config=k, world=world)
            try:
                if k == 1:
                    extras["config1_latency"] = measure_latency(ctx, ck)      # every rank runs its own replica
                    ctx.barrier()
                elif k == 4:
                    extras["config4_binning"] = measure_binning(ctx, ck, ksteps)
                elif k == 2:
                    m = measure_snn(ctx, ck, ksteps, 3, want_e2e=False)
                    m["config"] = workload_config(ck, world)
                    extras["config2"] = m
                elif k == 5:
                    m = measure_snn(ctx, ck, min(ksteps, 3), 3, W_out_sharded=True, want_e2e=False)
                    m["config"] = workload_config(ck, world)
                    extras["config5"] = m
                    if world > 1:
                        extras["config5_place_sharded"] = measure_place_sharded(ctx, ck, min(ksteps, 3))
            except Exception as e:                                   # an extra must never cost the main line
                extras["config%d_error" % k] = repr(e)[:300]
    if "config4_binning" in extras:
        line["binning"] = extras["config4_binning"]
        line.setdefault("rooflines", []).insert(0, extras["config4_binning"]["roofline"])
    if extras:
        line["extras"] = extras
    line["clocks"] = sampler.stop(0, main_rows if main_rows > 2 else None) if rank == 0 else None

    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        if "places" in c:
            line["cpu_baseline"], _ = cpu_arm(c, seconds=args.cpu_seconds)
            if "config1_latency" in extras or c["name"] == "config1":
                c1 = resolve(args, config=1, world=1)
                cb1, _ = cpu_arm(c1, seconds=3.0)
                (extras.get("config1_latency") or line["latency"])["cpu_us_per_step"] = 1e6 / cb1["value"] * cb1["cores"]
        else:
            line["cpu_baseline"] = cpu_binning(args.cpu_seconds)
    if rank == 0:
        emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
