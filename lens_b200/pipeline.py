"""The hot path as one object: events or frames -> pooled pixels -> spike counts -> sequence matching ->
top-N -> Recall@N counters, for a shard of independent query streams on one GPU.

This is what `LENS.evaluate` does for one stream and what bench.py / the multi-GPU driver do for
thousands: every stage is a call into liblens_b200.so; torch only owns the buffers.  With
`torch.distributed` initialised, streams are sharded contiguously across ranks (one process per
GPU, no data-path collective) and the Recall@N counters are summed with one all-reduce
(SURVEY.md 8e).
"""
import numpy as np
import torch

from . import ops
from ._lib import LensError
from .network import B200Network, MODE_AUTO


def shard_range(n, rank, world):
    """Contiguous [lo, hi) slice of n units owned by `rank` (first n % world ranks get one extra)."""
    base, extra = divmod(n, world)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def place_shard_range(P, L, rank, world):
    """Places a rank holds when the DATABASE is sharded: its own contiguous range [p0, p1) of the
    P - L + 1 sequence-matched rows plus the L - 1 places after it (every diagonal that starts in the
    range is complete without an exchange).  -> (p0, p1, p1_with_halo)."""
    Po = P - max(L, 1) + 1
    p0, p1 = shard_range(Po, rank, world)
    return p0, p1, min(P, p1 + max(L, 1) - 1)


class InferencePipeline:
    def __init__(self, W_feat, W_out, roi, k, T, L, n_top=25, ns=ops.RECALL_NS, max_streams=1,
                 device=None, mode=MODE_AUTO):
        self.net = B200Network(W_feat, W_out, roi=roi, k=k, num_timesteps=T, max_streams=max_streams,
                               device=device)
        self.L, self.n_top, self.ns, self.mode = int(L), int(n_top), tuple(ns), mode
        self.device = self.net.device
        # optional per-stage CUDA-event timing (bench.py): [(start, after similarity, after match)]
        self.stage_timing = False
        self._stage_events = []

    def similarity(self, frames=None, pooled=None):
        """u8 frames [B, Q, roi, roi] (or pooled [B, Q, I]) -> spike counts f32 [B, Q, P]."""
        return self.net.run_streams(frames=frames, pooled=pooled, mode=self.mode)

    def match(self, S, gt_dense=None, gt_center=None, gt_tol=0, want_D=False):
        """S [B, Q, P] -> dict(top_val, top_idx, D, hits, n_valid); hits are per-rank counters."""
        tv, ti, D = ops.seqmatch_topk(S, self.L, self.n_top, want_D=want_D)
        out = dict(top_val=tv, top_idx=ti, D=D, hits=None, n_valid=None)
        if gt_dense is not None or gt_center is not None:
            Po = S.shape[2] - self.L + 1
            out["hits"], out["n_valid"] = ops.recall_counts(ti, Po, gt_dense=gt_dense,
                                                            gt_center=gt_center, gt_tol=gt_tol, ns=self.ns)
        return out

    def step(self, frames=None, pooled=None, gt_dense=None, gt_center=None, gt_tol=0, reduce=True):
        """One pass of the hot path over this rank's shard; Recall counters all-reduced if distributed."""
        ev = None
        if self.stage_timing:
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            ev[0].record()
        S = self.similarity(frames=frames, pooled=pooled)
        if ev:
            ev[1].record()
        out = self.match(S, gt_dense=gt_dense, gt_center=gt_center, gt_tol=gt_tol)
        if ev:
            ev[2].record()
            self._stage_events.append(ev)
        out["S"] = S
        out["overflow"] = self.net.overflow_tensor()   # device counter, no synchronisation: check with .item()
        if reduce:
            self._all_reduce_hits(out)
        return out

    @staticmethod
    def _all_reduce_hits(out):
        if out["hits"] is not None and torch.distributed.is_available() \
                and torch.distributed.is_initialized() and torch.distributed.get_world_size() > 1:
            packed = torch.cat([out["hits"], out["n_valid"]])
            torch.distributed.all_reduce(packed)          # sum of 6 hit counters + valid count
            out["hits"], out["n_valid"] = packed[:-1], packed[-1:]

    def _bin_streams(self, t_us, x, y, offsets, t0_us, window_us, Q, roi_x0, roi_y0):
        net = self.net
        _, pooled, n_ev = ops.bin_event_streams(t_us, x, y, offsets, t0_us, window_us, Q, net.roi, net.k,
                                                roi_x0=roi_x0, roi_y0=roi_y0, want_frames=False, want_pooled=True)
        return pooled, n_ev

    def step_events(self, t_us, x, y, offsets, t0_us, window_us, Q, roi_x0=0, roi_y0=0, gt_dense=None,
                    gt_center=None, gt_tol=0, reduce=True):
        """The step fed from raw event streams: stream b is events [offsets[b], offsets[b+1]) of the device
        arrays t_us / x / y, and query q of stream b is its window [t0_us[b] + q * window_us, + window_us)
        (see ops.bin_event_streams).  The events are binned straight to pooled pixels (no frames are
        written) and run through the same work as `step(pooled=...)`.  Returns `step`'s dict plus
        "events_per_window" i32 [B, Q].

        Every stream yields exactly Q queries: a window without events becomes an all-zero pooled row and
        stays a query, unlike collect_data.create_images in the reference, which drops empty windows
        (collect_data.frames_from_events is the single-stream path that reproduces that)."""
        with torch.cuda.device(self.device):
            pooled, n_ev = self._bin_streams(t_us, x, y, offsets, t0_us, window_us, Q, roi_x0, roi_y0)
            out = self.step(pooled=pooled, gt_dense=gt_dense, gt_center=gt_center, gt_tol=gt_tol, reduce=reduce)
        out["events_per_window"] = n_ev
        return out

    def step_event_groups(self, groups, B, Q, window_us, roi_x0=0, roi_y0=0, gt_dense=None, gt_center=None,
                          gt_tol=0, reduce=True):
        """`step_events` for fleets whose events do not fit in device memory together.

        `groups` yields (b0, t_us, x, y, offsets, t0_us) for consecutive ranges of streams that cover
        [0, B): the group's streams are b0 .. b0 + len(t0_us) - 1, with offsets relative to its own arrays.
        b0 must be even (the network tiles streams in pairs).  Each group is binned and run through the
        network as soon as it arrives, into one spike-count tensor S [B, Q, P]; matching, top-N and recall
        run once at the end.  The results equal `step_events` on the same events bit for bit; the per-group
        event arrays may be released or refilled once the group's kernels have run (stream order)."""
        net = self.net
        with torch.cuda.device(self.device):
            net.ensure_streams(B)
            S = torch.empty((B, Q, net.P), dtype=torch.float32, device=self.device)
            n_ev = torch.empty((B, Q), dtype=torch.int32, device=self.device)
            b_next = 0
            for b0, t_us, x, y, offsets, t0_us in groups:
                nb = offsets.numel() - 1
                if b0 % 2:
                    raise LensError(f"event group starts at odd stream {b0}: b0 must be even")
                if b0 != b_next or b0 + nb > B:
                    raise LensError(f"event groups must cover streams [0, {B}) in order: got [{b0}, {b0 + nb}) "
                                    f"after [0, {b_next})")
                pooled, ev = self._bin_streams(t_us, x, y, offsets, t0_us, window_us, Q, roi_x0, roi_y0)
                n_ev[b0:b0 + nb] = ev
                net.run_streams_range(pooled, b0, S[b0:b0 + nb], mode=self.mode)
                b_next = b0 + nb
            if b_next != B:
                raise LensError(f"event groups cover streams [0, {b_next}) of {B}")
            out = self.match(S, gt_dense=gt_dense, gt_center=gt_center, gt_tol=gt_tol)
            out["S"] = S
            out["overflow"] = net.overflow_tensor()
        out["events_per_window"] = n_ev
        if reduce:
            self._all_reduce_hits(out)
        return out

    def step_host(self, frames_host, gt_dense=None, gt_center=None, gt_tol=0, next_frames=None, reduce=True):
        """The same step fed from PINNED HOST frames u8 [B, Q, roi, roi].

        The host->device copy runs on a side stream into one of two staging buffers.  Passing the
        following step's host tensor as `next_frames` starts its copy right after this step's kernels
        are queued, so in a stream of steps the PCIe transfer of step k+1 hides behind the compute of
        step k (every step still pays for its own copy; only the first one is exposed)."""
        net, dev = self.net, self.device
        main = torch.cuda.current_stream(dev)
        if not hasattr(self, "_copy_stream"):
            self._copy_stream = torch.cuda.Stream(device=dev)
            self._stage, self._stage_free, self._pending = [None, None], [None, None], {}
            self._slot = 0

        def start_copy(src):
            slot = self._slot
            self._slot ^= 1
            if self._stage[slot] is None or self._stage[slot].shape != src.shape:
                self._stage[slot] = torch.empty(src.shape, dtype=torch.uint8, device=dev)
                self._stage_free[slot] = None
                # the allocator may hand back a block that kernels queued on the main stream still read
                self._copy_stream.wait_stream(main)
            with torch.cuda.stream(self._copy_stream):
                if self._stage_free[slot] is not None:
                    self._copy_stream.wait_event(self._stage_free[slot])   # last reader of this buffer
                self._stage[slot].copy_(src, non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(self._copy_stream)
            self._pending[src.data_ptr()] = (slot, ev)

        if frames_host.data_ptr() not in self._pending:
            start_copy(frames_host)
        slot, ev = self._pending.pop(frames_host.data_ptr())
        main.wait_event(ev)
        out = self.step(frames=self._stage[slot], gt_dense=gt_dense, gt_center=gt_center, gt_tol=gt_tol,
                        reduce=reduce)
        self._stage_free[slot] = torch.cuda.Event()
        self._stage_free[slot].record(main)
        if next_frames is not None:
            start_copy(next_frames)
        return out

    def pop_stage_timing(self):
        """-> dict(similarity_ms, match_ms, n) summed over the steps recorded since the last call."""
        torch.cuda.synchronize(self.device)
        sim = sum(a.elapsed_time(b) for a, b, _ in self._stage_events)
        mat = sum(b.elapsed_time(c) for _, b, c in self._stage_events)
        n = len(self._stage_events)
        self._stage_events = []
        return dict(similarity_ms=sim, match_ms=mat, n=n)

    def precision_recall(self, S, gt_dense=None, gt_center=None, gt_tol=0, matching="single", best="place",
                         n_thresh=100, reduce=True):
        """createPR's precision-recall lists for the whole fleet, from the spike counts S f32 [B, Q, P] that the
        steps return; the sequence-matched matrices are recomputed on the GPU, never stored.
        -> dict(P, R, tp, fp, gtp): P / R python lists of length n_thresh + 1 (as createPR), tp / fp numpy i64.

        The fleet's curve is createPR over the streams' matrices concatenated along its column axis, so the
        thresholds span the whole fleet (and every rank, under torch.distributed with reduce=True):
          matching='single', best='place': createPR(D_b.T, GT_b.T, 'single') at B = 1, the reference's --PR_curve
          matching='single', best='query': createPR(D_b, GT_b, 'single') at B = 1, the SAD path's call
          matching='multi':                createPR(D_b, GT_b, 'multi') at B = 1
        Ground truth as `match`: gt_dense u8 [Po, Qo] or [B, Po, Qo], or gt_center i32 [B, Qo] with gt_tol.
        Under torch.distributed with reduce=True: one all-reduce MAX of the extremes between the two passes and one
        all-reduce SUM of [tp, fp, gtp]; reduce=False gives this rank's own curve."""
        from .src.metrics import pr_lists
        mode = ops.seqpr_mode(matching, best)
        ops._seqpr_check(S, self.L, mode, gt_dense, gt_center, n_thresh)
        gt = dict(gt_dense=gt_dense, gt_center=gt_center, gt_tol=gt_tol)
        dist = torch.distributed
        shared = reduce and dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1
        with torch.cuda.device(S.device):
            records, extremes, gtp = ops.seqpr_scan(S, self.L, mode, **gt)
            if shared:
                dist.all_reduce(extremes, op=dist.ReduceOp.MAX)     # {max, ~min} keys: max merges both
            tp, fp = ops.seqpr_counts(S, self.L, mode, records, extremes, n_thresh, **gt)
            packed = torch.cat([tp, fp, gtp])
            if shared:
                dist.all_reduce(packed)
        packed = packed.cpu().numpy()
        tp, fp, gtp = packed[:n_thresh], packed[n_thresh:2 * n_thresh], int(packed[-1])
        P, R = pr_lists(tp, fp, gtp)
        return dict(P=P, R=R, tp=tp, fp=fp, gtp=gtp)

    @staticmethod
    def recall(hits, n_valid):
        nv = int(n_valid.item())
        return [float(h) / nv if nv else float("nan") for h in hits.tolist()]


class StreamingPipeline(InferencePipeline):
    """The hot path for live cameras: a fixed fleet of `n_streams` streams that deliver a few query windows at a
    time (one 250 ms timebin per push, typically), with sequence matching that spans the pushes.

    A push carries Q >= 1 new windows for every stream (the fleet in lockstep), or for any subset of the streams in
    any order (`push(..., streams=...)`: cameras that start late, deliver at their own rate or drop out for a while);
    a stream outside a push keeps all of its state.  Number a stream's rows g = 0, 1, 2, ... since its last reset: new
    row g yields the top-N of the sequence that ends at it, once the stream has seen L rows (g >= L - 1); earlier
    (warm-up) rows are -inf / -1.  However a stream's windows are split into pushes, its valid rows equal, bit for
    bit, the columns of one `step` over all of them (column g - L + 1).

    The object owns the device state that makes this work: the SNN membrane potentials (as any pipeline), `ring`
    f32 [n_streams, L - 1, P] (the last L - 1 spike-count rows of every stream, row g at slot g mod (L - 1), g counted
    by `rows`), `seen` i32 [n_streams] (rows since each stream's reset, saturating at L - 1) and `rows` i64
    [n_streams] (rows pushed to each stream since construction or `reset()`; `reset_streams` leaves it alone).  `t`
    counts the rows pushed while the fleet moves in lockstep and equals every entry of `rows` until the first subset
    push; from then on it no longer describes the session (use `rows`) until `reset()`.  Under torch.distributed
    every rank builds one for its own shard of streams; the Recall@N counters are all-reduced like `step`'s.

    `track_pr` (any of "place", "query", "multi") also accumulates createPR's precision-recall curve of the session
    on the GPU, push by push, in bounded memory: see `session_precision_recall`.  The "place" accumulator holds
    4 bytes per (stream, place), the other two 1 MB each."""

    def __init__(self, W_feat, W_out, roi, k, T, L, n_streams, n_top=25, ns=ops.RECALL_NS, device=None,
                 mode=MODE_AUTO, track_pr=()):
        super().__init__(W_feat, W_out, roi, k, T, L, n_top=n_top, ns=ns, max_streams=n_streams, device=device,
                         mode=mode)
        self.n_streams = int(n_streams)
        if self.L < 1 or self.L > self.net.P:
            raise LensError(f"need 1 <= L <= P={self.net.P}, got L={self.L}")
        track_pr = (track_pr,) if isinstance(track_pr, str) else tuple(track_pr)
        unknown = set(track_pr) - set(ops.SEQPR_STREAM_MODES)
        if unknown:
            raise LensError(f"track_pr takes modes from {ops.SEQPR_STREAM_MODES}, got {sorted(unknown)}")
        # never read before it is written (a row is used only once its stream has seen it): left uninitialised
        self.ring = (torch.empty((self.n_streams, self.L - 1, self.net.P), dtype=torch.float32, device=self.device)
                     if self.L > 1 else None)
        self.seen = torch.zeros((self.n_streams,), dtype=torch.int32, device=self.device)
        self.t = 0
        # per-stream row counters: kept by the indexed kernels once a push has carried a subset of the streams (the
        # session is then no longer lockstep); until then every stream has t rows and the lockstep kernels run
        self._rows = torch.zeros((self.n_streams,), dtype=torch.int64, device=self.device)
        self._indexed = False
        self._all_ids = None
        # session accumulators of the tracked precision-recall modes (zeroed = empty session)
        self._pr_acc = {m: torch.zeros((ops.seqpr_stream_bytes(self.n_streams, self.net.P, self.L, i),),
                                       dtype=torch.uint8, device=self.device)
                        for i, m in enumerate(ops.SEQPR_STREAM_MODES) if m in track_pr}

    @property
    def rows(self):
        """i64 [n_streams] on the device: rows pushed to each stream since construction or `reset()`."""
        if not self._indexed:
            self._rows.fill_(self.t)
        return self._rows

    def _check_streams(self, B):
        if B != self.n_streams:
            raise LensError(f"this pipeline serves {self.n_streams} streams; the push has {B}")

    def _check_gt(self, gt_center, Q, gt_tol, n=None):
        n = self.n_streams if n is None else n
        if self._pr_acc and n and (gt_center is None or gt_tol < 0):
            raise LensError(f"precision-recall tracking ({', '.join(self._pr_acc)}) needs gt_center and gt_tol >= 0 "
                            "on every push")
        if gt_center is not None and (not torch.is_tensor(gt_center) or gt_center.dtype != torch.int32
                                      or tuple(gt_center.shape) != (n, Q)):
            raise LensError(f"gt_center must be i32 [{n}, {Q}]")

    def _stream_indices(self, streams):
        """A bool mask [n_streams] or integer stream indices (a host sequence, numpy array or tensor) -> list of int
        indices in [0, n_streams): the indices in the order given, or the mask's True entries in ascending order."""
        if isinstance(streams, np.ndarray):
            streams = torch.from_numpy(streams)
        is_tensor = torch.is_tensor(streams)
        items = streams.reshape(-1).tolist() if is_tensor else list(streams)
        if (streams.dtype == torch.bool) if is_tensor else (items and all(isinstance(v, bool) for v in items)):
            if len(items) != self.n_streams:
                raise LensError(f"a mask must have {self.n_streams} entries, got {len(items)}")
            return [b for b, v in enumerate(items) if v]
        if (is_tensor and (streams.dtype == torch.uint8 or streams.dtype.is_floating_point)) or \
                any(isinstance(v, bool) or not isinstance(v, int) for v in items):
            raise LensError("give a bool mask or integer stream indices (a u8 tensor is ambiguous)")
        if any(v < 0 or v >= self.n_streams for v in items):
            raise LensError(f"stream indices must lie in [0, {self.n_streams})")
        return items

    def _offline(self, *args, **kwargs):
        # the batch entry points advance the SNN state without the sequence history (and a different stream count
        # would recreate the handle): on a live session they would silently mix two timelines
        raise LensError("StreamingPipeline is a live session: feed it with push / push_events "
                        "(use an InferencePipeline for batch steps)")

    step = step_events = step_event_groups = step_host = _offline

    def precision_recall(self, *args, **kwargs):
        # the batch method needs whole sequences, and a push's S holds only the new rows
        raise LensError("StreamingPipeline is a live session: construct it with track_pr=(...) and call "
                        "session_precision_recall for the curve of the rows pushed so far")

    def push(self, frames=None, pooled=None, gt_center=None, gt_tol=0, reduce=True, streams=None):
        """Q new windows of every stream: frames u8 [B, Q, roi, roi] or pooled u8 [B, Q, I], B = n_streams.
        -> `step`'s dict with top_val / top_idx [B, Q, N] (row q = the sequence ending at new row q), S [B, Q, P],
        and hits / n_valid for this push.  gt_center i32 [B, Q] (optional; required with track_pr) is the expected
        place of the sequence ending at each new row (band ground truth, |idx - center| <= gt_tol, -1 = none);
        warm-up rows never count.  With track_pr the valid new rows also join the precision-recall session; what
        the push returns is the same as without tracking.

        `streams` (a bool mask [n_streams] or distinct integer indices, as a host sequence, numpy array or CPU
        tensor, in any order, possibly empty) makes it a push of those streams only: row i of frames / pooled /
        gt_center and of the results belongs to stream streams[i] (a mask: its True entries in ascending order), B =
        their number.  Each of them advances exactly as in a lockstep push of that one stream; every other stream
        keeps its SNN state, ring rows, seen, row counter and precision-recall records.  An empty push may omit
        frames / pooled (and gt_center, also with track_pr) and launches no kernel of this library; under
        torch.distributed with reduce=True, a rank with nothing to push calls it so that it takes part in the
        all-reduce of the counters."""
        x = frames if frames is not None else pooled
        if frames is not None and pooled is not None:
            raise LensError("give exactly one of frames / pooled")
        if streams is None:
            if x is None:
                raise LensError("give exactly one of frames / pooled")
            self._check_streams(x.shape[0])
            self._check_gt(gt_center, x.shape[1], gt_tol)
            if self._indexed:
                return self._push_ids(frames, pooled, None, gt_center, gt_tol, reduce)
            with torch.cuda.device(self.device):
                S = self.similarity(frames=frames, pooled=pooled)
                if self._pr_acc:      # before the match, which advances seen and overwrites ring slots
                    ops.seqpr_stream_accumulate(S, self.L, self.ring, self.seen, self.t, gt_center, gt_tol,
                                                **{"acc_" + m: a for m, a in self._pr_acc.items()})
                tv, ti = ops.seqmatch_topk_stream(S, self.L, self.n_top, self.ring, self.seen, self.t)
                self.t += S.shape[1]
            return self._finish(S, tv, ti, gt_center, gt_tol, reduce)
        ids = self._stream_indices(streams)
        if len(set(ids)) != len(ids):
            raise LensError("a push names every stream at most once")
        n = len(ids)
        if x is None and n:
            raise LensError("give exactly one of frames / pooled")
        if x is not None and x.shape[0] != n:
            raise LensError(f"the push names {n} streams but carries rows for {x.shape[0]}")
        if n == 0:
            return self._push_none(x.shape[1] if x is not None else None, gt_center, reduce)
        self._check_gt(gt_center, x.shape[1], gt_tol, n)
        net = self.net
        want = (n, x.shape[1], net.I) if pooled is not None else (n, x.shape[1], net.roi, net.roi)
        if not torch.is_tensor(x) or not x.is_cuda or x.dtype != torch.uint8 or tuple(x.shape) != want:
            raise LensError(f"{'pooled' if pooled is not None else 'frames'} must be a u8 CUDA tensor {list(want)}")
        return self._push_ids(frames, pooled, ids, gt_center, gt_tol, reduce)

    def _push_ids(self, frames, pooled, ids, gt_center, gt_tol, reduce):
        """The push on the indexed kernels: ids = the pushing streams (host list), None = all of them in order."""
        with torch.cuda.device(self.device):
            if not self._indexed:                  # the session leaves lockstep: every stream has t rows so far
                self._rows.fill_(self.t)
                self._indexed = True
            if ids is None:
                if self._all_ids is None:
                    self._all_ids = torch.arange(self.n_streams, dtype=torch.int32, device=self.device)
                dev_ids = self._all_ids
                S = self.similarity(frames=frames, pooled=pooled)
            else:
                dev_ids = torch.tensor(ids, dtype=torch.int32).pin_memory().to(self.device, non_blocking=True)
                if pooled is None:
                    n, Q = frames.shape[:2]
                    pooled = ops.pool_frames(frames.reshape(n * Q, self.net.roi, self.net.roi),
                                             self.net.k).reshape(n, Q, self.net.I)
                S = self.net.run_streams_ids(pooled, dev_ids, mode=self.mode)
            if self._pr_acc:          # before the match, which advances seen / rows and overwrites ring slots
                ops.seqpr_stream_accumulate_ids(S, self.L, dev_ids, self.ring, self.seen, self._rows, gt_center, gt_tol,
                                                **{"acc_" + m: a for m, a in self._pr_acc.items()})
            tv, ti = ops.seqmatch_topk_stream_ids(S, self.L, self.n_top, dev_ids, self.ring, self.seen, self._rows)
        return self._finish(S, tv, ti, gt_center, gt_tol, reduce)

    def _push_none(self, Q, gt_center, reduce):
        """A push that carries no stream (Q windows each; None: as gt_center says, else 0): empty results, zero
        counters when the other ranks count (gt_center given or precision-recall tracked)."""
        if gt_center is not None and (not torch.is_tensor(gt_center) or gt_center.dtype != torch.int32
                                      or gt_center.dim() != 2 or gt_center.shape[0] != 0
                                      or (Q is not None and gt_center.shape[1] != Q)):
            raise LensError("gt_center of an empty push must be i32 [0, Q]")
        if Q is None:
            Q = gt_center.shape[1] if gt_center is not None else 0
        dev = self.device
        out = dict(top_val=torch.empty((0, Q, self.n_top), dtype=torch.float32, device=dev),
                   top_idx=torch.empty((0, Q, self.n_top), dtype=torch.int32, device=dev), D=None, hits=None,
                   n_valid=None, S=torch.empty((0, Q, self.net.P), dtype=torch.float32, device=dev),
                   overflow=self.net.overflow_tensor())
        if gt_center is not None or self._pr_acc:
            out["hits"] = torch.zeros((len(self.ns),), dtype=torch.int64, device=dev)
            out["n_valid"] = torch.zeros((1,), dtype=torch.int64, device=dev)
        if reduce:
            self._all_reduce_hits(out)
        return out

    def _finish(self, S, tv, ti, gt_center, gt_tol, reduce):
        with torch.cuda.device(self.device):
            out = dict(top_val=tv, top_idx=ti, D=None, hits=None, n_valid=None, S=S,
                       overflow=self.net.overflow_tensor())
            if gt_center is not None:
                gt = torch.where(ti[..., 0] >= 0, gt_center, -1)      # warm-up rows: no ground truth
                out["hits"], out["n_valid"] = ops.recall_counts(ti, S.shape[2] - self.L + 1, gt_center=gt,
                                                                gt_tol=gt_tol, ns=self.ns)
        if reduce:
            self._all_reduce_hits(out)
        return out

    def push_events(self, t_us, x, y, offsets, t0_us, window_us, Q, roi_x0=0, roi_y0=0, gt_center=None, gt_tol=0,
                    reduce=True, streams=None):
        """`push` fed from raw events: the next Q windows of every stream, window q of stream b covering
        [t0_us[b] + q * window_us, + window_us) of its events [offsets[b], offsets[b+1]) (as in `step_events`).
        Returns `push`'s dict plus "events_per_window" i32 [B, Q].  With `streams` (as in `push`), offsets / t0_us
        describe the pushing streams in that order, B = their number."""
        if streams is None:
            self._check_streams(offsets.numel() - 1)
            self._check_gt(gt_center, int(Q), gt_tol)
        else:
            ids = self._stream_indices(streams)
            if len(set(ids)) != len(ids):
                raise LensError("a push names every stream at most once")
            if offsets.numel() - 1 != len(ids):
                raise LensError(f"the push names {len(ids)} streams but offsets describe {offsets.numel() - 1}")
            if not ids:
                out = self._push_none(int(Q), gt_center, reduce)
                out["events_per_window"] = torch.empty((0, int(Q)), dtype=torch.int32, device=self.device)
                return out
            self._check_gt(gt_center, int(Q), gt_tol, len(ids))
            streams = ids
        with torch.cuda.device(self.device):
            pooled, n_ev = self._bin_streams(t_us, x, y, offsets, t0_us, window_us, Q, roi_x0, roi_y0)
            out = self.push(pooled=pooled, gt_center=gt_center, gt_tol=gt_tol, reduce=reduce, streams=streams)
        out["events_per_window"] = n_ev
        return out

    def reset_streams(self, streams):
        """Restart some streams (a camera that rebooted or dropped out): their SNN state and their sequence
        history.  `streams` is a bool mask [n_streams] (tensor or sequence of bools) or integer stream indices
        (tensor, numpy array or sequence).  Their next L - 1 rows are warm-up rows again; the other streams are
        untouched.  Row counters (`rows`) are not reset."""
        mask = torch.zeros((self.n_streams,), dtype=torch.bool)
        mask[torch.tensor(self._stream_indices(streams), dtype=torch.int64)] = True
        with torch.cuda.device(self.device):
            mask = mask.to(self.device)
            self.net.reset_streams(mask)
            self.seen.masked_fill_(mask, 0)

    def reset(self):
        """Every stream from scratch: SNN state (and the overflow counter), sequence history, t and rows (the fleet is
        in lockstep again), and a new precision-recall session."""
        self.net.reset_states()
        self.seen.zero_()
        self.t = 0
        self._indexed = False
        self.reset_precision_recall()

    def reset_precision_recall(self):
        """Start a new precision-recall session; streams, ring and t are left alone.  (`reset_streams` does not
        start one: a restarted stream's later valid rows are more columns of the same session.)"""
        for acc in self._pr_acc.values():
            acc.zero_()

    def session_precision_recall(self, matching="single", best="place", n_thresh=100, reduce=True):
        """createPR's precision-recall lists over every valid row pushed since construction, `reset()` or
        `reset_precision_recall()`, in the format of InferencePipeline.precision_recall: dict(P, R, tp, fp, gtp).

        A stream's session matrix has its valid rows as query columns, in push order; the fleet (and, under
        torch.distributed with reduce=True, every rank) concatenates along createPR's column axis.  For a fresh
        pipeline without stream resets the result equals `precision_recall` of one batch step over all the windows,
        with gt_center[:, L - 1:].  The mode (matching / best as in `precision_recall`) must be tracked.  Raises
        LensError for an untracked mode, an empty session, or spike counts whose sequence sums are not integers in
        [0, 65 535].  Under torch.distributed: one all-reduce SUM of about 1 MB."""
        from .src.metrics import pr_lists
        mode = ops.seqpr_mode(matching, best)
        name = ops.SEQPR_STREAM_MODES[mode]
        if name not in self._pr_acc:
            raise LensError(f"precision-recall mode {name!r} is not tracked: construct the pipeline with "
                            f"track_pr=({name!r}, ...)")
        if not 2 <= n_thresh <= ops.SEQPR_MAX_THRESH:
            raise ValueError(f"n_thresh must be in [2, {ops.SEQPR_MAX_THRESH}], got {n_thresh}")
        dist = torch.distributed
        shared = reduce and dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1
        with torch.cuda.device(self.device):
            packed = ops.seqpr_stream_histogram(self._pr_acc[name], self.n_streams, self.net.P, self.L, mode)
            if shared:
                dist.all_reduce(packed)                     # [hist, gtp, n_bad]
            tp, fp, gtp = ops.seqpr_stream_counts(packed, self.L, n_thresh)
        P, R = pr_lists(tp, fp, gtp)
        return dict(P=P, R=R, tp=tp, fp=fp, gtp=gtp)


class PlaceShardedPipeline:
    """The same hot path with the DATABASE sharded across ranks instead of the streams (SURVEY.md 8e, the
    alternative for few streams / very large databases): every rank runs ALL streams against its own range
    of places (output layer is column-parallel; the tiny feature layer is replicated), ranks them locally,
    and the per-rank top-N lists are all-gathered (NCCL) and merged on the GPU (lens_topn_merge).  The merged
    lists equal the single-GPU lists bit for bit: the order (value desc, place index desc) is global."""

    def __init__(self, W_feat, W_out, roi, k, T, L, n_top=25, ns=ops.RECALL_NS, max_streams=1, device=None,
                 mode=MODE_AUTO, rank=None, world=None):
        import torch.distributed as dist
        self.dist = dist if (dist.is_available() and dist.is_initialized()) else None
        self.rank = rank if rank is not None else (self.dist.get_rank() if self.dist else 0)
        self.world = world if world is not None else (self.dist.get_world_size() if self.dist else 1)
        self.P = int(W_out.shape[0])
        self.L, self.n_top, self.ns, self.mode = int(L), int(n_top), tuple(ns), mode
        self.p0, self.p1, p1h = place_shard_range(self.P, self.L, self.rank, self.world)
        self.net = B200Network(W_feat, W_out[self.p0:p1h], roi=roi, k=k, num_timesteps=T, max_streams=max_streams,
                               device=device)
        self.device = self.net.device

    def step(self, frames=None, pooled=None, gt_center=None, gt_tol=0):
        """-> dict(top_val, top_idx (global place indices), hits, n_valid); every rank holds the merged result."""
        S = self.net.run_streams(frames=frames, pooled=pooled, mode=self.mode)       # [B, Q, local places + halo]
        tv, ti, _ = ops.seqmatch_topk(S, self.L, self.n_top)
        ti = torch.where(ti >= 0, ti + self.p0, ti)
        if self.world > 1:
            allv = torch.empty((self.world,) + tuple(tv.shape), dtype=tv.dtype, device=tv.device)
            alli = torch.empty((self.world,) + tuple(ti.shape), dtype=ti.dtype, device=ti.device)
            self.dist.all_gather_into_tensor(allv, tv.contiguous())
            self.dist.all_gather_into_tensor(alli, ti.contiguous())
        else:
            allv, alli = tv[None], ti[None]
        tv, ti = ops.topn_merge(allv, alli)
        out = dict(top_val=tv, top_idx=ti, hits=None, n_valid=None)
        if gt_center is not None:
            out["hits"], out["n_valid"] = ops.recall_counts(ti, self.P - self.L + 1, gt_center=gt_center,
                                                            gt_tol=gt_tol, ns=self.ns)
        return out
