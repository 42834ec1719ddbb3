"""Host-side wrappers of the C ABI (torch tensors in, torch tensors out).

PyTorch is used for device memory and streams only; every computation happens in
liblens_b200.so (hand-written sm_100a kernels).  All wrappers are asynchronous on
torch's current CUDA stream.
"""
import ctypes as C

import torch

from . import _lib
from ._lib import check, ptr, stream_ptr, require_cuda

RECALL_NS = (1, 5, 10, 15, 20, 25)   # lens/run_model.py:266


def pool_geometry(roi, k):
    """dims and centre index of the one-hot strided conv (lens/run_model.py:130-137)."""
    dims = roi // k
    c = (k // 2) - 1
    if c < 0:
        c += k
    return dims, c


def pool_frames(frames, k):
    """frames u8 [n, roi, roi] -> pooled u8 [n, dims*dims] (pixel pick of run_model.py:130-137)."""
    require_cuda(frames)
    assert frames.dtype == torch.uint8 and frames.dim() == 3 and frames.shape[1] == frames.shape[2]
    n, roi, _ = frames.shape
    dims, _ = pool_geometry(roi, k)
    out = torch.empty((n, dims * dims), dtype=torch.uint8, device=frames.device)
    check(_lib.lib().lens_pool_frames(ptr(frames), n, roi, k, ptr(out), stream_ptr()), "lens_pool_frames")
    return out


def bin_events(t_us, x, y, t0_us, window_us, n_win, roi, k, roi_x0=0, roi_y0=0, index_shift=1,
               wrap_u8=True, want_frames=True, want_pooled=True, check_sorted=False):
    """Event stream -> (frames u8 [n_win, roi, roi], pooled u8 [n_win, I], events-per-window i32).

    Mirrors lens/collect_data.py:186-202 (`frame[y-1, x-1] += 1`, `.astype(np.uint8)`); the
    caller drops windows whose count is 0 to reproduce create_images' "No events" branch.
    t_us must be ascending (window ranges are found by binary search); check_sorted=True verifies it with
    one extra pass over t_us (lens_check_sorted_u32, synchronises) and raises ValueError otherwise.
    """
    require_cuda(t_us, x, y)
    assert t_us.dtype == torch.int32 or t_us.dtype == torch.uint32
    assert x.dtype in (torch.int16, torch.uint16) and y.dtype in (torch.int16, torch.uint16)
    n = t_us.numel()
    dev = t_us.device
    if check_sorted:
        flag = torch.zeros(1, dtype=torch.int32, device=dev)
        check(_lib.lib().lens_check_sorted_u32(ptr(t_us), n, ptr(flag), stream_ptr()), "lens_check_sorted_u32")
        if int(flag.item()):
            raise ValueError("event timestamps must be ascending")
    dims, _ = pool_geometry(roi, k)
    frames = torch.empty((n_win, roi, roi), dtype=torch.uint8, device=dev) if want_frames else None
    pooled = torch.empty((n_win, dims * dims), dtype=torch.uint8, device=dev) if want_pooled else None
    cnt = torch.empty((n_win,), dtype=torch.int32, device=dev)
    offs = torch.empty((n_win + 1,), dtype=torch.int64, device=dev)
    check(_lib.lib().lens_bin_events(ptr(t_us), ptr(x), ptr(y), n, t0_us, window_us, roi_x0, roi_y0,
                                     roi, k, index_shift, int(wrap_u8), ptr(frames), ptr(pooled),
                                     ptr(cnt), ptr(offs), n_win, stream_ptr()), "lens_bin_events")
    return frames, pooled, cnt


def bin_event_streams(t_us, x, y, offsets, t0_us, window_us, Q, roi, k, roi_x0=0, roi_y0=0, index_shift=1,
                      wrap_u8=True, want_frames=False, want_pooled=True, check_sorted=False):
    """B independent event streams in one call -> (frames u8 [B, Q, roi, roi], pooled u8 [B, Q, I],
    events-per-window i32 [B, Q]); frames / pooled are None unless wanted.

    Stream b is events [offsets[b], offsets[b+1]) of t_us / x / y (offsets i64 [B + 1] on the device) and
    its window q covers [t0_us[b] + q * window_us, t0_us[b] + (q + 1) * window_us) (t0_us i32 / u32 [B]).
    Per stream the results equal `bin_events` on that stream's events with t0_us[b].  t_us must be ascending
    within every stream; check_sorted=True verifies that and the offsets (one extra pass over t_us,
    lens_check_sorted_segments_u32, synchronises) and raises ValueError before binning.
    """
    require_cuda(t_us, x, y, offsets, t0_us)
    assert t_us.dtype in (torch.int32, torch.uint32) and t0_us.dtype in (torch.int32, torch.uint32)
    assert x.dtype in (torch.int16, torch.uint16) and y.dtype in (torch.int16, torch.uint16)
    assert offsets.dtype == torch.int64 and offsets.dim() == 1 and offsets.numel() >= 1
    B, Q, n = offsets.numel() - 1, int(Q), t_us.numel()
    assert t0_us.shape == (B,) and x.numel() == n and y.numel() == n
    dev = t_us.device
    if check_sorted:
        flag = torch.zeros(1, dtype=torch.int32, device=dev)
        check(_lib.lib().lens_check_sorted_segments_u32(ptr(t_us), n, ptr(offsets), B, ptr(flag), stream_ptr()),
              "lens_check_sorted_segments_u32")
        if int(flag.item()):
            raise ValueError("event timestamps must be ascending within every stream, and offsets non-decreasing "
                             "inside [0, n_events]")
    dims, _ = pool_geometry(roi, k)
    frames = torch.empty((B, Q, roi, roi), dtype=torch.uint8, device=dev) if want_frames else None
    pooled = torch.empty((B, Q, dims * dims), dtype=torch.uint8, device=dev) if want_pooled else None
    cnt = torch.empty((B, Q), dtype=torch.int32, device=dev)
    offs = torch.empty((max(B, 1), Q + 1), dtype=torch.int64, device=dev)   # never NULL, even for B = 0
    check(_lib.lib().lens_bin_event_streams(ptr(t_us), ptr(x), ptr(y), n, ptr(offsets), ptr(t0_us), B, Q, window_us,
                                            roi_x0, roi_y0, roi, k, index_shift, int(wrap_u8), ptr(frames),
                                            ptr(pooled), ptr(cnt), ptr(offs), stream_ptr()), "lens_bin_event_streams")
    return frames, pooled, cnt


def seqmatch_topk(S, L, N=25, want_D=False):
    """S f32 [B, Q, P] -> (top_val [B, Qo, N], top_idx [B, Qo, N], D [B, Po, Qo] or None).

    lens/run_model.py:248-254 + the selection of lens/src/metrics.py:218.
    """
    require_cuda(S)
    assert S.dtype == torch.float32 and S.dim() == 3
    B, Q, P = S.shape
    Qo, Po = Q - L + 1, P - L + 1
    D = torch.empty((B, Po, Qo), dtype=torch.float32, device=S.device) if want_D else None
    tv = torch.empty((B, Qo, N), dtype=torch.float32, device=S.device)
    ti = torch.empty((B, Qo, N), dtype=torch.int32, device=S.device)
    check(_lib.lib().lens_seqmatch_topk(ptr(S), B, Q, P, L, N, ptr(D), ptr(tv), ptr(ti), stream_ptr()),
          "lens_seqmatch_topk")
    return tv, ti, D


def seqmatch_topk_stream(S, L, N, ring, seen, t):
    """Sequence matching across calls: S f32 [B, Q, P] = the Q new rows of B streams in lockstep ->
    (top_val [B, Q, N], top_idx [B, Q, N]); row q is the top-N of the sequence that ends at new row q, -inf / -1
    while its stream has seen fewer than L rows since its reset.

    ring f32 [B, L - 1, P] (None iff L == 1) and seen i32 [B] are the caller's device state, updated in place (the
    last L - 1 rows and the rows seen since each stream's reset, saturating at L - 1); t = rows pushed before this
    call.  See lens_seqmatch_topk_stream in include/lens_b200.h."""
    require_cuda(S, ring, seen)
    assert S.dtype == torch.float32 and S.dim() == 3 and seen.dtype == torch.int32
    B, Q, P = S.shape
    assert seen.shape == (B,) and (ring is None or (ring.dtype == torch.float32 and ring.shape == (B, L - 1, P)))
    tv = torch.empty((B, Q, N), dtype=torch.float32, device=S.device)
    ti = torch.empty((B, Q, N), dtype=torch.int32, device=S.device)
    check(_lib.lib().lens_seqmatch_topk_stream(ptr(S), B, Q, P, L, N, ptr(ring), ptr(seen), int(t), ptr(tv), ptr(ti),
                                               stream_ptr()), "lens_seqmatch_topk_stream")
    return tv, ti


def seqmatch_topk_stream_ids(S, L, N, ids, ring, seen, rows):
    """seqmatch_topk_stream for any subset of a fleet of B streams, in any order: S f32 [n, Q, P] = the Q new rows of
    the streams ids i32 [n] (device, distinct, in [0, B)) -> (top_val [n, Q, N], top_idx [n, Q, N]) by position.

    ring f32 [B, L - 1, P] (None iff L == 1), seen i32 [B] and rows i64 [B] (rows pushed to each stream, which replaces
    the scalar t) are the fleet's device state, updated in place for the pushed streams only.  See
    lens_seqmatch_topk_stream_ids in include/lens_b200.h."""
    require_cuda(S, ids, ring, seen, rows)
    assert S.dtype == torch.float32 and S.dim() == 3 and seen.dtype == torch.int32 and rows.dtype == torch.int64
    n, Q, P = S.shape
    B = seen.shape[0]
    assert ids.dtype == torch.int32 and ids.shape == (n,) and seen.shape == (B,) and rows.shape == (B,)
    assert ring is None or (ring.dtype == torch.float32 and ring.shape == (B, L - 1, P))
    tv = torch.empty((n, Q, N), dtype=torch.float32, device=S.device)
    ti = torch.empty((n, Q, N), dtype=torch.int32, device=S.device)
    check(_lib.lib().lens_seqmatch_topk_stream_ids(ptr(S), n, Q, P, L, N, ptr(ids), B, ptr(ring), ptr(seen), ptr(rows),
                                                   ptr(tv), ptr(ti), stream_ptr()), "lens_seqmatch_topk_stream_ids")
    return tv, ti


def recall_counts(top_idx, Po, gt_dense=None, gt_center=None, gt_tol=0, ns=RECALL_NS,
                  hits=None, n_valid=None):
    """Accumulate Recall@N hit counters (device int64) for top_idx [B, Qo, N].

    gt_dense: u8 [Po, Qo] (shared by all streams) or [B, Po, Qo]; or gt_center i32 [B, Qo].
    Returns (hits [len(ns)] i64, n_valid [1] i64) on the device.
    """
    require_cuda(top_idx, gt_dense, gt_center)
    B, Qo, N = top_idx.shape
    dev = top_idx.device
    if hits is None:
        hits = torch.zeros((len(ns),), dtype=torch.int64, device=dev)
    if n_valid is None:
        n_valid = torch.zeros((1,), dtype=torch.int64, device=dev)
    stride = 0
    if gt_dense is not None:
        assert gt_dense.dtype == torch.uint8
        if gt_dense.dim() == 3:
            assert gt_dense.shape == (B, Po, Qo)
            stride = Po * Qo
        else:
            assert gt_dense.shape == (Po, Qo)
    if gt_center is not None:
        assert gt_center.dtype == torch.int32 and gt_center.shape == (B, Qo)
    ns_arr = (C.c_int * len(ns))(*ns)
    check(_lib.lib().lens_recall(ptr(top_idx), B, Qo, Po, N, ptr(gt_dense), stride, ptr(gt_center),
                                 gt_tol, ns_arr, len(ns), ptr(hits), ptr(n_valid), stream_ptr()),
          "lens_recall")
    return hits, n_valid


SEQPR_MODES = {("single", "place"): 0, ("single", "query"): 1, ("multi", None): 2}   # LENS_SEQPR_*
SEQPR_MAX_THRESH = 4096


def seqpr_mode(matching, best="place"):
    """createPR's matching ('single' with best='place' or 'query', or 'multi') -> LENS_SEQPR_* mode."""
    key = (matching, best if matching == "single" else None)
    if key not in SEQPR_MODES:
        raise ValueError(f"matching must be 'single' (best='place' or 'query') or 'multi', got {matching!r}, "
                         f"best={best!r}")
    return SEQPR_MODES[key]


def _seqpr_check(S, L, mode, gt_dense, gt_center, n_thresh=2):
    """Shape and value checks of the fleet precision-recall calls (before anything touches the device)."""
    if not torch.is_tensor(S) or S.dtype != torch.float32 or S.dim() != 3:
        raise ValueError("S must be f32 [B, Q, P]")
    B, Q, P = S.shape
    if not 1 <= L <= min(Q, P):
        raise ValueError(f"need 1 <= L <= min(Q, P) = {min(Q, P)}, got L={L}")
    if mode not in SEQPR_MODES.values():
        raise ValueError(f"unknown mode {mode}")
    if not 2 <= n_thresh <= SEQPR_MAX_THRESH:
        raise ValueError(f"n_thresh must be in [2, {SEQPR_MAX_THRESH}], got {n_thresh}")
    Qo, Po = Q - L + 1, P - L + 1
    if (gt_dense is None) == (gt_center is None):
        raise ValueError("give exactly one of gt_dense / gt_center")
    if gt_dense is not None and (gt_dense.dtype != torch.uint8 or tuple(gt_dense.shape) not in ((Po, Qo), (B, Po, Qo))):
        raise ValueError(f"gt_dense must be u8 [{Po}, {Qo}] or [{B}, {Po}, {Qo}], got {tuple(gt_dense.shape)}")
    if gt_center is not None and (gt_center.dtype != torch.int32 or tuple(gt_center.shape) != (B, Qo)):
        raise ValueError(f"gt_center must be i32 [{B}, {Qo}], got {tuple(gt_center.shape)}")
    return B, Q, P, (Po * Qo if gt_dense is not None and gt_dense.dim() == 3 else 0)


def seqpr_scan(S, L, mode, gt_dense=None, gt_center=None, gt_tol=0, extremes=None, gtp=None):
    """Scan pass of the fleet precision-recall (lens_seqpr_scan): S f32 [B, Q, P] spike counts, ground truth as in
    `recall_counts`.  -> (records u8 [bytes] or None, extremes i64 [2], gtp i64 [1]) on the device.  extremes
    ({max, ~min} as order-preserving keys) are merged by max and gtp accumulated, so passing the tensors of an
    earlier scan makes one fleet of both groups of streams."""
    B, Q, P, stride = _seqpr_check(S, L, mode, gt_dense, gt_center)
    require_cuda(S, gt_dense, gt_center, extremes, gtp)
    nbytes = C.c_int64(0)
    check(_lib.lib().lens_seqpr_records_bytes(B, Q, P, L, mode, C.byref(nbytes)), "lens_seqpr_records_bytes")
    records = torch.empty((nbytes.value,), dtype=torch.uint8, device=S.device) if nbytes.value else None
    if extremes is None:
        extremes = torch.zeros((2,), dtype=torch.int64, device=S.device)
    if gtp is None:
        gtp = torch.zeros((1,), dtype=torch.int64, device=S.device)
    check(_lib.lib().lens_seqpr_scan(ptr(S), B, Q, P, L, mode, ptr(gt_dense), stride, ptr(gt_center), int(gt_tol),
                                     ptr(records), ptr(extremes), ptr(gtp), stream_ptr()), "lens_seqpr_scan")
    return records, extremes, gtp


def seqpr_counts(S, L, mode, records, extremes, n_thresh=100, gt_dense=None, gt_center=None, gt_tol=0, tp=None,
                 fp=None):
    """Count pass (lens_seqpr_counts) with the same S / L / mode / ground truth and the scan's records, over the
    thresholds np.linspace(max, min, n_thresh) of the (merged) extremes.  -> (tp, fp) i64 [n_thresh] on the device,
    accumulated into tp / fp when given."""
    B, Q, P, stride = _seqpr_check(S, L, mode, gt_dense, gt_center, n_thresh)
    require_cuda(S, gt_dense, gt_center, records, extremes, tp, fp)
    if tp is None:
        tp = torch.zeros((n_thresh,), dtype=torch.int64, device=S.device)
    if fp is None:
        fp = torch.zeros((n_thresh,), dtype=torch.int64, device=S.device)
    check(_lib.lib().lens_seqpr_counts(ptr(S), B, Q, P, L, mode, ptr(gt_dense), stride, ptr(gt_center), int(gt_tol),
                                       ptr(records), ptr(extremes), n_thresh, ptr(tp), ptr(fp), stream_ptr()),
          "lens_seqpr_counts")
    return tp, fp


SEQPR_STREAM_BINS = 65536                      # LENS_SEQPR_STREAM_BINS: sequence sums k in [0, 65 535]
SEQPR_STREAM_MODES = ("place", "query", "multi")   # index = LENS_SEQPR_* mode


def _seqpr_stream_check(S, L, ring, seen, gt_center, accs):
    """Shape checks of seqpr_stream_accumulate (before anything touches the device)."""
    if not torch.is_tensor(S) or S.dtype != torch.float32 or S.dim() != 3:
        raise ValueError("S must be f32 [B, Q, P]")
    B, Q, P = S.shape
    if not 1 <= L <= P:
        raise ValueError(f"need 1 <= L <= P = {P}, got L={L}")
    if not torch.is_tensor(seen) or seen.dtype != torch.int32 or tuple(seen.shape) != (B,):
        raise ValueError(f"seen must be i32 [{B}]")
    if L > 1 and (ring is None or ring.dtype != torch.float32 or tuple(ring.shape) != (B, L - 1, P)):
        raise ValueError(f"ring must be f32 [{B}, {L - 1}, {P}]")
    if not torch.is_tensor(gt_center) or gt_center.dtype != torch.int32 or tuple(gt_center.shape) != (B, Q):
        raise ValueError(f"gt_center must be i32 [{B}, {Q}]")
    for mode, acc in enumerate(accs):
        if acc is not None and (acc.dtype != torch.uint8 or acc.numel() != seqpr_stream_bytes(B, P, L, mode)):
            raise ValueError(f"the {SEQPR_STREAM_MODES[mode]} accumulator must be u8 "
                             f"[{seqpr_stream_bytes(B, P, L, mode)}] (seqpr_stream_bytes)")
    return B, Q, P


def seqpr_stream_bytes(B, P, L, mode):
    """Size in bytes of one mode's session accumulator (lens_seqpr_stream_bytes); zeroed = an empty session."""
    n = C.c_int64(0)
    check(_lib.lib().lens_seqpr_stream_bytes(B, P, L, mode, C.byref(n)), "lens_seqpr_stream_bytes")
    return int(n.value)


def seqpr_stream_accumulate(S, L, ring, seen, t, gt_center, gt_tol=0, acc_place=None, acc_query=None,
                            acc_multi=None):
    """Fold the valid new rows of one push (S f32 [B, Q, P], with the ring / seen / t the push's
    seqmatch_topk_stream call is about to use) into the session accumulators of the tracked modes (u8 tensors of
    seqpr_stream_bytes, None = not tracked).  gt_center i32 [B, Q]: expected place of each new row, -1 = none."""
    accs = (acc_place, acc_query, acc_multi)
    B, Q, P = _seqpr_stream_check(S, L, ring, seen, gt_center, accs)
    require_cuda(S, ring, seen, gt_center, *accs)
    check(_lib.lib().lens_seqpr_stream_accumulate(ptr(S), B, Q, P, L, ptr(ring), ptr(seen), int(t), ptr(gt_center),
                                                  int(gt_tol), *(ptr(a) for a in accs), stream_ptr()),
          "lens_seqpr_stream_accumulate")


def seqpr_stream_accumulate_ids(S, L, ids, ring, seen, rows, gt_center, gt_tol=0, acc_place=None, acc_query=None,
                                acc_multi=None):
    """seqpr_stream_accumulate for the push of seqmatch_topk_stream_ids: S f32 [n, Q, P] and gt_center i32 [n, Q] of the
    streams ids i32 [n] of a fleet of B, with the ring / seen / rows that call is about to use; the accumulators are
    the fleet's (seqpr_stream_bytes(B, ...))."""
    accs = (acc_place, acc_query, acc_multi)
    if not torch.is_tensor(seen) or seen.dtype != torch.int32 or seen.dim() != 1:
        raise ValueError("seen must be i32 [B]")
    B = seen.shape[0]
    if not torch.is_tensor(S) or S.dtype != torch.float32 or S.dim() != 3:
        raise ValueError("S must be f32 [n, Q, P]")
    n, Q, P = S.shape
    if not torch.is_tensor(ids) or ids.dtype != torch.int32 or tuple(ids.shape) != (n,):
        raise ValueError(f"ids must be i32 [{n}]")
    if not torch.is_tensor(rows) or rows.dtype != torch.int64 or tuple(rows.shape) != (B,):
        raise ValueError(f"rows must be i64 [{B}]")
    if not 1 <= L <= P:
        raise ValueError(f"need 1 <= L <= P = {P}, got L={L}")
    if L > 1 and (ring is None or ring.dtype != torch.float32 or tuple(ring.shape) != (B, L - 1, P)):
        raise ValueError(f"ring must be f32 [{B}, {L - 1}, {P}]")
    if not torch.is_tensor(gt_center) or gt_center.dtype != torch.int32 or tuple(gt_center.shape) != (n, Q):
        raise ValueError(f"gt_center must be i32 [{n}, {Q}]")
    for mode, acc in enumerate(accs):
        if acc is not None and (acc.dtype != torch.uint8 or acc.numel() != seqpr_stream_bytes(B, P, L, mode)):
            raise ValueError(f"the {SEQPR_STREAM_MODES[mode]} accumulator must be u8 "
                             f"[{seqpr_stream_bytes(B, P, L, mode)}] (seqpr_stream_bytes)")
    require_cuda(S, ids, ring, seen, rows, gt_center, *accs)
    check(_lib.lib().lens_seqpr_stream_accumulate_ids(ptr(S), n, Q, P, L, ptr(ids), B, ptr(ring), ptr(seen), ptr(rows),
                                                      ptr(gt_center), int(gt_tol), *(ptr(a) for a in accs),
                                                      stream_ptr()), "lens_seqpr_stream_accumulate_ids")


def seqpr_stream_histogram(acc, B, P, L, mode, packed=None):
    """One mode's accumulator -> packed i64 [2 * SEQPR_STREAM_BINS + 2] on the device: the histogram of k
    (positives | negatives), then gtp and n_bad; accumulated into `packed` when given.  Summing the packed tensors
    of several ranks makes one fleet."""
    require_cuda(acc, packed)
    if packed is None:
        packed = torch.zeros((2 * SEQPR_STREAM_BINS + 2,), dtype=torch.int64, device=acc.device)
    n = 2 * SEQPR_STREAM_BINS
    check(_lib.lib().lens_seqpr_stream_histogram(ptr(acc), B, P, L, mode, ptr(packed), ptr(packed[n:n + 1]),
                                                 ptr(packed[n + 1:]), stream_ptr()), "lens_seqpr_stream_histogram")
    return packed


def seqpr_stream_counts(packed, L, n_thresh=100):
    """createPR's counts of a (summed) packed histogram -> (tp, fp) numpy i64 [n_thresh], gtp.  Raises LensError
    when a sequence sum fell outside [0, 65 535] or was not an integer (the curve would be wrong), or when the
    session has no column yet."""
    if not 2 <= n_thresh <= SEQPR_MAX_THRESH:
        raise ValueError(f"n_thresh must be in [2, {SEQPR_MAX_THRESH}], got {n_thresh}")
    require_cuda(packed)
    n = 2 * SEQPR_STREAM_BINS
    out = torch.zeros((2 * n_thresh,), dtype=torch.int64, device=packed.device)
    check(_lib.lib().lens_seqpr_hist_counts(ptr(packed), int(L), n_thresh, ptr(out[:n_thresh]), ptr(out[n_thresh:]),
                                            stream_ptr()), "lens_seqpr_hist_counts")
    host = torch.cat([out, packed[n:]]).cpu().numpy()
    tp, fp, gtp, n_bad = host[:n_thresh], host[n_thresh:2 * n_thresh], int(host[-2]), int(host[-1])
    if n_bad:
        raise _lib.LensError(f"{n_bad} sequence sums were not integers in [0, {SEQPR_STREAM_BINS - 1}]: the session "
                             "precision-recall needs integer spike counts")
    if tp[-1] + fp[-1] == 0:
        raise _lib.LensError("the precision-recall session has no valid row yet")
    return tp, fp, gtp


def topn_merge(vals, idx):
    """Global top-N from W per-shard lists: vals f32 / idx i32 [W, B, Qo, N] (idx = global place index, -1 =
    empty) -> (val [B, Qo, N], idx [B, Qo, N]) under the order (value desc, place index desc)."""
    require_cuda(vals, idx)
    assert vals.dtype == torch.float32 and idx.dtype == torch.int32 and vals.shape == idx.shape and vals.dim() == 4
    vals, idx = vals.contiguous(), idx.contiguous()
    W, B, Qo, N = vals.shape
    ov = torch.empty((B, Qo, N), dtype=torch.float32, device=vals.device)
    oi = torch.empty((B, Qo, N), dtype=torch.int32, device=vals.device)
    check(_lib.lib().lens_topn_merge(ptr(vals), ptr(idx), W, B * Qo, N, ptr(ov), ptr(oi), stream_ptr()),
          "lens_topn_merge")
    return ov, oi


def recall_bounds(D, gt_dense, ns=RECALL_NS):
    """Tie-aware (lo, hi, n_valid) hit counters of Recall@N over every order of equal similarities.

    D f32 [Po, Qo], gt_dense u8 [Po, Qo] (rows = database) -> (lo [len(ns)] i64, hi, n_valid [1]) on the device;
    lo / n_valid <= the reference's recallAtK (numpy's unstable argsort, metrics.py:218) <= hi / n_valid."""
    require_cuda(D, gt_dense)
    assert D.dtype == torch.float32 and gt_dense.dtype == torch.uint8 and D.shape == gt_dense.shape and D.dim() == 2
    D, gt_dense = D.contiguous(), gt_dense.contiguous()
    Po, Qo = D.shape
    lo = torch.zeros((len(ns),), dtype=torch.int64, device=D.device)
    hi = torch.zeros((len(ns),), dtype=torch.int64, device=D.device)
    n_valid = torch.zeros((1,), dtype=torch.int64, device=D.device)
    ns_arr = (C.c_int * len(ns))(*ns)
    check(_lib.lib().lens_recall_bounds(ptr(D), ptr(gt_dense), Po, Qo, ns_arr, len(ns), ptr(lo), ptr(hi), ptr(n_valid),
                                        stream_ptr()), "lens_recall_bounds")
    return lo, hi, n_valid


def sad_matrix(query_frames, reference_frames):
    """u8 [Q, npix], u8 [R, npix] -> L1 distances f32 [Q, R] (torch.cdist(a, b, 1) of lens/src/sad.py:38)."""
    require_cuda(query_frames, reference_frames)
    assert query_frames.dtype == torch.uint8 and reference_frames.dtype == torch.uint8
    Q, npix = query_frames.shape
    R = reference_frames.shape[0]
    assert reference_frames.shape[1] == npix
    dist = torch.empty((Q, R), dtype=torch.float32, device=query_frames.device)
    check(_lib.lib().lens_sad_matrix(ptr(query_frames), ptr(reference_frames), Q, R, npix, ptr(dist), stream_ptr()),
          "lens_sad_matrix")
    return dist


def reciprocal(x):
    """1 / x elementwise in IEEE fp32 (numpy's `1 / dist_matrix_seq`, lens/src/sad.py:52,62)."""
    require_cuda(x)
    assert x.dtype == torch.float32
    out = torch.empty_like(x)
    check(_lib.lib().lens_reciprocal(ptr(x), x.numel(), ptr(out), stream_ptr()), "lens_reciprocal")
    return out


def event_windows(t, x, y, lut, use_first_event, start, interval, max_windows, check_sorted=True):
    """Frame index ranges of the event-driven representation (lens/tools/dvstools.py:286-349).

    t f64 [n] seconds ascending, x / y 16-bit [n], lut i16 [H, W] (-2 hot pixel, -1 unused, >= 0 slot).
    -> (win_begin i64 [max_windows], win_end i64, win_t0 f64, n_windows i64 [1]); raises if t is unsorted."""
    require_cuda(t, x, y, lut)
    assert t.dtype == torch.float64 and x.dtype in (torch.int16, torch.uint16) and y.dtype == x.dtype
    assert lut.dtype == torch.int16 and lut.dim() == 2
    n = t.numel()
    H, W = lut.shape
    dev = t.device
    nw = max(int(max_windows), 0)
    wb = torch.empty(max(nw, 1), dtype=torch.int64, device=dev)
    we = torch.empty(max(nw, 1), dtype=torch.int64, device=dev)
    wt = torch.empty(max(nw, 1), dtype=torch.float64, device=dev)
    n_win = torch.zeros(1, dtype=torch.int64, device=dev)
    unsorted = torch.zeros(1, dtype=torch.int32, device=dev) if check_sorted else None
    check(_lib.lib().lens_event_windows(ptr(t), ptr(x), ptr(y), n, ptr(lut), W, H, int(bool(use_first_event)),
                                        float(start), float(interval), nw, ptr(wb), ptr(we), ptr(wt), ptr(n_win),
                                        ptr(unsorted), stream_ptr()), "lens_event_windows")
    if check_sorted and int(unsorted.item()):
        raise ValueError("event timestamps must be ascending")
    return wb, we, wt, n_win


def bin_events_lut(x, y, lut, win_begin, win_end, n_slots, weight=1, events_per_window_hint=0):
    """Slot histograms of the given event ranges -> frames u8 [n_windows, n_slots]
    (`frame_data[index] += accum_factor`, dvstools.py:310-322; counts wrap mod 256)."""
    require_cuda(x, y, lut, win_begin, win_end)
    n_win = win_begin.numel()
    H, W = lut.shape
    frames = torch.empty((n_win, n_slots), dtype=torch.uint8, device=x.device)
    counts = torch.empty((n_win, n_slots), dtype=torch.int32, device=x.device)
    check(_lib.lib().lens_bin_events_lut(ptr(x), ptr(y), ptr(lut), W, H, ptr(win_begin), ptr(win_end), n_win, n_slots,
                                         int(weight), int(events_per_window_hint), ptr(counts), ptr(frames),
                                         stream_ptr()), "lens_bin_events_lut")
    return frames
