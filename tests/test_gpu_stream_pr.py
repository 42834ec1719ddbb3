"""Session precision-recall of live fleets (StreamingPipeline(track_pr=...).session_precision_recall,
lens_seqpr_stream_*): createPR over every valid row pushed in a session, accumulated on the GPU push by push.

For a fresh pipeline without stream resets the session's counts and lists equal InferencePipeline.precision_recall
over the concatenated spike counts of the pushes, for every chunking; with resets they equal the oracle's createPR
over the per-segment sequence-matched matrices stacked along the query axis.  Every comparison is exact."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import synth_pooled
from oracle import oracle as O
from test_gpu_fleet_pr import MODE_IDS, MODES, _free_port, kernels_and_launches, same_lists
from test_gpu_streaming import I, MODE_SIMT, MODE_TC, T, batch_pipe, chunkings, model

gpu = pytest.mark.gpu
f32 = np.float32
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ALL = ("place", "query", "multi")
KW = {"place": dict(matching="single", best="place"), "query": dict(matching="single", best="query"),
      "multi": dict(matching="multi")}


def cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def stream_pipe(W, L, B, mode=MODE_SIMT, track=ALL):
    from lens_b200.pipeline import StreamingPipeline
    return StreamingPipeline(*W, roi=80, k=8, T=T, L=L, n_streams=B, mode=mode, track_pr=track)


def centers(rng, B, Q_tot, L, Po, no_pos=0.15):
    """Band centres per pushed row; warm-up rows get real places so that only the pipeline keeps them out."""
    c = rng.integers(0, Po, size=(B, Q_tot)).astype(np.int32)
    c[:, L - 1:][rng.random((B, Q_tot - L + 1)) < no_pos] = -1
    c[0, L - 1] = 0
    c[-1, -1] = Po - 1
    return c


def push_all(sp, pooled, chunks, gt, tol):
    outs, q0 = [], 0
    for n in chunks:
        outs.append(sp.push(pooled=pooled[:, q0:q0 + n].contiguous(), gt_center=gt[:, q0:q0 + n].contiguous(),
                            gt_tol=tol))
        q0 += n
    return outs


def same_pr(got, want):
    same_lists((got["P"], got["R"]), (want["P"], want["R"]))
    assert np.array_equal(got["tp"], want["tp"]) and np.array_equal(got["fp"], want["fp"])
    assert got["gtp"] == want["gtp"]


def session_oracle(S, L, c, tol, segments, matching, best, n_thresh):
    """O.create_pr over the session matrices: stream b's columns are, for each (s, e, first) of segments[b], the
    columns of O.seqmatch(S[b, s:e]) whose row g (global) is >= first, stacked along the query axis."""
    B, _, P = S.shape
    Po = P - L + 1
    Ds, Gs = [], []
    for b in range(B):
        cols, gts = [np.zeros((Po, 0), f32)], [np.zeros((Po, 0), bool)]
        for s, e, first in segments[b]:
            if e - s < L:
                continue
            D = O.seqmatch(S[b, s:e], L)
            g = np.arange(s + L - 1, e)
            keep = g >= first
            cb = c[b, g[keep]]
            cols.append(D[:, keep])
            gts.append((cb[None, :] >= 0) & (np.abs(np.arange(Po)[:, None] - cb[None, :]) <= tol))
        Ds.append(np.concatenate(cols, axis=1))
        Gs.append(np.concatenate(gts, axis=1))
    if matching == "single" and best == "place":
        # streams may have different numbers of rows after resets: pad with -inf rows without positives, which
        # change no column's first maximum; a stream without a valid row has no column
        keep = [b for b in range(B) if Ds[b].shape[1]]
        n = max(Ds[b].shape[1] for b in keep)
        pad = lambda a, v: np.pad(a, ((0, 0), (0, n - a.shape[1])), constant_values=v)   # noqa: E731
        M = np.concatenate([pad(Ds[b], -np.inf).astype(f32).T for b in keep], axis=1)
        G = np.concatenate([pad(Gs[b], False).T for b in keep], axis=1)
    else:
        M, G = np.concatenate(Ds, axis=1), np.concatenate(Gs, axis=1)
    return O.create_pr(M, G, n_thresh=n_thresh, matching=matching)


class OpsSession:
    """A session driven through the ops API on crafted spike counts: accumulate, then the streaming match that
    advances the ring and seen, as StreamingPipeline.push does."""

    def __init__(self, B, P, L, track=ALL):
        from lens_b200 import ops
        self.ops, self.B, self.P, self.L, self.t = ops, B, P, L, 0
        self.ring = torch.zeros((B, L - 1, P), device="cuda") if L > 1 else None
        self.seen = torch.zeros((B,), dtype=torch.int32, device="cuda")
        self.acc = {m: torch.zeros((ops.seqpr_stream_bytes(B, P, L, i),), dtype=torch.uint8, device="cuda")
                    for i, m in enumerate(ALL) if m in track}

    def push(self, S, c, tol):
        S, c = cuda(S), cuda(c)
        self.ops.seqpr_stream_accumulate(S, self.L, self.ring, self.seen, self.t, c, tol,
                                         **{"acc_" + m: a for m, a in self.acc.items()})
        self.ops.seqmatch_topk_stream(S, self.L, 1, self.ring, self.seen, self.t)
        self.t += S.shape[1]

    def curve(self, name, n_thresh=100):
        from lens_b200.src.metrics import pr_lists
        packed = self.ops.seqpr_stream_histogram(self.acc[name], self.B, self.P, self.L, ALL.index(name))
        tp, fp, gtp = self.ops.seqpr_stream_counts(packed, self.L, n_thresh)
        P, R = pr_lists(tp, fp, gtp)
        return dict(P=P, R=R, tp=tp, fp=fp, gtp=gtp)


def ops_session(S, L, c, tol, chunks, track=ALL):
    B, _, P = S.shape
    s, q0 = OpsSession(B, P, L, track), 0
    for n in chunks:
        s.push(S[:, q0:q0 + n], c[:, q0:q0 + n], tol)
        q0 += n
    return s


# --------------------------------------------------------------------------- CPU: argument checks
def test_abi_rejects_bad_arguments_before_any_cuda_call():
    from lens_b200 import _lib
    L = _lib.lib()
    a = C.c_void_p(0x10000)                                        # never dereferenced: checks come first
    n = C.c_int64(0)

    def acc(B=2, Q=3, P=50, Ls=4, ring=a, seen=a, t=0, gt=a, tol=0, accs=(a, a, a)):
        return L.lens_seqpr_stream_accumulate(a, B, Q, P, Ls, ring, seen, t, gt, tol, *accs, None)
    cases = [(lambda: acc(Ls=0), b"L"), (lambda: acc(Ls=51), b"L"), (lambda: acc(Q=0), b"sizes"),
             (lambda: acc(B=-1), b"sizes"), (lambda: acc(t=-1), b"t and gt_tol"), (lambda: acc(tol=-1), b"gt_tol"),
             (lambda: acc(B=1 << 16, Q=1 << 16), b"too many"), (lambda: acc(seen=None), b"NULL"),
             (lambda: acc(gt=None), b"NULL"), (lambda: acc(ring=None), b"ring"),
             (lambda: acc(accs=(a, C.c_void_p(0x10004), None)), b"aligned"),
             (lambda: L.lens_seqpr_stream_bytes(2, 50, 51, 0, C.byref(n)), b"sizes"),
             (lambda: L.lens_seqpr_stream_bytes(2, 50, 2, 3, C.byref(n)), b"mode"),
             (lambda: L.lens_seqpr_stream_histogram(a, 2, 50, 2, 3, a, a, a, None), b"mode"),
             (lambda: L.lens_seqpr_stream_histogram(None, 2, 50, 2, 0, a, a, a, None), b"NULL"),
             (lambda: L.lens_seqpr_hist_counts(a, 2, 1, a, a, None), b"n_thresh"),
             (lambda: L.lens_seqpr_hist_counts(a, 2, 4097, a, a, None), b"n_thresh"),
             (lambda: L.lens_seqpr_hist_counts(a, 0, 100, a, a, None), b"L")]
    for call, what in cases:
        assert call() == -1 and what in L.lens_last_error(), (what, L.lens_last_error())
    assert acc(B=0, ring=None, seen=None, gt=None) == 0                 # B == 0 launches nothing
    assert acc(accs=(None, None, None)) == 0                             # nothing tracked: nothing to do
    for mode, want in ((0, 16 + 4 * 3 * 49), (1, 16 + 16 * 65536), (2, 16 + 16 * 65536)):
        assert L.lens_seqpr_stream_bytes(3, 50, 2, mode, C.byref(n)) == 0 and n.value == want


def test_ops_checks_shapes_without_a_gpu():
    from lens_b200 import ops
    S = torch.zeros((2, 3, 50))
    seen = torch.zeros((2,), dtype=torch.int32)
    ring = torch.zeros((2, 1, 50))
    c = torch.zeros((2, 3), dtype=torch.int32)
    ok = dict(acc_place=torch.zeros((ops.seqpr_stream_bytes(2, 50, 2, 0),), dtype=torch.uint8))
    for args, kw, what in [((S.double(), 2, ring, seen, 0, c), ok, "S must"),
                           ((S, 0, ring, seen, 0, c), ok, "L"),
                           ((S, 2, None, seen, 0, c), ok, "ring"),
                           ((S, 2, ring, seen[:1], 0, c), ok, "seen"),
                           ((S, 2, ring, seen, 0, c[:, :2]), ok, "gt_center"),
                           ((S, 2, ring, seen, 0, c.long()), ok, "gt_center"),
                           ((S, 2, ring, seen, 0, c), dict(acc_query=ok["acc_place"]), "query accumulator")]:
        with pytest.raises(ValueError, match=what):
            ops.seqpr_stream_accumulate(*args, **kw)
    for n in (1, 4097):
        with pytest.raises(ValueError, match="n_thresh"):
            ops.seqpr_stream_counts(torch.zeros(3), 2, n)


# --------------------------------------------------------------------------- batch equivalence
CASES = [  # (L, B, P, SNN path): ragged / tiny P, both SNN paths
    (1, 1, 100, MODE_SIMT),
    (2, 3, 97, MODE_TC),
    (10, 3, 20, MODE_SIMT),       # Po = 11
    (10, 64, 300, MODE_TC),
    (2, 64, 130, MODE_SIMT),
]


@gpu
@pytest.mark.parametrize("L,B,P,snn", CASES)
def test_every_chunking_equals_the_batch_method(L, B, P, snn):
    """All three modes tracked at once, chunkings ones / mixed / one_chunk / random, n_thresh 2, 100 and 4096."""
    Q_tot, tol = 3 * L + 3, 2
    W = model(P, seed=L + P)
    rng = np.random.default_rng(L * 100 + B)
    pooled = cuda(synth_pooled(B, Q_tot, I, seed=L * 1000 + P))
    c = centers(rng, B, Q_tot, L, P - L + 1)
    bp = batch_pipe(W, L, 25, B, snn)
    want = None
    for name, chunks in chunkings(L, Q_tot, seed=L + P).items():
        sp = stream_pipe(W, L, B, snn)
        S = torch.cat([o["S"] for o in push_all(sp, pooled, chunks, cuda(c), tol)], dim=1)
        assert float(S.sum()) > 0
        if want is None:
            want = {(m, n): bp.precision_recall(S, gt_center=cuda(c[:, L - 1:]), gt_tol=tol, n_thresh=n, **KW[m])
                    for m in ALL for n in (2, 100, 4096)}
        for (m, n), w in want.items():
            try:
                same_pr(sp.session_precision_recall(n_thresh=n, **KW[m]), w)
            except AssertionError as e:
                raise AssertionError(f"chunking {name} {chunks}, mode {m}, n_thresh {n}") from e


@gpu
@pytest.mark.parametrize("mode", ALL)
def test_each_mode_alone(mode):
    L, B, P, Q_tot, tol = 3, 5, 140, 10, 1
    W = model(P, seed=4)
    pooled = cuda(synth_pooled(B, Q_tot, I, seed=21))
    c = centers(np.random.default_rng(1), B, Q_tot, L, P - L + 1)
    sp = stream_pipe(W, L, B, track=(mode,))
    S = torch.cat([o["S"] for o in push_all(sp, pooled, [1, 3, 2, 4], cuda(c), tol)], dim=1)
    want = batch_pipe(W, L, 25, B, MODE_SIMT).precision_recall(S, gt_center=cuda(c[:, L - 1:]), gt_tol=tol, **KW[mode])
    same_pr(sp.session_precision_recall(**KW[mode]), want)


@gpu
@pytest.mark.parametrize("tol", [0, 1, 2, 3])
def test_band_tolerance_and_map_ends(tol):
    """Centres at -1, 0 and Po - 1 on valid rows of every stream; |p - c| <= tol, inclusive."""
    L, B, P, Q_tot = 2, 3, 120, 9
    Po = P - L + 1
    W = model(P, seed=tol)
    pooled = cuda(synth_pooled(B, Q_tot, I, seed=30 + tol))
    c = centers(np.random.default_rng(tol), B, Q_tot, L, Po)
    c[:, L], c[:, L + 1], c[:, L + 2] = -1, 0, Po - 1
    sp = stream_pipe(W, L, B)
    S = torch.cat([o["S"] for o in push_all(sp, pooled, [2, 1, 6], cuda(c), tol)], dim=1)
    bp = batch_pipe(W, L, 25, B, MODE_SIMT)
    for m in ALL:
        same_pr(sp.session_precision_recall(**KW[m]),
                bp.precision_recall(S, gt_center=cuda(c[:, L - 1:]), gt_tol=tol, **KW[m]))


# --------------------------------------------------------------------------- the oracle, crafted spike counts
@gpu
@pytest.mark.parametrize("matching,best", MODES, ids=MODE_IDS)
def test_pipeline_session_equals_the_oracle(matching, best):
    L, B, P, Q_tot, tol = 4, 3, 150, 11, 1
    W = model(P, seed=8)
    pooled = cuda(synth_pooled(B, Q_tot, I, seed=6))
    c = centers(np.random.default_rng(2), B, Q_tot, L, P - L + 1)
    sp = stream_pipe(W, L, B)
    S = torch.cat([o["S"] for o in push_all(sp, pooled, [1, 2, 3, 1, 4], cuda(c), tol)], dim=1).cpu().numpy()
    want = session_oracle(S, L, c, tol, [[(0, Q_tot, 0)]] * B, matching, best, 100)
    got = sp.session_precision_recall(matching=matching, best=best or "place")
    same_lists((got["P"], got["R"]), want)


@gpu
@pytest.mark.parametrize("chunks", [[1] * 6, [6]], ids=["ones", "one_chunk"])
def test_tied_maxima_take_the_first(chunks):
    """Maxima tied between a positive and a negative entry, in both orders, across pushes: the first maximum (the
    earliest row per place, the lowest place per row) decides the hit, as np.argmax does."""
    B, Q, P, L, tol = 2, 6, 40, 1, 0
    S = np.zeros((B, Q, P), f32)
    c = np.full((B, Q), 30, np.int32)
    S[:, 1, 3] = S[:, 4, 3] = 7                    # place 3: row 1 positive, row 4 negative
    S[:, 1, 5] = S[:, 4, 5] = 7                    # place 5: row 1 negative, row 4 positive
    c[:, 1], c[:, 4] = 3, 5
    S[:, 2, 10] = S[:, 2, 20] = 5                  # row 2: place 10 positive, 20 negative
    S[:, 3, 10] = S[:, 3, 20] = 5                  # row 3: place 10 negative, 20 positive
    c[:, 2], c[:, 3] = 10, 20
    S[1] += (np.arange(P) % 3 == 0)[None, :].astype(f32)
    s = ops_session(S, L, c, tol, chunks)
    segs = [[(0, Q, 0)]] * B
    for m, (matching, best) in zip(ALL, MODES):
        for n in (2, 7, 100):
            got = s.curve(m, n)
            same_lists((got["P"], got["R"]), session_oracle(S, L, c, tol, segs, matching, best, n))


@gpu
def test_constant_spike_counts():
    B, Q, P, L = 2, 7, 70, 2
    S = np.full((B, Q, P), 3.0, f32)
    c = centers(np.random.default_rng(1), B, Q, L, P - L + 1)
    s = ops_session(S, L, c, 1, [2, 1, 4])
    for m, (matching, best) in zip(ALL, MODES):
        got = s.curve(m)
        same_lists((got["P"], got["R"]), session_oracle(S, L, c, 1, [[(0, Q, 0)]] * B, matching, best, 100))
        assert len(set(got["tp"].tolist())) == 1


@gpu
@pytest.mark.parametrize("bad", [65536.0, 0.5, -1.0], ids=["above_65535", "not_integer", "negative"])
def test_sums_outside_the_exact_range_raise(bad):
    from lens_b200._lib import LensError
    B, Q, P, L = 2, 3, 40, 1
    S = np.ones((B, Q, P), f32)
    c = np.zeros((B, Q), np.int32)
    ok = ops_session(S, L, c, 0, [Q])
    S[1, 2, 17] = bad
    s = ops_session(S, L, c, 0, [Q])
    for m in ALL:
        ok.curve(m)
        with pytest.raises(LensError, match="not integers"):
            s.curve(m)
    S = np.full((B, Q, P), 65535.0, f32)                              # the largest exact sum is fine
    ops_session(S, L, c, 0, [Q]).curve("multi")


# --------------------------------------------------------------------------- session boundaries
@gpu
@pytest.mark.parametrize("L", [1, 3])
def test_reset_streams_mid_session(L):
    """A restarted stream's later valid rows are more columns of the same session: the oracle over each stream's
    segments stacked along the query axis."""
    B, P, Q1, Q2, tol = 4, 160, 5, 6, 1
    W = model(P, seed=11)
    pooled = cuda(synth_pooled(B, Q1 + Q2, I, seed=12))
    c = centers(np.random.default_rng(3), B, Q1 + Q2, L, P - L + 1)
    sp = stream_pipe(W, L, B)
    first = push_all(sp, pooled[:, :Q1], [2, 3], cuda(c[:, :Q1]), tol)
    sp.reset_streams([1, 3])
    after = push_all(sp, pooled[:, Q1:], [1, 4, 1], cuda(c[:, Q1:]), tol)
    S = torch.cat([o["S"] for o in first + after], dim=1).cpu().numpy()
    whole, split = [(0, Q1 + Q2, 0)], [(0, Q1, 0), (Q1, Q1 + Q2, 0)]
    segs = [whole, split, whole, split]
    for m, (matching, best) in zip(ALL, MODES):
        got = sp.session_precision_recall(**KW[m])
        same_lists((got["P"], got["R"]), session_oracle(S, L, c, tol, segs, matching, best, 100))


@gpu
def test_reset_precision_recall_counts_only_later_rows():
    L, B, P, Q1, Q2, tol = 3, 3, 130, 4, 5, 1
    W = model(P, seed=14)
    pooled = cuda(synth_pooled(B, Q1 + Q2, I, seed=15))
    c = centers(np.random.default_rng(4), B, Q1 + Q2, L, P - L + 1)
    sp = stream_pipe(W, L, B)
    outs = push_all(sp, pooled[:, :Q1], [Q1], cuda(c[:, :Q1]), tol)
    t, seen = sp.t, sp.seen.clone()
    sp.reset_precision_recall()
    assert sp.t == t and torch.equal(sp.seen, seen)
    outs += push_all(sp, pooled[:, Q1:], [2, 3], cuda(c[:, Q1:]), tol)
    S = torch.cat([o["S"] for o in outs], dim=1).cpu().numpy()
    for m, (matching, best) in zip(ALL, MODES):
        got = sp.session_precision_recall(**KW[m])
        same_lists((got["P"], got["R"]), session_oracle(S, L, c, tol, [[(0, Q1 + Q2, Q1)]] * B, matching, best, 100))


@gpu
def test_reset_starts_a_new_session():
    L, B, P, Q, tol = 2, 3, 120, 6, 2
    W = model(P, seed=16)
    pooled = cuda(synth_pooled(B, 2 * Q, I, seed=17))
    c = cuda(centers(np.random.default_rng(5), B, Q, L, P - L + 1))
    sp = stream_pipe(W, L, B)
    push_all(sp, pooled[:, :Q], [Q], c, tol)
    sp.reset()
    push_all(sp, pooled[:, Q:], [1, 5], c, tol)
    fresh = stream_pipe(W, L, B)
    push_all(fresh, pooled[:, Q:], [Q], c, tol)
    for m in ALL:
        same_pr(sp.session_precision_recall(**KW[m]), fresh.session_precision_recall(**KW[m]))


# --------------------------------------------------------------------------- outputs and errors
@gpu
@pytest.mark.parametrize("snn", [MODE_SIMT, MODE_TC])
def test_push_outputs_do_not_change(snn):
    L, B, P, Q_tot, tol = 4, 6, 200, 12, 2
    W = model(P, seed=18)
    pooled = cuda(synth_pooled(B, Q_tot, I, seed=19))
    c = cuda(centers(np.random.default_rng(6), B, Q_tot, L, P - L + 1))
    chunks = [1, 3, 2, 6]
    a = push_all(stream_pipe(W, L, B, snn), pooled, chunks, c, tol)
    b = push_all(stream_pipe(W, L, B, snn, track=()), pooled, chunks, c, tol)
    for x, y in zip(a, b):
        for k in ("top_val", "top_idx", "S", "hits", "n_valid"):
            assert torch.equal(x[k], y[k]), k


@gpu
def test_errors_and_unchanged_state():
    from lens_b200._lib import LensError
    L, B, P = 3, 4, 120
    W = model(P, seed=2)
    pooled = cuda(synth_pooled(B, 4, I, seed=3))
    c = cuda(np.zeros((B, 4), np.int32))
    sp = stream_pipe(W, L, B, track=("place", "query"))
    with pytest.raises(LensError, match="no valid row"):
        sp.session_precision_recall()                                  # nothing pushed yet
    push_all(sp, pooled[:, :2], [2], c, 0)
    with pytest.raises(LensError, match="no valid row"):
        sp.session_precision_recall()                                  # warm-up rows only
    push_all(sp, pooled[:, 2:3], [1], c, 0)
    before = [v.clone() for v in sp.net.state()] + [sp.ring.clone(), sp.seen.clone()] + \
        [a.clone() for a in sp._pr_acc.values()]
    t_before = sp.t
    for kw in (dict(), dict(gt_center=c[:, 3:].contiguous(), gt_tol=-1)):
        with pytest.raises(LensError, match="gt_center"):
            sp.push(pooled=pooled[:, 3:].contiguous(), **kw)
    with pytest.raises(LensError, match="'multi' is not tracked"):
        sp.session_precision_recall(matching="multi")
    with pytest.raises(ValueError, match="n_thresh"):
        sp.session_precision_recall(n_thresh=1)
    after = list(sp.net.state()) + [sp.ring, sp.seen] + list(sp._pr_acc.values())
    assert sp.t == t_before and all(torch.equal(x, y) for x, y in zip(after, before))
    pr = sp.session_precision_recall()
    assert pr["tp"][-1] + pr["fp"][-1] == B * (P - L + 1)                # one column per (stream, place)
    with pytest.raises(LensError, match="live session.*session_precision_recall"):
        sp.precision_recall(torch.zeros((B, 3, P), device="cuda"), gt_center=c[:, :1].contiguous())
    with pytest.raises(LensError, match="track_pr"):
        stream_pipe(W, L, B, track=("places",))


# --------------------------------------------------------------------------- structure
@gpu
def test_kernels_and_launches_do_not_grow_with_B():
    from lens_b200 import ops
    from lens_b200._lib import launch_count
    L, P, Q = 3, 300, 1
    seen = {}
    for B in (2, 512):
        S = torch.randint(0, 5, (B, Q, P), device="cuda").float()
        c = cuda(np.zeros((B, Q), np.int32))
        per = {}
        for track in [("place",), ("query",), ("multi",), ALL]:
            s = OpsSession(B, P, L, track)
            s.seen.fill_(L - 1)
            n0 = launch_count()
            ops.seqpr_stream_accumulate(S, L, s.ring, s.seen, 0, c, 1, **{"acc_" + m: a for m, a in s.acc.items()})
            per[track] = launch_count() - n0
        s = OpsSession(B, P, L)
        s.seen.fill_(L - 1)
        names, _ = kernels_and_launches(lambda: s.push(S.cpu().numpy(), c.cpu().numpy(), 1))
        assert any("seqpr_stream_accumulate_kernel" in n for n in names), names
        assert any("seqpr_stream_query_fold_kernel" in n for n in names), names
        names, _ = kernels_and_launches(lambda: [s.curve(m) for m in ALL])
        for k in ("seqpr_stream_place_hist_kernel", "seqpr_stream_add_kernel", "seqpr_stream_bin_kernel",
                  "seqpr_prefix_kernel"):
            assert any(k in n for n in names), (k, names)
        seen[B] = per
    assert seen[2] == seen[512], seen
    assert seen[2] == {("place",): 1, ("query",): 2, ("multi",): 1, ALL: 2}, seen


@gpu
def test_memory_grows_by_the_accumulators_only():
    from lens_b200 import ops
    L, B, P, tol = 2, 64, 2000, 1
    W = model(P, seed=20)
    pooled = cuda(synth_pooled(B, 3, I, seed=22))
    c = cuda(centers(np.random.default_rng(7), B, 3, L, P - L + 1))
    grown = {}
    push_all(stream_pipe(W, L, B, track=()), pooled, [2, 1], c, tol)      # anything created once, before measuring
    for track in ((), ALL):
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        sp = stream_pipe(W, L, B, track=track)
        owned = torch.cuda.memory_allocated() - base
        push_all(sp, pooled[:, :2], [2], c[:, :2].contiguous(), tol)
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        before = torch.cuda.memory_allocated()
        out = sp.push(pooled=pooled[:, 2:].contiguous(), gt_center=c[:, 2:].contiguous(), gt_tol=tol)
        torch.cuda.synchronize()
        grown[track] = (owned, torch.cuda.max_memory_allocated() - before)
        del sp, out
    accs = sum(ops.seqpr_stream_bytes(B, P, L, i) for i in range(3))
    assert accs <= grown[ALL][0] - grown[()][0] <= accs + 3 * 512, (grown, accs)   # allocator granularity
    assert grown[ALL][1] == grown[()][1], grown                                      # a push allocates nothing more


@gpu
def test_two_ranks_equal_one_rank():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
           "--master-addr", "127.0.0.1", "--master-port", str(_free_port()),
           os.path.join(ROOT, "tests", "stream_pr_dist_check.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-2000:]
    assert "OK" in res.stdout, res.stdout[-2000:]
