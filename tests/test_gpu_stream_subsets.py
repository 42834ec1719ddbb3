"""Pushes that carry windows for any subset of a live fleet's streams, in any order (StreamingPipeline.push(...,
streams=...), lens_seqmatch_topk_stream_ids, lens_seqpr_stream_accumulate_ids, lens_snn_forward_streams).

The central property: under any schedule of pushes (lockstep, subsets, permutations, empty pushes, different Q per
push, stream resets), each stream's valid rows equal, bit for bit, the columns of one batch step over its own windows
since its last reset, and a stream outside a push keeps every piece of its state."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import synth_pooled
from test_gpu_event_streams import W_US, device_streams, kernels_run
from test_gpu_fleet_pr import _free_port, same_lists
from test_gpu_stream_pr import ALL, KW, session_oracle
from test_gpu_streaming import CASES, I, MODE_AUTO, MODE_SIMT, T, batch_pipe, cuda, model, ran, recall_ns

gpu = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def stream_pipe(W, L, N, B, mode, track=()):
    from lens_b200.pipeline import StreamingPipeline
    return StreamingPipeline(*W, roi=80, k=8, T=T, L=L, n_streams=B, n_top=N, ns=recall_ns(N), mode=mode,
                             track_pr=track)


def schedule(rng, B, n_push=10, reset_at=None):
    """[(streams or None, Q)] plus ("reset", streams) entries: subsets in random order, sometimes empty, sometimes all
    of them permuted, sometimes streams=None."""
    out = []
    for k in range(n_push):
        if k == reset_at:
            out.append(("reset", sorted(rng.choice(B, size=int(rng.integers(1, B)), replace=False).tolist())))
        Q = int(rng.integers(1, 4))
        kind = rng.choice(["none", "empty", "all", "subset", "subset", "subset"])
        if kind == "none":
            out.append((None, Q))
        elif kind == "empty":
            out.append(([], Q))
        elif kind == "all":
            out.append((rng.permutation(B).tolist(), Q))
        else:
            out.append((rng.choice(B, size=int(rng.integers(1, B)), replace=False).tolist(), Q))
    out.insert(1, (None, 2))       # lockstep first, so that the session switches to the indexed kernels mid-way
    return out


class Fleet:
    """Drives a StreamingPipeline through a schedule and records, per stream and per segment since its last reset,
    the windows it was fed, the ground truth and the rows it got back."""

    def __init__(self, sp, B, P, L, seed, tol=1):
        self.sp, self.B, self.Po, self.L, self.tol = sp, B, P - L + 1, L, tol
        self.pool = cuda(synth_pooled(B, 64, I, seed=seed))
        self.rng = np.random.default_rng(seed)
        self.cursor = [0] * B
        self.segs = [[self._seg()] for _ in range(B)]
        self.hits = self.n_valid = 0

    @staticmethod
    def _seg():
        return dict(win=[], gt=[], S=[], tv=[], ti=[])

    def run(self, sched):
        for item in sched:
            if item[0] == "reset":
                self.sp.reset_streams(item[1])
                for b in item[1]:
                    self.segs[b].append(self._seg())
                continue
            streams, Q = item
            ids = list(range(self.B)) if streams is None else list(streams)
            win = torch.stack([self.pool[b, self.cursor[b]:self.cursor[b] + Q] for b in ids]) if ids else None
            gt = self.rng.integers(-1, self.Po, size=(len(ids), Q)).astype(np.int32)
            out = self.sp.push(pooled=win, gt_center=cuda(gt), gt_tol=self.tol, streams=streams)
            assert out["top_idx"].shape == (len(ids), Q, self.sp.n_top)
            self.hits = self.hits + out["hits"].cpu()
            self.n_valid = self.n_valid + out["n_valid"].cpu()
            for i, b in enumerate(ids):
                seg = self.segs[b][-1]
                seg["win"].append(win[i])
                seg["gt"].append(gt[i])
                for k in ("S", "top_val", "top_idx"):
                    seg[{"top_val": "tv", "top_idx": "ti"}.get(k, k)].append(out[k][i])
                self.cursor[b] += Q

    def check_against_batch(self, W, N, mode):
        """Every stream segment against a batch step over its windows (S, top_val, top_idx, warm-up rows), and the
        summed Recall@N counters against the summed batch counters."""
        from lens_b200 import ops
        L = self.L
        bp = batch_pipe(W, L, N, 1, mode)
        hits, n_valid = torch.zeros(len(recall_ns(N)), dtype=torch.int64), torch.zeros(1, dtype=torch.int64)
        for b in range(self.B):
            for seg in self.segs[b]:
                if not seg["win"]:
                    continue
                win = torch.cat(seg["win"])[None].contiguous()
                S, tv, ti = (torch.cat(seg[k])[None] for k in ("S", "tv", "ti"))
                bp.net.reset_states()
                want_S = bp.similarity(pooled=win)
                assert torch.equal(S, want_S), f"stream {b}: spike counts"
                warm = min(L - 1, S.shape[1])
                assert bool((tv[:, :warm] == float("-inf")).all()) and bool((ti[:, :warm] == -1).all())
                if S.shape[1] < L:
                    continue
                wv, wi, _ = ops.seqmatch_topk(want_S, L, N)
                assert torch.equal(tv[:, L - 1:], wv) and torch.equal(ti[:, L - 1:], wi), f"stream {b}: top-N"
                gt = cuda(np.concatenate(seg["gt"])[None, L - 1:])
                h, v = ops.recall_counts(wi, self.Po, gt_center=gt, gt_tol=self.tol, ns=recall_ns(N))
                hits += h.cpu()
                n_valid += v.cpu()
        assert torch.equal(self.hits, hits) and torch.equal(self.n_valid, n_valid), (self.hits, hits)


# --------------------------------------------------------------------------- CPU: argument checks
def test_abi_rejects_bad_arguments_before_any_cuda_call():
    from lens_b200 import _lib
    L = _lib.lib()
    a = C.c_void_p(0x10000)                                        # never dereferenced: checks come first

    def match(n=2, Q=3, P=50, Ls=4, N=25, ids=a, B=4, ring=a, seen=a, rows=a):
        return L.lens_seqmatch_topk_stream_ids(a, n, Q, P, Ls, N, ids, B, ring, seen, rows, a, a, None)

    def acc(n=2, Q=3, P=50, Ls=4, ids=a, B=4, rows=a, gt=a):
        return L.lens_seqpr_stream_accumulate_ids(a, n, Q, P, Ls, ids, B, a, a, rows, gt, 0, a, None, None, None)
    for call, what in [(lambda: match(Ls=0), b"L"), (lambda: match(N=65), b"N=65"), (lambda: match(n=-1), b"sizes"),
                       (lambda: match(ids=None), b"ids"), (lambda: match(rows=None), b"rows"),
                       (lambda: match(B=-1), b"fleet"), (lambda: match(seen=None), b"seen"),
                       (lambda: match(ring=None), b"ring"), (lambda: match(n=1 << 16, Q=1 << 16), b"too many"),
                       (lambda: acc(Ls=51), b"L"), (lambda: acc(ids=None), b"ids"), (lambda: acc(gt=None), b"NULL"),
                       (lambda: acc(B=-1), b"fleet"),
                       (lambda: L.lens_snn_forward_streams(None, a, a, 1, 1, a, 0, None), b"handle")]:
        assert call() == -1 and what in L.lens_last_error(), (what, L.lens_last_error())
    assert match(n=0, ids=None, rows=None) == 0 and acc(n=0, ids=None, rows=None) == 0   # n = 0 launches nothing


def test_ops_checks_shapes_without_a_gpu():
    from lens_b200 import ops
    S, ids = torch.zeros((2, 3, 50)), torch.zeros((2,), dtype=torch.int32)
    ring, seen, rows = torch.zeros((4, 1, 50)), torch.zeros((4,), dtype=torch.int32), torch.zeros(4, dtype=torch.int64)
    c = torch.zeros((2, 3), dtype=torch.int32)
    for args, what in [((S.double(), 2, ids, ring, seen, rows, c), "S must"),
                       ((S, 2, ids[:1], ring, seen, rows, c), "ids"),
                       ((S, 2, ids.long(), ring, seen, rows, c), "ids"),
                       ((S, 2, ids, ring, seen, rows.int(), c), "rows"),
                       ((S, 2, ids, ring[:2], seen, rows, c), "ring"),
                       ((S, 2, ids, ring, seen, rows, c[:1]), "gt_center")]:
        with pytest.raises(ValueError, match=what):
            ops.seqpr_stream_accumulate_ids(*args)


# --------------------------------------------------------------------------- the central property
@gpu
@pytest.mark.parametrize("L,N,P,mode", CASES)
def test_random_schedules_equal_per_stream_batch_steps(L, N, P, mode):
    W = model(P)
    for seed in (1, 2):
        rng = np.random.default_rng(L * 100 + N + seed)
        B = int(rng.integers(5, 8))
        f = Fleet(stream_pipe(W, L, N, B, mode), B, P, L, seed=L * 1000 + P + seed)
        f.run(schedule(rng, B, reset_at=5))
        assert f.sp._indexed
        f.check_against_batch(W, N, mode)


@gpu
def test_one_camera_of_three_takes_the_segmented_path():
    L, N, P, B = 10, 25, 20000, 3                 # Po = 19 991 >= 8 192: one row per push splits its places
    W = model(P, seed=5)
    f = Fleet(stream_pipe(W, L, N, B, MODE_AUTO), B, P, L, seed=9)
    f.run([(None, 3)])
    for _ in range(L + 1):
        _, names = kernels_run(lambda: f.run([([1], 1)]))
        assert ran(names, "seqmatch_topk_stream_ids_warp_kernel<true>") and ran(names, "topn_merge_kernel"), names
        assert not ran(names, "seqmatch_topk_stream_warp_kernel<true>"), names
    f.run([([2, 0], 2)])
    f.check_against_batch(W, N, MODE_AUTO)


@gpu
def test_lockstep_then_subsets_then_lockstep():
    """A session that never pushes a subset runs the lockstep kernels only; after a subset push, streams=None pushes run
    the indexed ones with every stream in order, and all of it equals the per-stream batch steps."""
    from lens_b200._lib import launch_count
    L, N, P, B = 4, 25, 300, 5
    W = model(P, seed=7)
    f = Fleet(stream_pipe(W, L, N, B, MODE_SIMT), B, P, L, seed=17)
    lock = ["seqmatch_topk_stream_warp_kernel<false>", "ring_append_kernel"]
    indexed = ["seqmatch_topk_stream_ids_warp_kernel<false>", "ring_append_ids_kernel", "stream_advance_kernel",
               "state_rows_kernel<false>", "state_rows_kernel<true>"]
    n0 = launch_count()
    f.run([(None, 1)])
    n_lock = launch_count() - n0
    for Q in (2, 1, 3):
        _, names = kernels_run(lambda: f.run([(None, Q)]))
        assert all(ran(names, k) for k in lock) and not any(ran(names, k) for k in indexed), names
        assert not any("_ids_" in n for n in names), names
    assert torch.equal(f.sp.rows.cpu(), torch.full((B,), 7, dtype=torch.int64)) and f.sp.t == 7
    n0 = launch_count()
    f.run([(None, 1)])
    assert launch_count() - n0 == n_lock                             # SNN, match, append, recall
    _, names = kernels_run(lambda: f.run([([3, 1], 2)]))
    assert all(ran(names, k) for k in indexed), names
    f.run([([0, 4, 2], 1), ([], 2), ([4, 3, 2, 1, 0], 1)])
    _, names = kernels_run(lambda: f.run([(None, 2)]))
    assert ran(names, "seqmatch_topk_stream_ids_warp_kernel<false>") and not ran(names, "state_rows_kernel<false>")
    assert not ran(names, "seqmatch_topk_stream_warp_kernel<false>"), names
    f.run([(None, 1)])
    assert f.sp.rows.cpu().tolist() == [f.cursor[b] for b in range(B)]
    f.check_against_batch(W, N, MODE_SIMT)
    f.sp.reset()                                                     # back to lockstep
    _, names = kernels_run(lambda: f.sp.push(pooled=f.pool[:, :2].contiguous()))
    assert ran(names, "seqmatch_topk_stream_warp_kernel<false>") and not any("_ids_" in n for n in names), names
    assert f.sp.rows.cpu().tolist() == [2] * B


@gpu
def test_push_events_of_a_subset():
    from lens_b200 import ops
    B, Q, L, N, P = 5, 3, 2, 25, 250
    W = model(P, seed=13)
    t, x, y, off, t0 = device_streams(3, Q, 40_000, seed=17)
    window = W_US * 250
    sp, ref = stream_pipe(W, L, N, B, MODE_SIMT), stream_pipe(W, L, N, B, MODE_SIMT)
    got = sp.push_events(t, x, y, off, t0, window, Q, roi_x0=23, streams=[4, 0, 2])
    _, pooled, n_ev = ops.bin_event_streams(t, x, y, off, t0, window, Q, 80, 8, roi_x0=23, want_frames=False)
    want = ref.push(pooled=pooled, streams=[4, 0, 2])
    for k in ("top_val", "top_idx", "S"):
        assert torch.equal(got[k], want[k]), k
    assert torch.equal(got["events_per_window"], n_ev)
    empty = sp.push_events(t, x, y, off[:1].contiguous(), t0[:0].contiguous(), window, Q, streams=[])
    assert empty["events_per_window"].shape == (0, Q) and empty["top_idx"].shape == (0, Q, N)


# --------------------------------------------------------------------------- untouched state and errors
def snapshot(sp):
    return [v.clone() for v in sp.net.state()] + [sp.ring.clone(), sp.seen.clone(), sp.rows.clone(),
                                                  sp._pr_acc["place"][16:].view(torch.int32).view(sp.n_streams, -1)
                                                  .clone()]


@gpu
@pytest.mark.parametrize("mode", [MODE_SIMT, MODE_AUTO])
def test_streams_outside_a_push_are_untouched(mode):
    L, N, P, B = 3, 25, 200, 6
    W = model(P, seed=3)
    sp = stream_pipe(W, L, N, B, mode, track=("place",))
    pool = cuda(synth_pooled(B, 8, I, seed=4))
    c = torch.zeros((B, 4), dtype=torch.int32, device="cuda")
    sp.push(pooled=pool[:, :4].contiguous(), gt_center=c, gt_tol=1)
    for streams in ([5, 1, 3], [2], [0, 4]):
        before = snapshot(sp)
        sp.push(pooled=pool[streams, 4:6].contiguous(), gt_center=c[:len(streams), :2].contiguous(), gt_tol=1,
                streams=streams)
        after = snapshot(sp)
        keep = [b for b in range(B) if b not in streams]
        for x, y in zip(before, after):
            assert torch.equal(x[keep], y[keep])
        for x, y in zip(before[1:3], after[1:3]):                 # the pushed streams did advance (v1, v2)
            assert not torch.equal(x[streams], y[streams])
        assert (after[5][streams] - before[5][streams]).tolist() == [2] * len(streams)


@gpu
def test_bad_pushes_raise_and_change_nothing():
    from lens_b200._lib import LensError
    L, N, P, B = 3, 25, 120, 4
    W = model(P, seed=2)
    pool = cuda(synth_pooled(B, 4, I, seed=3))
    sp = stream_pipe(W, L, N, B, MODE_SIMT, track=("place",))
    c = torch.zeros((B, 2), dtype=torch.int32, device="cuda")
    sp.push(pooled=pool[:, :2].contiguous(), gt_center=c, gt_tol=0)
    before, t = snapshot(sp), sp.t
    two = pool[:2, 2:].contiguous()
    bad = [dict(streams=[1, 1]), dict(streams=[0, B]), dict(streams=[-1, 0]), dict(streams=[True, False]),
           dict(streams=torch.tensor([0, 1], dtype=torch.uint8)), dict(streams=[0.0, 1.0]), dict(streams=[0, 1, 2]),
           dict(streams=[0]), dict(streams=[0, 1], gt_center=c[:1]), dict(streams=[0, 1], gt_center=c.long()[:2]),
           dict(streams=[0, 1], gt_center=None), dict(streams=[0, 1], pooled=pool[:2, 2:, :50].contiguous())]
    for kw in bad:
        args = dict(pooled=two, gt_center=c[:2].contiguous(), gt_tol=0)
        args.update(kw)
        with pytest.raises(LensError):
            sp.push(**args)
    with pytest.raises(LensError):
        sp.push(streams=[0])                                      # rows for a stream, but no windows
    after = snapshot(sp)
    assert sp.t == t and not sp._indexed and all(torch.equal(x, y) for x, y in zip(before, after))
    # the accepted forms: a mask, a numpy array, a CPU tensor
    outs = [stream_pipe(W, L, N, B, MODE_SIMT).push(pooled=two, streams=s)["top_val"]
            for s in ([True, True, False, False], np.array([0, 1]), torch.tensor([0, 1]))]
    assert all(torch.equal(o, outs[0]) for o in outs)


@gpu
def test_out_of_range_ids_are_skipped_by_the_abi():
    """Direct ABI calls: an id outside [0, B) touches no memory; the other positions are computed as usual."""
    from lens_b200 import _lib, ops
    from lens_b200._lib import ptr, stream_ptr
    L, N, P, B, Q = 3, 8, 64, 2, 2
    S = torch.randint(0, 5, (2, Q, P), device="cuda").float()
    guard = torch.full((4 * B * (L - 1) * P,), 7.0, device="cuda")   # the ring with guard zones around it
    ring = guard[B * (L - 1) * P:2 * B * (L - 1) * P].view(B, L - 1, P)
    ring.zero_()
    seen = torch.full((B,), L - 1, dtype=torch.int32, device="cuda")
    rows = torch.full((B,), 5, dtype=torch.int64, device="cuda")
    for bad in (B, -1, 1 << 30):
        ids = torch.tensor([1, bad], dtype=torch.int32, device="cuda")
        tv, ti = ops.seqmatch_topk_stream_ids(S, L, N, ids, ring, seen, rows)
        assert bool(torch.isfinite(tv[0]).all()) and bool((ti[1] == -1).all()) and bool((tv[1] == -float("inf")).all())
        acc = torch.zeros((ops.seqpr_stream_bytes(B, P, L, 0),), dtype=torch.uint8, device="cuda")
        ops.seqpr_stream_accumulate_ids(S, L, ids, ring, seen, rows, torch.zeros((2, Q), dtype=torch.int32,
                                                                                 device="cuda"), 0, acc_place=acc)
    torch.cuda.synchronize()
    assert bool((guard[:B * (L - 1) * P] == 7).all()) and bool((guard[2 * B * (L - 1) * P:] == 7).all())
    assert rows.cpu().tolist() == [5, 5 + 3 * Q] and seen.cpu().tolist() == [L - 1, L - 1]
    W = model(P)
    net = stream_pipe(W, L, N, B, MODE_SIMT).net
    state = [v.clone() for v in net.state()]
    pooled = cuda(synth_pooled(2, Q, I, seed=1))
    ids = torch.tensor([B, 1], dtype=torch.int32, device="cuda")
    counts = torch.empty((2, Q, P), device="cuda")
    _lib.check(_lib.lib().lens_snn_forward_streams(net._h, ptr(pooled), ptr(ids), 2, Q, ptr(counts), MODE_SIMT,
                                                   stream_ptr()), "lens_snn_forward_streams")
    after = net.state()
    assert bool(torch.isfinite(counts).all())
    assert all(torch.equal(x[0], y[0]) for x, y in zip(state, after))
    assert not torch.equal(state[2][1], after[2][1])


# --------------------------------------------------------------------------- session precision-recall
def group_reference(S_rows, gts, L, tol, n_thresh, mode):
    """The documented group API: streams grouped by their number of rows, every group scanned into one extremes /
    gtp, then counted; the counts added."""
    from lens_b200 import ops
    from lens_b200.src.metrics import pr_lists
    groups = {}
    for b, S in enumerate(S_rows):
        if S.shape[0] >= L:
            groups.setdefault(S.shape[0], []).append(b)
    ext = torch.zeros((2,), dtype=torch.int64, device="cuda")
    gtp = torch.zeros((1,), dtype=torch.int64, device="cuda")
    recs = {}
    for k, members in groups.items():
        S = torch.stack([S_rows[b] for b in members]).contiguous()
        c = cuda(np.stack([gts[b][L - 1:] for b in members]))
        recs[k] = (S, c, ops.seqpr_scan(S, L, mode, gt_center=c, gt_tol=tol, extremes=ext, gtp=gtp)[0])
    tp = torch.zeros((n_thresh,), dtype=torch.int64, device="cuda")
    fp = torch.zeros((n_thresh,), dtype=torch.int64, device="cuda")
    for S, c, rec in recs.values():
        ops.seqpr_counts(S, L, mode, rec, ext, n_thresh, gt_center=c, gt_tol=tol, tp=tp, fp=fp)
    tp, fp, g = tp.cpu().numpy(), fp.cpu().numpy(), int(gtp.item())
    P, R = pr_lists(tp, fp, g)
    return dict(P=P, R=R, tp=tp, fp=fp, gtp=g)


@gpu
@pytest.mark.parametrize("L,P", [(1, 100), (3, 140), (10, 200)])
def test_session_precision_recall_over_a_random_schedule(L, P):
    N, tol = 25, 1
    W = model(P, seed=L)
    rng = np.random.default_rng(L + 40)
    B = int(rng.integers(5, 8))
    f = Fleet(stream_pipe(W, L, N, B, MODE_SIMT, track=ALL), B, P, L, seed=L + 50, tol=tol)
    f.run(schedule(rng, B, n_push=12))
    S_rows = [torch.cat(f.segs[b][0]["S"]) if f.segs[b][0]["S"] else torch.zeros((0, P), device="cuda")
              for b in range(B)]
    gts = [np.concatenate(f.segs[b][0]["gt"]) if f.segs[b][0]["gt"] else np.zeros(0, np.int32) for b in range(B)]
    for m, mode in zip(ALL, range(3)):
        for n in (2, 100):
            got = f.sp.session_precision_recall(n_thresh=n, **KW[m])
            want = group_reference(S_rows, gts, L, tol, n, mode)
            same_lists((got["P"], got["R"]), (want["P"], want["R"]))
            assert np.array_equal(got["tp"], want["tp"]) and np.array_equal(got["fp"], want["fp"])
            assert got["gtp"] == want["gtp"]
    # the oracle on the per-stream matrices (streams padded to one length; each one's columns end at its own rows)
    Qmax = max(s.shape[0] for s in S_rows)
    S = np.zeros((B, Qmax, P), np.float32)
    c = np.full((B, Qmax), -1, np.int32)
    for b in range(B):
        S[b, :S_rows[b].shape[0]] = S_rows[b].cpu().numpy()
        c[b, :len(gts[b])] = gts[b]
    segs = [[(0, S_rows[b].shape[0], 0)] for b in range(B)]
    for m in ALL:
        kw = KW[m]
        got = f.sp.session_precision_recall(**kw)
        want = session_oracle(S, L, c, tol, segs, kw["matching"], kw.get("best"), 100)
        same_lists((got["P"], got["R"]), want)


@gpu
def test_two_ranks_equal_one_rank():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
           "--master-addr", "127.0.0.1", "--master-port", str(_free_port()),
           os.path.join(ROOT, "tests", "stream_subset_dist_check.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-2000:]
    assert "OK" in res.stdout, res.stdout[-2000:]
