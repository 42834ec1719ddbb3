"""Sequence matching across calls (lens_seqmatch_topk_stream) and the live-fleet pipeline built on it
(StreamingPipeline).

The central property: a fresh stream fed Q_tot windows in any chunking returns, for its rows g = L - 1 .. Q_tot - 1,
exactly the columns 0 .. Q_tot - L of one InferencePipeline.step over all Q_tot windows (top_val, top_idx, spike
counts), and -inf / -1 for the warm-up rows before them; the Recall@N counters summed over the pushes equal the
batch counters."""
import ctypes as C

import numpy as np
import pytest
import torch

from conftest import synth_pooled, synth_weights
from oracle import oracle as O
from test_gpu_event_streams import W_US, device_streams, kernels_run

gpu = pytest.mark.gpu
MODE_AUTO, MODE_SIMT, MODE_TC = 0, 1, 2
T, F, I = 30, 96, 100


def cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def model(P, seed=3):
    Wf, Wo = synth_weights(I, F, P, seed=seed)
    return torch.from_numpy(Wf), torch.from_numpy(Wo)


def recall_ns(N):
    from lens_b200.ops import RECALL_NS
    return tuple(n for n in RECALL_NS if n <= N)


def batch_pipe(W, L, N, B, mode):
    from lens_b200.pipeline import InferencePipeline
    return InferencePipeline(*W, roi=80, k=8, T=T, L=L, n_top=N, ns=recall_ns(N), max_streams=B, mode=mode)


def stream_pipe(W, L, N, B, mode):
    from lens_b200.pipeline import StreamingPipeline
    return StreamingPipeline(*W, roi=80, k=8, T=T, L=L, n_streams=B, n_top=N, ns=recall_ns(N), mode=mode)


def chunkings(L, Q_tot, seed):
    m = max(L - 1, 1)
    mixed = [max(m - 1, 1), m, m + 1]                 # shorter than, equal to and longer than L - 1
    mixed.append(Q_tot - sum(mixed))
    rng = np.random.default_rng(seed)
    cuts = sorted(rng.choice(np.arange(1, Q_tot), size=min(4, Q_tot - 1), replace=False).tolist())
    rand = np.diff([0] + cuts + [Q_tot]).tolist()
    out = {"ones": [1] * Q_tot, "mixed": mixed, "one_chunk": [Q_tot], "random": rand}
    assert all(min(c) >= 1 and sum(c) == Q_tot for c in out.values()), out
    return out


def streamed_gt(gt_batch, L):
    """Band ground truth per streamed row: row g >= L - 1 expects the batch column g - L + 1; warm-up rows get a
    real place (0) so that only the pipeline's masking keeps them out of the counters."""
    B, Qo = gt_batch.shape
    return torch.cat([torch.zeros((B, L - 1), dtype=torch.int32, device=gt_batch.device), gt_batch], dim=1)


def push_all(sp, pooled, chunks, gt=None, gt_tol=0):
    outs, q0 = [], 0
    for c in chunks:
        outs.append(sp.push(pooled=pooled[:, q0:q0 + c].contiguous(),
                            gt_center=None if gt is None else gt[:, q0:q0 + c].contiguous(), gt_tol=gt_tol))
        q0 += c
    cat = {k: torch.cat([o[k] for o in outs], dim=1) for k in ("top_val", "top_idx", "S")}
    if gt is not None:
        cat["hits"] = sum(o["hits"] for o in outs)
        cat["n_valid"] = sum(o["n_valid"] for o in outs)
    return cat


def assert_matches_batch(got, want, L):
    assert torch.equal(got["S"], want["S"])
    assert torch.equal(got["top_val"][:, L - 1:], want["top_val"])
    assert torch.equal(got["top_idx"][:, L - 1:], want["top_idx"])
    warm_v, warm_i = got["top_val"][:, :L - 1], got["top_idx"][:, :L - 1]
    assert bool((warm_v == float("-inf")).all()) and bool((warm_i == -1).all())
    if "hits" in got:
        assert torch.equal(got["hits"], want["hits"]) and torch.equal(got["n_valid"], want["n_valid"])


CASES = [  # (L, N, P, mode): warp kernel (N <= 32) and CTA kernel (N > 32), empty slots, ragged / tiny P
    (1, 1, 100, MODE_SIMT),
    (1, 33, 50, MODE_TC),
    (2, 25, 300, MODE_TC),
    (2, 64, 97, MODE_SIMT),       # P < 128, not a multiple of 32; N = 64 > Po = 96
    (10, 32, 300, MODE_SIMT),
    (10, 33, 200, MODE_TC),
    (10, 25, 20, MODE_SIMT),      # N > Po = 11: empty slots in the warp kernel
    (10, 64, 70, MODE_TC),        # N > Po = 61: empty slots in the CTA kernel
]


@gpu
@pytest.mark.parametrize("L,N,P,mode", CASES)
def test_any_chunking_equals_one_batch_step(L, N, P, mode):
    from lens_b200 import synth
    B, Q_tot = 3, 3 * L + 3
    W = model(P)
    pooled = cuda(synth_pooled(B, Q_tot, I, seed=L * 1000 + P))
    gt = cuda(synth.gt_centers(B, Q_tot - L + 1, P - L + 1, seed=4))
    want = batch_pipe(W, L, N, B, mode).step(pooled=pooled, gt_center=gt, gt_tol=2)
    assert float(want["S"].sum()) > 0
    for name, chunks in chunkings(L, Q_tot, seed=L + P).items():
        got = push_all(stream_pipe(W, L, N, B, mode), pooled, chunks, gt=streamed_gt(gt, L), gt_tol=2)
        try:
            assert_matches_batch(got, want, L)
        except AssertionError as e:
            raise AssertionError(f"chunking {name} {chunks}") from e


@gpu
def test_streamed_rows_equal_the_oracle():
    B, L, N, P, Q_tot = 3, 4, 25, 150, 9
    W = model(P, seed=8)
    pooled = synth_pooled(B, Q_tot, I, seed=6)
    got = push_all(stream_pipe(W, L, N, B, MODE_SIMT), cuda(pooled), [1, 2, 3, 1, 2])
    onet = O.OracleSNN(W[0].numpy(), W[1].numpy(), O.raster_uniforms(T, 80, 8), T, n_streams=B)
    So = onet.run_streams(pooled)
    assert So.sum() > 0 and np.array_equal(got["S"].cpu().numpy(), So)
    for b in range(B):
        io, vo = O.topk(O.seqmatch(So[b], L), N)
        assert np.array_equal(got["top_idx"][b, L - 1:].cpu().numpy(), io)
        assert np.array_equal(got["top_val"][b, L - 1:].cpu().numpy(), vo)


def ran(names, kernel):
    """kernel: name as the profiler prints it after `lens::`, template arguments included."""
    return any(("::" + kernel + "(") in n for n in names)


@gpu
def test_one_camera_large_map_takes_the_segmented_path():
    B, L, N, P, Q_tot = 1, 10, 25, 20000, 12         # Po = 19 991 >= 8 192, one query per push
    W = model(P, seed=5)
    pooled = cuda(synth_pooled(B, Q_tot, I, seed=9))
    want = batch_pipe(W, L, N, B, MODE_AUTO).step(pooled=pooled)
    sp = stream_pipe(W, L, N, B, MODE_AUTO)
    outs = []
    for q in range(Q_tot):
        out, names = kernels_run(lambda: sp.push(pooled=pooled[:, q:q + 1].contiguous()))
        assert ran(names, "seqmatch_topk_stream_warp_kernel<true>"), names
        assert ran(names, "topn_merge_kernel"), names
        assert not ran(names, "seqmatch_topk_stream_warp_kernel<false>"), names
        outs.append(out)
    got = {k: torch.cat([o[k] for o in outs], dim=1) for k in ("top_val", "top_idx", "S")}
    assert_matches_batch(got, want, L)


@gpu
@pytest.mark.parametrize("L", [1, 3])
def test_reset_streams_mid_session(L):
    B, N, P, Q1, Q2 = 4, 25, 160, 5, 6
    W = model(P, seed=11)
    pooled = cuda(synth_pooled(B, Q1 + Q2, I, seed=12))
    reset = [1, 3]
    a, full = stream_pipe(W, L, N, B, MODE_SIMT), stream_pipe(W, L, N, B, MODE_SIMT)
    first = push_all(a, pooled[:, :Q1], [2, 3])
    v_before = a.net.state()
    a.reset_streams(reset)
    v_after = a.net.state()
    keep = [0, 2]
    for vb, va in zip(v_before, v_after):          # lens_snn_reset_streams: unmasked rows bit-identical
        assert torch.equal(va[keep], vb[keep]) and bool((va[reset] == 0).all())
    assert bool((v_before[2][reset] != 0).any())   # the reset had something to clear
    after = push_all(a, pooled[:, Q1:], [1, 4, 1])
    whole = push_all(full, pooled, [Q1 + Q2])
    fresh = stream_pipe(W, L, N, B, MODE_SIMT)
    tail = push_all(fresh, pooled[:, Q1:], [Q2])
    for k in ("top_val", "top_idx", "S"):
        got = torch.cat([first[k], after[k]], dim=1)
        assert torch.equal(got[keep], whole[k][keep]), k            # untouched streams: as if uninterrupted
        assert torch.equal(after[k][reset], tail[k][reset]), k      # reset streams: a fresh session, warm-up included
    for va, vw, vf in zip(a.net.state(), full.net.state(), fresh.net.state()):
        assert torch.equal(va[keep], vw[keep]) and torch.equal(va[reset], vf[reset])
    # a mask works like the index list
    m = stream_pipe(W, L, N, B, MODE_SIMT)
    push_all(m, pooled[:, :Q1], [Q1])
    m.reset_streams(torch.tensor([False, True, False, True]))
    assert torch.equal(push_all(m, pooled[:, Q1:], [Q2])["top_idx"], after["top_idx"])
    # so does a list of bools (not indices 0 / 1), and a device tensor of indices
    for streams in ([False, True, False, True], torch.tensor(reset, device="cuda")):
        m = stream_pipe(W, L, N, B, MODE_SIMT)
        push_all(m, pooled[:, :Q1], [Q1])
        m.reset_streams(streams)
        assert torch.equal(push_all(m, pooled[:, Q1:], [Q2])["top_idx"], after["top_idx"]), streams


@gpu
def test_push_events_equals_step_events():
    from lens_b200 import synth
    B, Q_tot, L, N, P = 5, 7, 3, 25, 250
    W = model(P, seed=13)
    t, x, y, off, t0 = device_streams(B, Q_tot, 40_000, seed=17)
    window = W_US * 250
    gt = cuda(synth.gt_centers(B, Q_tot - L + 1, P - L + 1, seed=3))
    want = batch_pipe(W, L, N, B, MODE_SIMT).step_events(t, x, y, off, t0, window, Q_tot, roi_x0=23, gt_center=gt,
                                                         gt_tol=1)
    sp, gts = stream_pipe(W, L, N, B, MODE_SIMT), streamed_gt(gt, L)
    outs, q0 = [], 0
    for c in [2, 1, 3, 1]:
        outs.append(sp.push_events(t, x, y, off, t0 + q0 * window, window, c, roi_x0=23,
                                   gt_center=gts[:, q0:q0 + c].contiguous(), gt_tol=1))
        q0 += c
    got = {k: torch.cat([o[k] for o in outs], dim=1) for k in ("top_val", "top_idx", "S", "events_per_window")}
    got["hits"], got["n_valid"] = sum(o["hits"] for o in outs), sum(o["n_valid"] for o in outs)
    assert_matches_batch(got, want, L)
    assert torch.equal(got["events_per_window"], want["events_per_window"])
    assert int(want["n_valid"]) == B * (Q_tot - L + 1)


@gpu
def test_launch_counts_do_not_depend_on_B():
    from lens_b200 import _lib, ops
    L, N, P, Q = 10, 25, 300, 2
    counts = {}
    for B in (1, 2, 64):
        S = torch.randint(0, 20, (B, Q, P), device="cuda").float()
        ring = torch.zeros((B, L - 1, P), device="cuda")
        seen = torch.zeros((B,), dtype=torch.int32, device="cuda")
        W = model(P)
        sp = stream_pipe(W, L, N, B, MODE_SIMT)
        torch.cuda.synchronize()
        l0 = _lib.launch_count()
        ops.seqmatch_topk_stream(S, L, N, ring, seen, 0)
        l1 = _lib.launch_count()
        ops.seqmatch_topk_stream(S, L, 40, ring, seen, Q)            # CTA kernel
        l2 = _lib.launch_count()
        ops.seqmatch_topk_stream(S, 1, N, None, seen, 0)             # L = 1: no ring to append to
        l3 = _lib.launch_count()
        sp.net.reset_streams(torch.ones((B,), dtype=torch.uint8, device="cuda"))
        l4 = _lib.launch_count()
        counts[B] = (l1 - l0, l2 - l1, l3 - l2, l4 - l3)
    assert counts[1] == counts[2] == counts[64] == (2, 2, 1, 1), counts
    # segmented: one stream against many places
    S = torch.randint(0, 20, (1, 1, 20000), device="cuda").float()
    seen = torch.zeros((1,), dtype=torch.int32, device="cuda")
    l0 = _lib.launch_count()
    ops.seqmatch_topk_stream(S, L, N, torch.zeros((1, L - 1, 20000), device="cuda"), seen, 0)
    assert _lib.launch_count() - l0 == 3


@gpu
def test_wrong_stream_count_raises_and_changes_nothing():
    from lens_b200._lib import LensError
    B, L, N, P = 4, 3, 25, 120
    W = model(P, seed=2)
    pooled = cuda(synth_pooled(B + 2, 4, I, seed=3))
    sp = stream_pipe(W, L, N, B, MODE_SIMT)
    push_all(sp, pooled[:B, :3].contiguous(), [3])
    before = [v.clone() for v in sp.net.state()] + [sp.ring.clone(), sp.seen.clone()]
    t_before, h_before = sp.t, sp.net._h.value
    for bad in (pooled[:B - 2, 3:].contiguous(), pooled[:, 3:].contiguous()):
        with pytest.raises(LensError):
            sp.push(pooled=bad)
    gt_ok = torch.zeros((B, 1), dtype=torch.int32, device="cuda")
    for gt in (gt_ok[:, 0].contiguous(), gt_ok.long(), torch.zeros((B, 2), dtype=torch.int32, device="cuda")):
        with pytest.raises(LensError):                             # checked before anything runs
            sp.push(pooled=pooled[:B, 3:].contiguous(), gt_center=gt)
    for streams in ([B], [-1], [True, False], torch.ones((B,), dtype=torch.uint8), [0.0, 1.0]):
        with pytest.raises(LensError):
            sp.reset_streams(streams)
    # the batch entry points would advance the SNN state without the sequence history
    with pytest.raises(LensError):
        sp.step(pooled=pooled[:B, 3:].contiguous())
    with pytest.raises(LensError):
        sp.step(pooled=pooled[:, 3:].contiguous())
    for name in ("step_events", "step_event_groups", "step_host"):
        with pytest.raises(LensError):
            getattr(sp, name)()
    after = list(sp.net.state()) + [sp.ring, sp.seen]
    assert sp.t == t_before and sp.net._h.value == h_before and sp.net.max_streams == B
    assert all(torch.equal(a, b) for a, b in zip(after, before))


def test_argument_validation_without_a_gpu():
    from lens_b200 import _lib
    L = _lib.lib()
    a = C.c_void_p(0x10000)                                        # never dereferenced: checks come first

    def call(B=2, Q=3, P=50, Ls=4, N=25, ring=a, seen=a, t=0):
        return L.lens_seqmatch_topk_stream(a, B, Q, P, Ls, N, ring, seen, t, a, a, None)
    for kw, word in ((dict(Ls=0), b"L"), (dict(Ls=51), b"L"), (dict(N=65), b"N=65"), (dict(N=0), b"N=0"),
                     (dict(ring=None), b"ring"), (dict(seen=None), b"seen"), (dict(Q=0), b"sizes"),
                     (dict(B=-1), b"sizes"), (dict(t=-1), b"t "), (dict(B=1 << 16, Q=1 << 16), b"too many")):
        assert call(**kw) == -1, kw
        assert word in L.lens_last_error(), (kw, L.lens_last_error())
    assert call(ring=None, Ls=1, B=0) == 0                          # L == 1 needs no ring; B == 0 launches nothing
    assert L.lens_snn_reset_streams(None, a, None) == -1
    assert L.lens_snn_reset_streams(a, None, None) == -1
