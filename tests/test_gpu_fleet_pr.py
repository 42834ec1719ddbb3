"""Fleet precision-recall (InferencePipeline.precision_recall, lens_seqpr_scan / lens_seqpr_counts) against the
reference's own lists and the oracle: createPR over the streams' sequence-matched matrices concatenated along its
column axis.  Every comparison is exact: counts equal, lists equal with NaN == NaN."""
import ctypes as C
import os
import socket
import subprocess
import sys
import types

import numpy as np
import pytest
import torch

from oracle import oracle as O

gpu = pytest.mark.gpu
f32 = np.float32
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MODES = [("single", "place"), ("single", "query"), ("multi", None)]
MODE_IDS = ["place", "query", "multi"]


def cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


_PIPES = {}


def pipe(L):
    """An InferencePipeline of sequence length L (the network itself is not used by precision_recall)."""
    from lens_b200 import synth
    from lens_b200.pipeline import InferencePipeline
    if L not in _PIPES:
        Wf, Wo = synth.weights(4, 8, 3, seed=1)
        _PIPES[L] = InferencePipeline(torch.from_numpy(Wf), torch.from_numpy(Wo), roi=2, k=1, T=1, L=L, device="cuda:0")
    return _PIPES[L]


def dense_gt(gt, B, Po, Qo):
    """The ground truth of stream b as a dense bool [Po, Qo] matrix, for every b."""
    kind = gt[0]
    if kind == "dense":
        G = gt[1].astype(bool)
        return [G if G.ndim == 2 else G[b] for b in range(B)]
    centers, tol = gt[1], gt[2]
    p = np.arange(Po)[:, None]
    return [(centers[b][None, :] >= 0) & (np.abs(p - centers[b][None, :]) <= tol) for b in range(B)]


def oracle_pr(S, L, gt, matching, best, n_thresh):
    """O.create_pr over the concatenation of O.seqmatch per stream."""
    B, Q, P = S.shape
    Ds = [O.seqmatch(S[b], L) for b in range(B)]
    Gs = dense_gt(gt, B, P - L + 1, Q - L + 1)
    if matching == "single" and best == "place":
        M, G = np.concatenate([D.T for D in Ds], axis=1), np.concatenate([g.T for g in Gs], axis=1)
    else:
        M, G = np.concatenate(Ds, axis=1), np.concatenate(Gs, axis=1)
    return O.create_pr(M, G, n_thresh=n_thresh, matching=matching)


def gt_kwargs(gt):
    if gt[0] == "dense":
        return dict(gt_dense=cuda(gt[1].astype(np.uint8)))
    return dict(gt_center=cuda(gt[1].astype(np.int32)), gt_tol=gt[2])


def run_pr(S, L, gt, matching, best, n_thresh, **kw):
    return pipe(L).precision_recall(cuda(S), matching=matching, best=best, n_thresh=n_thresh, **gt_kwargs(gt), **kw)


def same_lists(got, want):
    P, R = got
    Pw, Rw = want
    assert len(P) == len(R) == len(Pw)
    assert np.array_equal(np.array(P, np.float64), np.array(Pw, np.float64), equal_nan=True)
    assert np.array_equal(np.array(R, np.float64), np.array(Rw, np.float64), equal_nan=True)


def check(S, L, gt, matching, best, n_thresh):
    out = run_pr(S, L, gt, matching, best, n_thresh)
    same_lists((out["P"], out["R"]), oracle_pr(S, L, gt, matching, best, n_thresh))
    return out


def spikes(rng, B, Q, P, lam=1.3):
    return rng.poisson(lam, size=(B, Q, P)).astype(f32)


def band(rng, B, Qo, Po, tol, no_pos=0.15):
    c = rng.integers(0, Po, size=(B, Qo)).astype(np.int32)
    c[rng.random((B, Qo)) < no_pos] = -1
    c[0, 0] = 0                                   # the map's ends
    c[-1, -1] = Po - 1
    return ("band", c, tol)


# --------------------------------------------------------------------------- CPU: arguments and the table property
def test_arguments_are_rejected_without_a_gpu():
    from lens_b200 import ops
    from lens_b200.pipeline import InferencePipeline
    S = torch.zeros((2, 5, 7), dtype=torch.float32)
    c = torch.zeros((2, 4), dtype=torch.int32)
    me = types.SimpleNamespace(L=2)
    pr = InferencePipeline.precision_recall
    for kw, what in [(dict(n_thresh=1), "n_thresh"), (dict(n_thresh=4097), "n_thresh"),
                     (dict(matching="multiple"), "matching"), (dict(best="stream"), "matching")]:
        with pytest.raises(ValueError, match=what):
            pr(me, S, gt_center=c, **kw)
    with pytest.raises(ValueError, match="exactly one"):
        pr(me, S)
    with pytest.raises(ValueError, match="exactly one"):
        pr(me, S, gt_center=c, gt_dense=torch.zeros((6, 4), dtype=torch.uint8))
    with pytest.raises(ValueError, match="gt_center"):
        pr(me, S, gt_center=torch.zeros((2, 5), dtype=torch.int32))
    with pytest.raises(ValueError, match="gt_dense"):
        pr(me, S, gt_dense=torch.zeros((4, 6), dtype=torch.uint8))      # [Qo, Po] instead of [Po, Qo]
    with pytest.raises(ValueError, match="gt_dense"):
        pr(me, S, gt_dense=torch.zeros((3, 6, 4), dtype=torch.uint8))
    for L in (0, 6):
        with pytest.raises(ValueError, match="L"):
            pr(types.SimpleNamespace(L=L), S, gt_center=c)
    with pytest.raises(ValueError, match="S must be"):
        pr(me, S.double(), gt_center=c)
    with pytest.raises(ValueError, match="n_thresh"):
        ops.seqpr_counts(S, 2, 0, None, None, 5000, gt_center=c)


def test_abi_rejects_bad_arguments_before_any_cuda_call():
    from lens_b200 import _lib
    L = _lib.lib()
    n = C.c_int64(0)
    cases = [
        (lambda: L.lens_seqpr_scan(None, 1, 4, 4, 5, 0, None, 0, C.c_void_p(8), 0, C.c_void_p(8), C.c_void_p(8),
                           C.c_void_p(8), None), b"L"),
        (lambda: L.lens_seqpr_scan(None, 1, 4, 4, 2, 3, None, 0, C.c_void_p(8), 0, C.c_void_p(8), C.c_void_p(8),
                           C.c_void_p(8), None), b"mode"),
        (lambda: L.lens_seqpr_scan(C.c_void_p(8), 1, 4, 4, 2, 0, C.c_void_p(8), 0, C.c_void_p(8), 0, C.c_void_p(8),
                           C.c_void_p(8), C.c_void_p(8), None), b"exactly one"),
        (lambda: L.lens_seqpr_scan(C.c_void_p(8), 1, 4, 4, 2, 0, None, 0, C.c_void_p(8), 0, C.c_void_p(12), C.c_void_p(8),
                           C.c_void_p(8), None), b"aligned"),
        (lambda: L.lens_seqpr_counts(C.c_void_p(8), 1, 4, 4, 2, 2, None, 0, C.c_void_p(8), 0, None, C.c_void_p(8), 1,
                             C.c_void_p(8), C.c_void_p(8), None), b"n_thresh"),
        (lambda: L.lens_seqpr_counts(C.c_void_p(8), 1, 4, 4, 2, 2, None, 0, C.c_void_p(8), 0, None, C.c_void_p(8), 4097,
                             C.c_void_p(8), C.c_void_p(8), None), b"n_thresh"),
        (lambda: L.lens_seqpr_records_bytes(1, 4, 4, 0, 0, C.byref(n)), b"sizes"),
    ]
    for call, what in cases:
        assert call() == -1 and what in L.lens_last_error(), L.lens_last_error()
    for mode, want in ((0, 5 * 3 * 2), (1, 9 * 3 * 3), (2, 0)):
        assert L.lens_seqpr_records_bytes(3, 4, 3, 2, mode, C.byref(n)) == 0 and n.value == want


def test_linspace32_is_non_increasing_before_its_last_element():
    """The property binning by binary search rests on: np.linspace(max, min, n) in float32 is non-increasing over
    indices 0 .. n - 2 (only the last element, forced to `stop`, can break the order), over the ranges of
    test_gpu_metrics.test_linspace32_restates_numpy plus the subnormal pair whose table does break at the end."""
    rng = np.random.default_rng(0)
    cases = [(1.0, 0.0), (10.0, 0.0), (2.5, 2.5), (0.0, 0.0), (1e-45, 0.0), (3e-45, -1e-45), (1e-38, 0.0),
             (1.7e38, -1.7e38), (-0.1, -7.3), (5.0, 1e-45)]
    cases += [tuple(sorted(rng.standard_normal(2) * 10.0 ** rng.integers(-40, 38), reverse=True)) for _ in range(40)]
    cases += [(float(k) / 10, 0.0) for k in range(1, 30)]
    cases += [(1.607e-43, 8.83e-44)]
    for start, stop in cases:
        for n in (2, 3, 7, 100, 101, 4096, 65535):
            y = np.linspace(f32(start), f32(stop), n)
            assert y.dtype == np.float32
            assert np.all(y[1:n - 1] <= y[:n - 2]), (start, stop, n)
    y = np.linspace(f32(1.607e-43), f32(8.83e-44), 100)
    assert y[98] < y[99]                          # the case test_subnormal_table_out_of_order runs on the GPU


# --------------------------------------------------------------------------- against the reference's own lists
@gpu
@pytest.mark.parametrize("name", ["config1", "brisevent"])
def test_reference_pr_curve(name):
    """--PR_curve of the reference (createPR(D.T, GTtol.T, 'single')) from the spike counts, per place."""
    g = np.load(os.path.join(ROOT, "tests", "golden", f"{name}.npz"))
    L = int(g["sequence_length"])
    out = run_pr(g["S"].astype(f32)[None], L, ("dense", g["GTtol"]), "single", "place", 100)
    same_lists((out["P"], out["R"]), (g["PR_P"], g["PR_R"]))


@gpu
def test_reference_sad_pr_curve():
    """The SAD path's createPR(sim, GTtol, 'single'): best place per query, S = simᵀ at L = 1."""
    g = np.load(os.path.join(ROOT, "tests", "golden", "config1.npz"))
    out = run_pr(np.ascontiguousarray(g["sad_sim"].T)[None], 1, ("dense", g["GTtol"]), "single", "query", 100)
    same_lists((out["P"], out["R"]), (g["sad_P"], g["sad_R"]))


# --------------------------------------------------------------------------- against the oracle
@gpu
@pytest.mark.parametrize("mode", MODES, ids=MODE_IDS)
@pytest.mark.parametrize("B,Q,P,L", [(1, 12, 200, 1), (3, 12, 200, 2), (64, 11, 200, 10), (3, 10, 333, 10),
                                     (64, 2, 97, 2), (1, 12, 70000, 10)])
def test_oracle_shapes(mode, B, Q, P, L):
    """B in {1, 3, 64}, L in {1, 2, 10}, Po not a multiple of 32, Qo = 1, a 70 000-place map; band ground truth."""
    rng = np.random.default_rng(B * 1000 + Q * 10 + L)
    S = spikes(rng, B, Q, P)
    check(S, L, band(rng, B, Q - L + 1, P - L + 1, 2), *mode, 100)


@gpu
@pytest.mark.parametrize("mode", MODES, ids=MODE_IDS)
@pytest.mark.parametrize("per_stream", [False, True], ids=["shared", "per_stream"])
def test_oracle_dense_gt(mode, per_stream):
    rng = np.random.default_rng(5)
    B, Q, P, L = 3, 14, 150, 3
    Po, Qo = P - L + 1, Q - L + 1
    G = rng.random((B, Po, Qo) if per_stream else (Po, Qo)) < 0.05
    G[..., 2] = False                                                    # a query without positives
    G[..., 7, :] = False                                                 # a place without positives
    check(spikes(rng, B, Q, P), L, ("dense", G), *mode, 100)


@gpu
@pytest.mark.parametrize("mode", MODES, ids=MODE_IDS)
@pytest.mark.parametrize("tol", [0, 1, 2, 3])
def test_oracle_band_tolerance(mode, tol):
    """Centres at -1, 0 and Po - 1 in every stream; |p - c| <= tol, inclusive."""
    rng = np.random.default_rng(tol)
    B, Q, P, L = 3, 9, 120, 2
    Po, Qo = P - L + 1, Q - L + 1
    _, c, _ = band(rng, B, Qo, Po, tol)
    c[:, 1], c[:, 2], c[:, 3] = -1, 0, Po - 1
    check(spikes(rng, B, Q, P, lam=2.0), L, ("band", c, tol), *mode, 100)


@gpu
@pytest.mark.parametrize("mode", MODES, ids=MODE_IDS)
@pytest.mark.parametrize("n_thresh", [2, 3, 100, 101, 4096])
def test_oracle_thresholds(mode, n_thresh):
    rng = np.random.default_rng(n_thresh)
    B, Q, P, L = 3, 12, 130, 10
    check(spikes(rng, B, Q, P), L, band(rng, B, Q - L + 1, P - L + 1, 1), *mode, n_thresh)


@gpu
@pytest.mark.parametrize("mode", MODES, ids=MODE_IDS)
def test_tied_maxima_take_the_first(mode):
    """Columns whose maximum is tied between a positive and a negative entry, in both orders: the first maximum
    (lowest query per place, lowest place per query) decides the hit, as np.argmax does."""
    B, Q, P, L = 2, 6, 40, 1
    S = np.zeros((B, Q, P), f32)
    G = np.zeros((P, Q), bool)                     # [Po, Qo] shared
    # per place: place 3 ties at queries 1 (positive) and 4 (negative); place 5 the other way round
    S[:, 1, 3] = S[:, 4, 3] = 7
    G[3, 1] = True
    S[:, 1, 5] = S[:, 4, 5] = 7
    G[5, 4] = True
    # per query: query 2 ties at places 10 (positive) and 20 (negative); query 3 the other way round
    S[:, 2, 10] = S[:, 2, 20] = 5
    G[10, 2] = True
    S[:, 3, 10] = S[:, 3, 20] = 5
    G[20, 3] = True
    S[1] += (np.arange(P) % 3 == 0)[None, :].astype(f32)             # a second stream with other values
    for n in (2, 7, 100):
        check(S, L, ("dense", G), *mode, n)


@gpu
@pytest.mark.parametrize("mode", MODES, ids=MODE_IDS)
def test_constant_matrix(mode):
    """step = 0: every threshold equals the value, every column counts at every threshold."""
    B, Q, P, L = 2, 5, 70, 2
    rng = np.random.default_rng(1)
    out = check(np.full((B, Q, P), 3.0, f32), L, band(rng, B, Q - L + 1, P - L + 1, 1), *mode, 100)
    assert len(set(out["tp"].tolist())) == 1


@gpu
@pytest.mark.parametrize("mode", MODES, ids=MODE_IDS)
def test_subnormal_table_out_of_order(mode):
    """L = 1 and the values {8.83e-44, 1.607e-43} at n_thresh = 100: the float32 table has y[98] < y[99] = min, so
    only the rule 'threshold n - 1 counts everything' bins the minimum right."""
    lo, hi = f32(8.83e-44), f32(1.607e-43)
    y = np.linspace(hi, lo, 100)
    assert y[98] < y[99]
    rng = np.random.default_rng(2)
    B, Q, P = 2, 6, 50
    S = np.where(rng.random((B, Q, P)) < 0.5, lo, hi).astype(f32)
    S[0, :, 0] = lo                                # a column whose best is the minimum (per place)
    S[1, 0, :] = lo                                # and one per query
    check(S, 1, band(rng, B, Q, P, 2), *mode, 100)


@gpu
def test_counts_and_invariants():
    """tp[-1] + fp[-1] counts every column (every entry in multi mode); gtp counts what createPR counts."""
    rng = np.random.default_rng(9)
    B, Q, P, L = 5, 9, 110, 3
    Po, Qo = P - L + 1, Q - L + 1
    gt = band(rng, B, Qo, Po, 1)
    Gs = dense_gt(gt, B, Po, Qo)
    n_cols = {"place": B * Po, "query": B * Qo, None: B * Po * Qo}
    gtp = {"place": sum(int(g.any(1).sum()) for g in Gs), "query": sum(int(g.any(0).sum()) for g in Gs),
           None: sum(int(g.sum()) for g in Gs)}
    for matching, best in MODES:
        out = check(spikes(rng, B, Q, P), L, gt, matching, best, 100)
        assert out["tp"][-1] + out["fp"][-1] == n_cols[best]
        assert out["gtp"] == gtp[best]
        assert np.all(np.diff(out["tp"]) >= 0) and np.all(np.diff(out["fp"]) >= 0)


# --------------------------------------------------------------------------- split invariance
@gpu
@pytest.mark.parametrize("mode", MODES, ids=MODE_IDS)
def test_two_groups_make_one_fleet(mode):
    """Two halves of a fleet scanned into one {max, min} / gtp and counted separately: the summed counts are the
    whole fleet's, which differ from either half's own curve."""
    from lens_b200 import ops
    rng = np.random.default_rng(4)
    B, Q, P, L = 6, 8, 90, 2
    S = spikes(rng, B, Q, P)
    S[:3] *= 2                                     # the halves have different ranges
    _, c, _ = band(rng, B, Q - L + 1, P - L + 1, 1)
    m = ops.seqpr_mode(*mode)
    whole = check(S, L, ("band", c, 1), *mode, 50)
    halves = [(cuda(S[:3]), cuda(c[:3])), (cuda(S[3:]), cuda(c[3:]))]
    ext = torch.zeros(2, dtype=torch.int64, device="cuda")
    gtp = torch.zeros(1, dtype=torch.int64, device="cuda")
    recs = [ops.seqpr_scan(s, L, m, gt_center=g, gt_tol=1, extremes=ext, gtp=gtp)[0] for s, g in halves]
    counts = [ops.seqpr_counts(s, L, m, r, ext, 50, gt_center=g, gt_tol=1) for (s, g), r in zip(halves, recs)]
    tp = sum(t.cpu().numpy() for t, _ in counts)
    fp = sum(f.cpu().numpy() for _, f in counts)
    assert np.array_equal(tp, whole["tp"]) and np.array_equal(fp, whole["fp"]) and int(gtp.item()) == whole["gtp"]
    own = run_pr(S[3:], L, ("band", c[3:], 1), *mode, 50)
    assert not np.array_equal(own["tp"], counts[1][0].cpu().numpy())


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@gpu
def test_two_ranks_equal_one_rank():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
           "--master-addr", "127.0.0.1", "--master-port", str(_free_port()),
           os.path.join(ROOT, "tests", "fleet_pr_dist_check.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-2000:]
    assert "OK" in res.stdout, res.stdout[-2000:]


# --------------------------------------------------------------------------- structure
def kernels_and_launches(fn):
    from torch.profiler import profile, ProfilerActivity
    from lens_b200._lib import launch_count
    n0 = launch_count()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = ["".join(e.name.split()) for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    return [n for n in names if "kernel" in n], launch_count() - n0


@gpu
@pytest.mark.parametrize("mode", MODES, ids=MODE_IDS)
def test_kernels_and_launch_count_do_not_grow_with_B(mode):
    rng = np.random.default_rng(3)
    Q, P, L = 4, 300, 2
    seen = {}
    for B in (2, 512):
        S = cuda(spikes(rng, B, Q, P))
        c = cuda(band(rng, B, Q - L + 1, P - L + 1, 1)[1])
        pipe(L).precision_recall(S, gt_center=c, gt_tol=1, matching=mode[0], best=mode[1])    # warm-up
        names, launches = kernels_and_launches(
            lambda: pipe(L).precision_recall(S, gt_center=c, gt_tol=1, matching=mode[0], best=mode[1]))
        ours = sorted(n for n in names if "seqpr" in n)
        assert any("seqpr_scan_kernel" in n for n in ours) and any("seqpr_count_kernel" in n for n in ours)
        assert any("seqpr_prefix_kernel" in n for n in ours)
        seen[B] = (ours, launches)
    assert seen[2] == seen[512]
    assert seen[2][1] == (4 if mode[1] == "query" else 3)


@gpu
@pytest.mark.parametrize("mode", MODES, ids=MODE_IDS)
def test_memory_grows_by_the_records_not_by_D(mode):
    from lens_b200 import _lib, ops
    rng = np.random.default_rng(6)
    B, Q, P, L = 64, 64, 2000, 2
    S = cuda(spikes(rng, B, Q, P))
    c = cuda(band(rng, B, Q - L + 1, P - L + 1, 1)[1])
    n = C.c_int64(0)
    _lib.check(_lib.lib().lens_seqpr_records_bytes(B, Q, P, L, ops.seqpr_mode(*mode), C.byref(n)))
    d_bytes = B * (P - L + 1) * (Q - L + 1) * 4
    pipe(L).precision_recall(S, gt_center=c, gt_tol=1, matching=mode[0], best=mode[1])
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    pipe(L).precision_recall(S, gt_center=c, gt_tol=1, matching=mode[0], best=mode[1])
    torch.cuda.synchronize()
    grown = torch.cuda.max_memory_allocated() - base
    assert grown <= n.value + (1 << 20), (grown, n.value)
    assert grown < d_bytes // 8


@gpu
def test_streaming_pipeline_refuses():
    from lens_b200 import synth
    from lens_b200._lib import LensError
    from lens_b200.pipeline import StreamingPipeline
    Wf, Wo = synth.weights(4, 8, 3, seed=1)
    sp = StreamingPipeline(torch.from_numpy(Wf), torch.from_numpy(Wo), roi=2, k=1, T=1, L=2, n_streams=2)
    with pytest.raises(LensError, match="live session"):
        sp.precision_recall(torch.zeros((2, 3, 3), device="cuda"), gt_center=torch.zeros((2, 2), dtype=torch.int32,
                                                                                          device="cuda"))
