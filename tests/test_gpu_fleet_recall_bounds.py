"""Tie-aware Recall@N bounds for whole fleets and live sessions, straight from the spike counts
(lens_seq_recall_bounds, lens_seq_recall_bounds_stream, lens_seq_recall_bounds_stream_ids, `bounds=True`).

Every count is compared for exact equality: against lens_recall_bounds on each stream's own sequence-matched matrix
(which tests/test_gpu_metrics.py pins to the oracle) and against the oracle itself on sampled streams; for pushes,
against the batch bounds over each stream's valid rows since its last reset."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import oracle as O
from test_gpu_fleet_pr import _free_port
from test_gpu_stream_subsets import Fleet, schedule, stream_pipe
from test_gpu_event_streams import kernels_run
from test_gpu_streaming import MODE_AUTO, MODE_SIMT, batch_pipe, chunkings, cuda, model, recall_ns

gpu = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEFAULT_NS = (1, 5, 10, 15, 20, 25)
NS_SETS = (DEFAULT_NS, (1,), (2, 3, 40))


# --------------------------------------------------------------------------- CPU: argument checks
def test_abi_rejects_bad_arguments_before_any_cuda_call():
    from lens_b200 import _lib
    L = _lib.lib()
    a = C.c_void_p(0x10000)                                        # never dereferenced: checks come first
    ns_ok = (C.c_int * 3)(1, 5, 10)

    def batch(B=2, Q=5, P=50, Ls=3, dense=a, stride=0, center=None, tol=0, ns=ns_ok, n_ns=3, lo=a, S=a):
        return L.lens_seq_recall_bounds(S, B, Q, P, Ls, dense, stride, center, tol, ns, n_ns, lo, a, a, None)

    def stream(B=2, Q=3, P=50, Ls=4, ring=a, seen=a, t=0, gt=a, ns=ns_ok, n_ns=3):
        return L.lens_seq_recall_bounds_stream(a, B, Q, P, Ls, ring, seen, t, gt, 0, ns, n_ns, a, a, a, None)

    def ids(n=2, Q=3, P=50, Ls=4, idv=a, B=4, rows=a, gt=a, ns=ns_ok, hi=a):
        return L.lens_seq_recall_bounds_stream_ids(a, n, Q, P, Ls, idv, B, a, a, rows, gt, 0, ns, 3, a, hi, a, None)
    desc = (C.c_int * 3)(5, 1, 10)
    zero = (C.c_int * 1)(0)
    for call, what in [(lambda: batch(Ls=6), b"L"), (lambda: batch(Ls=0), b"L"), (lambda: batch(B=-1), b"sizes"),
                       (lambda: batch(Q=0), b"sizes"), (lambda: batch(dense=None), b"exactly one"),
                       (lambda: batch(center=a), b"exactly one"), (lambda: batch(stride=-1), b">= 0"),
                       (lambda: batch(dense=None, center=a, tol=-1), b">= 0"), (lambda: batch(S=None), b"NULL S"),
                       (lambda: batch(ns=desc), b"ascending"), (lambda: batch(ns=zero, n_ns=1), b"ascending"),
                       (lambda: batch(n_ns=9), b"n_ns"), (lambda: batch(n_ns=0), b"n_ns"),
                       (lambda: batch(ns=None), b"n_ns"), (lambda: batch(lo=None), b"NULL lo"),
                       (lambda: batch(B=1 << 16, Q=1 << 16, Ls=1), b"too many"),
                       (lambda: stream(Ls=51), b"L"), (lambda: stream(t=-1), b"t and gt_tol"),
                       (lambda: stream(seen=None), b"NULL"), (lambda: stream(gt=None), b"NULL"),
                       (lambda: stream(ring=None), b"ring"), (lambda: stream(ns=desc), b"ascending"),
                       (lambda: stream(B=1 << 16, Q=1 << 16), b"too many"),
                       (lambda: ids(idv=None), b"ids"), (lambda: ids(rows=None), b"rows"), (lambda: ids(B=-1), b"fleet"),
                       (lambda: ids(gt=None), b"NULL"), (lambda: ids(hi=None), b"NULL lo"),
                       (lambda: ids(ns=desc), b"ascending")]:
        assert call() == -1 and what in L.lens_last_error(), (what, L.lens_last_error())
    # no stream: nothing to count, no launch (and no CUDA call)
    assert batch(B=0, S=None) == 0 and stream(B=0, seen=None, gt=None, ring=None) == 0
    assert ids(n=0, idv=None, rows=None, gt=None) == 0
    assert stream(Ls=1, ring=None, B=0) == 0


def test_ops_checks_shapes_without_a_gpu():
    from lens_b200 import ops
    S = torch.zeros((2, 5, 50))
    dense, c = torch.zeros((48, 3), dtype=torch.uint8), torch.zeros((2, 3), dtype=torch.int32)
    for kw, what in [(dict(S=S.double(), gt_dense=dense), "S must"), (dict(S=S, gt_dense=dense, L=6), "L <="),
                     (dict(S=S), "exactly one"), (dict(S=S, gt_dense=dense, gt_center=c), "exactly one"),
                     (dict(S=S, gt_dense=dense[:, :2]), "gt_dense"), (dict(S=S, gt_center=c.long()), "gt_center"),
                     (dict(S=S, gt_center=c, gt_tol=-1), "gt_tol"), (dict(S=S, gt_center=c, ns=(5, 1)), "ns"),
                     (dict(S=S, gt_center=c, ns=()), "ns"), (dict(S=S, gt_center=c, ns=tuple(range(1, 10))), "ns"),
                     (dict(S=S, gt_center=c, ns=(0, 1)), "ns"),
                     (dict(S=S, gt_center=c, lo=torch.zeros(3, dtype=torch.int64)), "lo")]:
        args = dict(L=3)
        args.update(kw)
        with pytest.raises(ValueError, match=what):
            ops.seq_recall_bounds(args.pop("S"), args.pop("L"), **args)
    ring, seen, rows = torch.zeros((4, 2, 50)), torch.zeros((4,), dtype=torch.int32), torch.zeros(4, dtype=torch.int64)
    Ss, cs = torch.zeros((4, 3, 50)), torch.zeros((4, 3), dtype=torch.int32)
    for args, what in [((Ss.double(), 3, ring, seen, 0, cs), "S must"), ((Ss, 3, ring[:, :1], seen, 0, cs), "ring"),
                       ((Ss, 3, ring, seen[:2], 0, cs), "seen"), ((Ss, 3, ring, seen, 0, cs[:2]), "gt_center"),
                       ((Ss, 3, ring, seen, -1, cs), "t must")]:
        with pytest.raises(ValueError, match=what):
            ops.seq_recall_bounds_stream(*args)
    S2, ids, c2 = torch.zeros((2, 3, 50)), torch.zeros((2,), dtype=torch.int32), torch.zeros((2, 3), dtype=torch.int32)
    for args, what in [((S2.double(), 3, ids, ring, seen, rows, c2), "S must"),
                       ((S2, 3, ids[:1], ring, seen, rows, c2), "ids"), ((S2, 3, ids.long(), ring, seen, rows, c2), "ids"),
                       ((S2, 3, ids, ring, seen, rows.int(), c2), "rows"), ((S2, 3, ids, ring[:2], seen, rows, c2), "ring"),
                       ((S2, 3, ids, ring, seen, rows, c2[:1]), "gt_center")]:
        with pytest.raises(ValueError, match=what):
            ops.seq_recall_bounds_stream_ids(*args)


# --------------------------------------------------------------------------- references
def band_dense(centres, Po, tol):
    """Band ground truth i32 [Qo] -> the equivalent dense u8 [Po, Qo] (what lens_recall_bounds takes)."""
    c = np.asarray(centres)[None, :]
    p = np.arange(Po)[:, None]
    return ((c >= 0) & (np.abs(p - c) <= tol)).astype(np.uint8)


def per_stream_reference(S, L, ns, gt_dense=None, gt_center=None, tol=0):
    """(lo, hi, n_valid) numpy: lens_recall_bounds on every stream's own D (seqmatch_topk, want_D=True), summed;
    n_valid from lens_recall (a band column outside [0, Po) is valid for it, but has no positive in dense form)."""
    from lens_b200 import ops
    B, Q, P = S.shape
    Qo, Po = Q - L + 1, P - L + 1
    lo, hi = np.zeros(len(ns), np.int64), np.zeros(len(ns), np.int64)
    for b in range(B):
        _, _, D = ops.seqmatch_topk(S[b:b + 1].contiguous(), L, 1, want_D=True)
        if gt_dense is not None:
            G = gt_dense if gt_dense.dim() == 2 else gt_dense[b]
        else:
            G = cuda(band_dense(gt_center[b].cpu().numpy(), Po, tol))
        l, h, _ = ops.recall_bounds(D[0], G.contiguous(), ns)
        lo += l.cpu().numpy()
        hi += h.cpu().numpy()
    _, ti, _ = ops.seqmatch_topk(S, L, 1)
    _, nv = ops.recall_counts(ti, Po, gt_dense=gt_dense, gt_center=gt_center, gt_tol=tol, ns=(1,))
    return lo, hi, int(nv.item())


def oracle_counts(S, L, ns, G):
    """The oracle's bounds on one stream: S [1, Q, P] device, G u8 [Po, Qo] numpy -> (lo, hi) counts."""
    from lens_b200 import ops
    _, _, D = ops.seqmatch_topk(S, L, 1, want_D=True)
    D = D[0].cpu().numpy()
    n = int((G.sum(0) > 0).sum())
    lo, hi = [], []
    for K in ns:
        fl, fh = O.recall_bounds(D, G, K) if n else (0.0, 0.0)
        lo.append(int(round(fl * n)))
        hi.append(int(round(fh * n)))
    return np.array(lo), np.array(hi)


def spike_counts(kind, B, Q, P, seed):
    rng = np.random.default_rng(seed)
    if kind == "constant":
        return np.full((B, Q, P), 2.0, np.float32)
    lam = {"poisson": 0.8, "planted": 0.3}[kind]
    return rng.poisson(lam, size=(B, Q, P)).astype(np.float32)


def planted_centres(S, L, rank, order):
    """Per column, the lowest (order 'low') or highest ('high') place of the tie group at the rank-th largest value of
    D: positives in tie groups that straddle K, on either side of their negatives in index order."""
    from lens_b200 import ops
    _, _, D = ops.seqmatch_topk(S, L, 1, want_D=True)
    D = D.cpu().numpy()
    B, Po, Qo = D.shape
    c = np.empty((B, Qo), np.int32)
    for b in range(B):
        for q in range(Qo):
            col = D[b, :, q]
            v = np.sort(col)[::-1][min(rank, Po - 1)]
            where = np.flatnonzero(col == v)
            c[b, q] = where[0] if order == "low" else where[-1]
    return c


def check_batch(S, L, ns, gt_dense=None, gt_center=None, tol=0, oracle_streams=2):
    from lens_b200 import ops
    lo, hi, nv = ops.seq_recall_bounds(S, L, gt_dense=gt_dense, gt_center=gt_center, gt_tol=tol, ns=ns)
    rlo, rhi, rnv = per_stream_reference(S, L, ns, gt_dense=gt_dense, gt_center=gt_center, tol=tol)
    assert np.array_equal(lo.cpu().numpy(), rlo) and np.array_equal(hi.cpu().numpy(), rhi), (lo, rlo, hi, rhi)
    assert int(nv.item()) == rnv
    B, Q, P = S.shape
    Po = P - L + 1
    for b in sorted({0, B - 1})[:oracle_streams]:
        one = S[b:b + 1].contiguous()
        if gt_dense is not None:
            g1 = gt_dense if gt_dense.dim() == 2 else gt_dense[b]
            G = g1.cpu().numpy()
            l1, h1, _ = ops.seq_recall_bounds(one, L, gt_dense=g1.contiguous(), ns=ns)
        else:
            G = band_dense(gt_center[b].cpu().numpy(), Po, tol)
            l1, h1, _ = ops.seq_recall_bounds(one, L, gt_center=gt_center[b:b + 1].contiguous(), gt_tol=tol, ns=ns)
        olo, ohi = oracle_counts(one, L, ns, G)
        assert np.array_equal(l1.cpu().numpy(), olo) and np.array_equal(h1.cpu().numpy(), ohi), (b, l1, olo, h1, ohi)
    return lo, hi, nv


def centres_grid(rng, B, Qo, Po, tol):
    """Band centres mixing -1, 0, Po - 1, Po + tol (outside the map: valid, never a hit) and random places."""
    c = rng.integers(0, Po, size=(B, Qo)).astype(np.int32)
    special = np.array([-1, 0, Po - 1, Po + tol, Po + tol + 5], np.int32)
    pick = rng.random((B, Qo)) < 0.4
    c[pick] = rng.choice(special, size=int(pick.sum()))
    return c


# --------------------------------------------------------------------------- batch against the references
@gpu
@pytest.mark.parametrize("B", [1, 3, 64])
@pytest.mark.parametrize("L", [1, 2, 10])
@pytest.mark.parametrize("kind", ["poisson", "constant", "planted"])
def test_batch_bounds_equal_per_stream_reference(B, L, kind):
    rng = np.random.default_rng(B * 100 + L)
    Q, P = 14, 203 + 7 * B % 5                                     # ragged P
    S = cuda(spike_counts(kind, B, Q, P, seed=B + L))
    Qo, Po = Q - L + 1, P - L + 1
    for i, ns in enumerate(NS_SETS):
        tol = i % 4
        if kind == "planted":
            for order in ("low", "high"):
                c = cuda(planted_centres(S, L, rank=[0, 2, 4][i], order=order))
                check_batch(S, L, ns, gt_center=c, tol=0)
        else:
            check_batch(S, L, ns, gt_center=cuda(centres_grid(rng, B, Qo, Po, tol)), tol=tol)
        shared = cuda((rng.random((Po, Qo)) < 0.03).astype(np.uint8))
        shared[:, 0] = 0                                            # a column without a positive: not valid
        check_batch(S, L, ns, gt_dense=shared)
        per = cuda((rng.random((B, Po, Qo)) < 0.02).astype(np.uint8))
        check_batch(S, L, ns, gt_dense=per)


@gpu
@pytest.mark.parametrize("tol", [0, 1, 2, 3])
def test_band_tolerances_at_the_ends_of_the_map(tol):
    L, B, Q, P = 3, 5, 9, 120
    Po = P - L + 1
    S = cuda(spike_counts("poisson", B, Q, P, seed=tol))
    base = np.array([-1, 0, 1, Po - 1, Po - 2, Po + tol, Po + tol + 3], np.int32)
    c = np.resize(base, (B, Q - L + 1)).astype(np.int32)
    for ns in NS_SETS:
        check_batch(S, L, ns, gt_center=cuda(c), tol=tol)


@gpu
def test_small_shapes_qo_one_and_few_places():
    for (B, Q, P, L) in [(3, 10, 60, 10), (4, 5, 7, 2), (2, 1, 30, 1), (5, 3, 3, 3)]:   # Qo = 1, Po < max(ns), Po = 1
        S = cuda(spike_counts("poisson", B, Q, P, seed=Q + P))
        Qo, Po = Q - L + 1, P - L + 1
        rng = np.random.default_rng(P)
        for ns in NS_SETS:
            check_batch(S, L, ns, gt_center=cuda(rng.integers(-1, Po + 1, size=(B, Qo)).astype(np.int32)), tol=1)
            check_batch(S, L, ns, gt_dense=cuda((rng.random((Po, Qo)) < 0.3).astype(np.uint8)))


@gpu
def test_one_camera_against_a_100k_place_map_takes_the_segmented_path():
    from lens_b200 import _lib, ops
    L, Q, P = 10, 12, 100_009
    S = cuda(spike_counts("poisson", 1, Q, P, seed=5))
    Qo, Po = Q - L + 1, P - L + 1
    rng = np.random.default_rng(5)
    c = rng.integers(0, Po, size=(1, Qo)).astype(np.int32)
    _, ti, _ = ops.seqmatch_topk(S, L, 1)
    c[0, 0] = int(ti[0, 0, 0])                                     # a centre at K4's own top-1: scanned to the end
    for ns in (DEFAULT_NS, (2, 3, 40)):
        check_batch(S, L, ns, gt_center=cuda(c), tol=2, oracle_streams=1)
    n0 = _lib.launch_count()
    ops.seq_recall_bounds(S, L, gt_center=cuda(c), gt_tol=2)
    assert _lib.launch_count() - n0 == 3


# --------------------------------------------------------------------------- invariants and the reference anchor
@gpu
@pytest.mark.parametrize("L", [1, 2, 10])
def test_bounds_bracket_the_step_and_share_its_n_valid(L):
    from lens_b200 import ops
    B, Q, P = 6, 16, 300
    pipe = batch_pipe(model(P), L, 25, B, MODE_AUTO)
    S = cuda(spike_counts("poisson", B, Q, P, seed=L))
    rng = np.random.default_rng(L)
    c = cuda(centres_grid(rng, B, Q - L + 1, P - L + 1, 1))
    out = pipe.match(S, gt_center=c, gt_tol=1, bounds=True)
    lo, hi, h = out["hits_lo"].cpu(), out["hits_hi"].cpu(), out["hits"].cpu()
    assert bool((lo <= h).all() and (h <= hi).all()) and bool((lo < hi).any()), (lo, h, hi)
    _, _, nv = ops.seq_recall_bounds(S, L, gt_center=c, gt_tol=1, ns=pipe.ns)
    assert torch.equal(nv, out["n_valid"])
    # no two D of a column tie: the bounds collapse onto the deterministic hits
    for seed in range(20):
        S = cuda(np.random.default_rng(seed).random((B, Q, P), dtype=np.float32))
        _, _, D = ops.seqmatch_topk(S, L, 1, want_D=True)
        D = D.cpu().numpy()
        if all(len(np.unique(D[b, :, q])) == D.shape[1] for b in range(B) for q in range(D.shape[2])):
            break
    else:
        pytest.fail("could not draw S without ties")
    out = pipe.match(S, gt_center=c, gt_tol=1, bounds=True)
    assert torch.equal(out["hits_lo"], out["hits"]) and torch.equal(out["hits_hi"], out["hits"])


@gpu
def test_config1_golden_matches_evaluate_and_brackets_the_reference(golden):
    from lens_b200.src.metrics import recall_detail
    g = golden("config1")
    L = int(g["sequence_length"])
    S = cuda(g["S"].astype(np.float32)[None])
    pipe = batch_pipe(model(S.shape[2]), L, 25, 1, MODE_AUTO)
    GT = g["GTtol"]
    out = pipe.match(S, gt_dense=cuda(GT.astype(np.uint8)), bounds=True)
    nv = int(out["n_valid"].item())
    det = recall_detail(g["D"], GT.astype(bool), DEFAULT_NS)              # what LENS.evaluate reports as recall_bounds
    lo, hi = out["hits_lo"].cpu().numpy() / nv, out["hits_hi"].cpu().numpy() / nv
    assert np.allclose(lo, det["lo"], rtol=0, atol=1e-12) and np.allclose(hi, det["hi"], rtol=0, atol=1e-12)
    gpu_r1 = float(out["hits"][0].item()) / nv
    assert round(gpu_r1, 2) == 0.62 and lo[0] <= gpu_r1 <= hi[0]
    assert lo[0] - 0.005 <= float(g["R"][0]) <= hi[0] + 0.005 and round(float(g["R"][0]), 2) == 0.63
    assert (lo < hi).any()


# --------------------------------------------------------------------------- live sessions
class BoundsFleet(Fleet):
    """Fleet that pushes with bounds=True and sums hits_lo / hits_hi over the pushes."""

    def __init__(self, *args, **kw):
        super().__init__(*args, **kw)
        self.lo = self.hi = 0

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
            gt = self.rng.integers(-1, self.Po + 2, size=(len(ids), Q)).astype(np.int32)
            out = self.sp.push(pooled=win, gt_center=cuda(gt), gt_tol=self.tol, streams=streams, bounds=True)
            assert bool((out["hits_lo"] <= out["hits"]).all() and (out["hits"] <= out["hits_hi"]).all())
            self.hits = self.hits + out["hits"].cpu()
            self.n_valid = self.n_valid + out["n_valid"].cpu()
            self.lo = self.lo + out["hits_lo"].cpu()
            self.hi = self.hi + out["hits_hi"].cpu()
            for i, b in enumerate(ids):
                seg = self.segs[b][-1]
                seg["win"].append(win[i])
                seg["gt"].append(gt[i])
                for k in ("S", "top_val", "top_idx"):
                    seg[{"top_val": "tv", "top_idx": "ti"}.get(k, k)].append(out[k][i])
                self.cursor[b] += Q

    def check_bounds(self):
        """The pushes' summed bounds equal the batch bounds over each stream segment's valid rows."""
        from lens_b200 import ops
        ns = self.sp.ns
        lo, hi, nv = (torch.zeros(n, dtype=torch.int64, device="cuda") for n in (len(ns), len(ns), 1))
        for b in range(self.B):
            for seg in self.segs[b]:
                if not seg["win"] or sum(s.shape[0] for s in seg["S"]) < self.L:
                    continue
                S = torch.cat(seg["S"])[None].contiguous()
                gt = cuda(np.concatenate(seg["gt"])[None, self.L - 1:])
                ops.seq_recall_bounds(S, self.L, gt_center=gt, gt_tol=self.tol, ns=ns, lo=lo, hi=hi, n_valid=nv)
        assert torch.equal(self.lo, lo.cpu()) and torch.equal(self.hi, hi.cpu()), (self.lo, lo, self.hi, hi)
        assert torch.equal(self.n_valid, nv.cpu()), (self.n_valid, nv)


@gpu
@pytest.mark.parametrize("L", [1, 2, 10])
def test_lockstep_chunkings_equal_batch_bounds(L):
    B, P, Q_tot = 3, 150, 30
    W = model(P)
    cuts = chunkings(L, Q_tot, seed=L)
    cuts["threes"] = [3] * (Q_tot // 3)
    for name in ("ones", "threes", "one_chunk", "mixed", "random"):
        chunks = cuts[name]
        f = BoundsFleet(stream_pipe(W, L, 25, B, MODE_SIMT), B, P, L, seed=L + 3)
        f.run([(None, c) for c in chunks])
        assert not f.sp._indexed
        f.check_bounds()
        f.check_against_batch(W, 25, MODE_SIMT)


@gpu
@pytest.mark.parametrize("L", [1, 2, 10])
def test_random_subset_schedules_with_resets_equal_batch_bounds(L):
    P = 130
    W = model(P)
    for seed in (1, 2):
        rng = np.random.default_rng(L * 10 + seed)
        B = int(rng.integers(4, 7))
        f = BoundsFleet(stream_pipe(W, L, 25, B, MODE_SIMT), B, P, L, seed=seed, tol=int(rng.integers(0, 4)))
        f.run(schedule(rng, B, n_push=12, reset_at=6))
        assert f.sp._indexed
        f.check_bounds()


@gpu
def test_segmented_push_of_one_camera():
    L, P, B = 10, 20000, 2
    W = model(P, seed=5)
    f = BoundsFleet(stream_pipe(W, L, 25, B, MODE_AUTO), B, P, L, seed=9)
    f.run([(None, 3)] + [([1], 1)] * (L + 1) + [([0, 1], 2)])
    f.check_bounds()


@gpu
def test_empty_push_returns_zeros_and_launches_nothing():
    from lens_b200._lib import launch_count
    L, P, B = 3, 100, 3
    sp = stream_pipe(model(P), L, 25, B, MODE_SIMT)
    n0 = launch_count()
    out = sp.push(streams=[], gt_center=torch.zeros((0, 2), dtype=torch.int32, device="cuda"), bounds=True)
    assert launch_count() == n0
    assert out["hits_lo"].tolist() == [0] * len(sp.ns) and out["hits_hi"].tolist() == [0] * len(sp.ns)


# --------------------------------------------------------------------------- structure
@gpu
def test_bounds_false_changes_nothing():
    from lens_b200._lib import launch_count
    L, B, Q, P = 3, 4, 8, 200
    W = model(P)
    pipe = batch_pipe(W, L, 25, B, MODE_SIMT)
    pooled = cuda(np.random.default_rng(1).integers(0, 4, size=(B, Q, 100)).astype(np.uint8))
    c = cuda(np.random.default_rng(2).integers(-1, P - L + 1, size=(B, Q - L + 1)).astype(np.int32))
    runs = {}
    for key, kw in (("none", {}), ("false", dict(bounds=False)), ("true", dict(bounds=True))):
        pipe.net.reset_states()
        n0 = launch_count()
        out, names = kernels_run(lambda: pipe.step(pooled=pooled, gt_center=c, gt_tol=1, **kw))
        runs[key] = (out, names, launch_count() - n0)
    (a, na, la), (b, nb, lb), (t, nt, lt) = runs["none"], runs["false"], runs["true"]
    assert list(a) == list(b) and na == nb and la == lb
    assert all(torch.equal(a[k], b[k]) for k in a if torch.is_tensor(a[k]))
    assert set(t) - set(a) == {"hits_lo", "hits_hi"} and lt == la + 3
    assert not any("rbounds" in n for n in na) and any("rbounds_count_kernel" in n for n in nt)
    # pushes: lockstep and indexed
    for streams in (None, [2, 0]):
        outs = {}
        for key, kw in (("none", {}), ("false", dict(bounds=False))):
            sp = stream_pipe(W, L, 25, B, MODE_SIMT)
            n = B if streams is None else len(streams)
            win = pooled[:n, :2].contiguous()
            sp.push(pooled=win, gt_center=c[:n, :2].contiguous(), streams=streams)
            n0 = launch_count()
            out, names = kernels_run(lambda: sp.push(pooled=win, gt_center=c[:n, :2].contiguous(), streams=streams, **kw))
            outs[key] = (out, names, launch_count() - n0)
        (a, na, la), (b, nb, lb) = outs["none"], outs["false"]
        assert list(a) == list(b) and na == nb and la == lb
        assert all(torch.equal(a[k], b[k]) for k in a if torch.is_tensor(a[k]))


@gpu
def test_launch_count_does_not_depend_on_the_fleet_size():
    from lens_b200 import ops
    from lens_b200._lib import launch_count
    L, Q, P = 3, 4, 90
    counts = []
    for B in (2, 512):
        S = cuda(spike_counts("poisson", B, Q, P, seed=B))
        c = cuda(np.random.default_rng(B).integers(-1, P - L + 1, size=(B, Q)).astype(np.int32))
        ring = torch.zeros((B, L - 1, P), dtype=torch.float32, device="cuda")
        seen = torch.full((B,), L - 1, dtype=torch.int32, device="cuda")
        rows = torch.full((B,), 7, dtype=torch.int64, device="cuda")
        ids = torch.arange(B, dtype=torch.int32, device="cuda").flip(0).contiguous()
        n = []
        for call in (lambda: ops.seq_recall_bounds(S, L, gt_center=c[:, :Q - L + 1].contiguous()),
                     lambda: ops.seq_recall_bounds_stream(S, L, ring, seen, 7, c),
                     lambda: ops.seq_recall_bounds_stream_ids(S, L, ids, ring, seen, rows, c)):
            n0 = launch_count()
            call()
            n.append(launch_count() - n0)
        counts.append(n)
    assert counts[0] == counts[1] == [3, 3, 3], counts


@gpu
def test_two_ranks_equal_one_rank():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
           "--master-addr", "127.0.0.1", "--master-port", str(_free_port()),
           os.path.join(ROOT, "tests", "recall_bounds_dist_check.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-2000:]
    assert "OK" in res.stdout, res.stdout[-2000:]
