"""Recall@K with the reference's call signature (lens/src/metrics.py:183-226), on the GPU.

`recallAtK(S_in, GThard, GTsoft=None, K=1)` takes numpy matrices [database, query] and returns a
float.  The K best rows of every query column are selected by the CUDA top-N kernel
(lens_seqmatch_topk with L = 1) under the deterministic rule "larger value first, larger
database index first among equals" (the order `np.argsort(kind='stable')[-K:]` yields), and
lens_recall_bounds counts, over EVERY order equal similarities can take, the queries that hit for
sure and those that can hit.  When the two bounds coincide the ties cannot change the answer and
the kernel's value is the reference's.  When they differ, the reference's own number is whatever
numpy's default (unstable) argsort happens to do with the ties (metrics.py:218): only in that case
the tie order is taken from the same numpy call on the host copy of the matrix, so that the value
returned is the one the reference returns in this environment (DESIGN.md, H5).
"""
import numpy as np
import torch

from .. import ops

MAX_K = 64


def _topk_hits(S, GT, K):
    """hits / valid for one K through the CUDA kernels.  S, GT: [Po, Qo] numpy."""
    Po, Qo = S.shape
    # the kernel consumes query-major similarity rows: S_in[r][q] = S_t[q][r]
    S_t = torch.from_numpy(np.ascontiguousarray(S.T, dtype=np.float32)).cuda()[None]
    _, ti, _ = ops.seqmatch_topk(S_t, 1, K)
    gt = torch.from_numpy(np.ascontiguousarray(GT, dtype=np.uint8)).cuda()
    hits, nv = ops.recall_counts(ti, Po, gt_dense=gt, ns=(K,))
    return int(hits[0].item()), int(nv.item())


def numpy_tie_order_recall(S, GT, K):
    """Recall@K with the ties ordered by numpy's default argsort, the call the reference makes
    (metrics.py:218: take the last K rows of the ascending argsort of every query column that has a
    positive).  Host-side tie arbitration only; S, GT numpy [database, query]."""
    keep = GT.any(axis=0)
    if not keep.any():
        return float("nan")
    S, GT = S[:, keep], GT[:, keep]
    top = np.argsort(S, axis=0)[-K:, :]
    return float(np.take_along_axis(GT, top, axis=0).any(axis=0).mean())


def recall_detail(S, GT, Ks, top_idx=None, S_dev=None):
    """Recall for every K in Ks (ascending) -> dict(gpu, lo, hi, reference, n_valid, ties_decided).

    gpu: deterministic tie rule of the CUDA top-N kernel; lo / hi: tie-aware bounds (lens_recall_bounds);
    reference: the reference's value -- gpu where lo == hi, numpy's tie order otherwise.
    S, GT numpy [Po, Qo]; top_idx (device i32 [1, Qo, >= max K]) and S_dev (device f32 [Po, Qo]) may be
    passed when the caller already holds them."""
    Po, Qo = S.shape
    Ks = tuple(int(k) for k in Ks)
    if S_dev is None:
        S_dev = torch.from_numpy(np.ascontiguousarray(S, dtype=np.float32)).cuda()
    if top_idx is None:
        _, top_idx, _ = ops.seqmatch_topk(S_dev.t().contiguous()[None], 1, max(Ks))
    gt = torch.from_numpy(np.ascontiguousarray(GT, dtype=np.uint8)).to(S_dev.device)
    hits, nv = ops.recall_counts(top_idx, Po, gt_dense=gt, ns=Ks)
    lo, hi, nv2 = ops.recall_bounds(S_dev, gt, ns=Ks)
    hits, lo, hi, nv, nv2 = hits.cpu().numpy(), lo.cpu().numpy(), hi.cpu().numpy(), int(nv.item()), int(nv2.item())
    assert nv == nv2
    nan = float("nan")
    out = dict(gpu=[h / nv if nv else nan for h in hits], lo=[x / nv if nv else nan for x in lo],
               hi=[x / nv if nv else nan for x in hi], n_valid=nv, reference=[], ties_decided=[])
    for i, K in enumerate(Ks):
        if not nv or lo[i] == hi[i]:
            out["reference"].append(out["gpu"][i])
        else:
            out["reference"].append(numpy_tie_order_recall(S, GT.astype(bool), K))
            out["ties_decided"].append(K)
    return out


def recallAtK(S_in, GThard, GTsoft=None, K=1):
    S_in, GThard = np.asarray(S_in), np.asarray(GThard)
    assert S_in.shape == GThard.shape, "S_in and GThard must have the same shape"
    assert S_in.ndim == 2, "S_in, GThard and GTsoft must be two-dimensional"
    assert K >= 1, "K must be >=1"
    if K > MAX_K:
        raise ValueError(f"K={K} exceeds the supported maximum {MAX_K}")
    GT = GThard.astype(bool)
    S = S_in.copy()
    if GTsoft is not None:
        soft = np.asarray(GTsoft).astype(bool)
        assert S_in.shape == soft.shape, "S_in and GTsoft must have the same shape"
        S[soft & ~GT] = S.min()
    return recall_detail(S, GT, (K,))["reference"][0]


def createPR(S_in, GThard, outputdir=None, datatype="LENS", GTsoft=None, matching="multi", n_thresh=100):
    """Precision / recall lists of lens/src/metrics.py:21-139: matching='single' (best match per query, the mode
    the reference's inference path uses, lens/run_model.py:321) or 'multi' (every entry of the matrix, the
    reference's default).  S_in, GThard: numpy [database, query].  Returns (P, R): python lists of length
    n_thresh + 1 starting with P = 1, R = 0.  The figure the reference saves on the last threshold is not produced.

    The thresholds are np.linspace(max, min, n_thresh), which numpy (>= 2.0) evaluates in the matrix's own type:
    float32 arithmetic for a float32 S_in, float64 for float64, integer and bool ones.  The kernels read S_in as
    float32, so a float64 S_in gives the reference's lists only when every value is representable in float32 (the
    spike-count averages and SAD similarities of this package are).  Other dtypes (float16, longdouble, ...) raise
    ValueError."""
    from .._lib import lib, check, ptr, stream_ptr
    S_in, GThard = np.asarray(S_in), np.asarray(GThard)
    assert S_in.shape == GThard.shape, "S_in, GThard and GTsoft must have the same shape"
    assert S_in.ndim == 2, "S_in, GThard and GTsoft must be two-dimensional"
    assert matching in ("single", "multi"), "matching should contain one of the following strings: [single, multi]"
    assert n_thresh > 1, "n_thresh must be >1"
    if S_in.dtype == np.float32:
        thresh_f64 = 0
    elif S_in.dtype == np.float64 or S_in.dtype.kind in "biu":
        thresh_f64 = 1
    else:
        raise ValueError(f"createPR: S_in of dtype {S_in.dtype} is not supported (float32, float64, integer or bool)")
    GT = GThard.astype(bool)
    S = S_in.astype(np.float32, copy=True)
    if GTsoft is not None:
        soft = np.asarray(GTsoft).astype(bool)
        S[soft & ~GT] = S.min()
    Po, Qo = S.shape
    dS = torch.from_numpy(np.ascontiguousarray(S)).cuda()
    dG = torch.from_numpy(np.ascontiguousarray(GT, dtype=np.uint8)).cuda()
    tp = torch.zeros(n_thresh, dtype=torch.int64, device="cuda")
    fp = torch.zeros(n_thresh, dtype=torch.int64, device="cuda")
    gtp = torch.zeros(1, dtype=torch.int64, device="cuda")
    if matching == "single":
        check(lib().lens_pr_counts(ptr(dS), ptr(dG), Po, Qo, n_thresh, ptr(tp), ptr(fp), ptr(gtp), stream_ptr(),
                                   thresh_f64), "lens_pr_counts")
    else:
        check(lib().lens_pr_counts_multi(ptr(dS), ptr(dG), Po, Qo, n_thresh, ptr(tp), ptr(fp), ptr(gtp), stream_ptr(),
                                         thresh_f64), "lens_pr_counts_multi")
    return pr_lists(tp.cpu().numpy(), fp.cpu().numpy(), int(gtp.item()))


def pr_lists(tp, fp, gtp):
    """createPR's (P, R) from the counts at its thresholds (lens/src/metrics.py:21-139): lists of length
    len(tp) + 1 starting with P = 1, R = 0, each entry a float64 division as the reference makes it."""
    P, R = [1], [0]
    with np.errstate(divide="ignore", invalid="ignore"):
        for a, b in zip(tp, fp):
            P.append(np.float64(a) / np.float64(a + b))
            R.append(np.float64(a) / np.float64(gtp))
    return P, R
