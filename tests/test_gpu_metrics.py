"""The evaluation kernels of csrc/match.cu against the oracle, at the shapes and values where they can go wrong.

createPR (lens_pr_counts / lens_pr_counts_multi), the Recall@N counters (lens_recall), their tie-aware bounds
(lens_recall_bounds), the batch top-N paths (warp kernel, segmented warp kernel + topn_merge_kernel, CTA kernel),
the SAD baseline (lens_sad_matrix / lens_reciprocal) and the online matcher (lens_online_match).  Every comparison
is exact: integer counters equal, lists equal with NaN == NaN, indices included."""
import re

import numpy as np
import pytest
import torch

from oracle import oracle as O

gpu = pytest.mark.gpu
f32 = np.float32


def cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def kernels_run(fn):
    """(fn(), whitespace-free names of the CUDA kernels it launched), from torch.profiler."""
    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    names = {"".join(e.name.split()) for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}
    names = {n for n in names if "kernel" in n}
    assert names, "torch.profiler recorded no CUDA kernel: cannot tell which kernels ran"
    return out, names


def ran(names, kernel):
    """kernel: name as the profiler prints it after `lens::`, template arguments included."""
    return any(re.search("::" + re.escape(kernel) + "[(<]", n) for n in names)


# --------------------------------------------------------------------------- A. createPR
def linspace32(start, stop, n):
    """np.linspace(start, stop, n) for two float32 scalars, as numpy >= 2.0 evaluates it: float32 throughout,
    every operation rounded on its own, the denormal branch when the step underflows, the last element = stop."""
    start, stop, div = f32(start), f32(stop), f32(n - 1)
    delta = f32(stop - start)
    step = f32(delta / div)
    i = np.arange(n, dtype=f32)
    y = (i / div) * delta + start if step == 0 else i * step + start
    y[-1] = stop
    return y


def test_linspace32_restates_numpy():
    """The float32 threshold recipe the createPR kernels implement is numpy's, bit for bit (no GPU needed)."""
    rng = np.random.default_rng(0)
    cases = [(1.0, 0.0), (10.0, 0.0), (2.5, 2.5), (0.0, 0.0), (1e-45, 0.0), (3e-45, -1e-45), (1e-38, 0.0),
             (1.7e38, -1.7e38), (-0.1, -7.3), (5.0, 1e-45)]
    cases += [tuple(sorted(rng.standard_normal(2) * 10.0 ** rng.integers(-40, 38), reverse=True)) for _ in range(40)]
    cases += [(float(k) / 10, 0.0) for k in range(1, 30)]
    for start, stop in cases:
        for n in (2, 3, 7, 100, 101, 65535):
            want = np.linspace(f32(start), f32(stop), n)
            assert want.dtype == np.float32
            got = linspace32(start, stop, n)
            assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), (start, stop, n)


def test_createPR_rejects_unsupported_dtypes():
    from lens_b200.src.metrics import createPR
    GT = np.eye(4, dtype=bool)
    for dt in (np.float16, np.longdouble, np.complex64):
        with pytest.raises(ValueError, match="dtype"):
            createPR(np.ones((4, 4), dtype=dt), GT, None)


def check_pr(S, GT, n_thresh, matching, GTsoft=None):
    from lens_b200.src.metrics import createPR
    P, R = createPR(S, GT, None, GTsoft=GTsoft, matching=matching, n_thresh=n_thresh)
    Pw, Rw = O.create_pr(S, GT, n_thresh=n_thresh, matching=matching, GTsoft=GTsoft)
    assert len(P) == len(R) == n_thresh + 1
    assert np.array_equal(np.array(P, np.float64), np.array(Pw, np.float64), equal_nan=True), (matching, n_thresh)
    assert np.array_equal(np.array(R, np.float64), np.array(Rw, np.float64), equal_nan=True), (matching, n_thresh)


def random_gt(rng, Po, Qo, density=0.3, empty_cols=0.1):
    GT = rng.random((Po, Qo)) < density
    GT[:, rng.random(Qo) < empty_cols] = False          # queries without a positive
    return GT


@gpu
def test_createPR_tenths_reproducer():
    """S = k/10 for k = 0..100 (the values D takes at L = 10): float64 thresholds select differently at 38 of the
    101 thresholds, the float32 ones numpy uses are the reference's."""
    S = (np.arange(101, dtype=f32) / f32(10))[None]
    GT = (np.arange(101) % 3 == 0)[None]
    t32, t64 = np.linspace(S.max(), S.min(), 101), np.linspace(float(S.max()), float(S.min()), 101)
    assert t32.dtype == np.float32
    assert sum((S[0] >= a).sum() != (S[0].astype(np.float64) >= b).sum() for a, b in zip(t32, t64)) > 0
    for matching in ("single", "multi"):
        check_pr(S, GT, 101, matching)
        check_pr(S.T.copy(), GT.T.copy(), 101, matching)


@gpu
@pytest.mark.parametrize("matching", ["single", "multi"])
@pytest.mark.parametrize("L", [1, 2, 3, 7, 10])
def test_createPR_grids(L, matching):
    """k / L grids (the values of a sequence-matched spike-count matrix), negative ones too."""
    rng = np.random.default_rng(L)
    for Po, Qo, lo, hi in ((5, 400, 0, 10 * L), (2, 301, 0, 3 * L), (7, 300, -10 * L, 2 * L)):
        S = rng.integers(lo, hi + 1, size=(Po, Qo)).astype(f32) / f32(L)
        GT = random_gt(rng, Po, Qo)
        for n in (2, 3, 100, 101):
            check_pr(S, GT, n, matching)


@gpu
@pytest.mark.parametrize("matching", ["single", "multi"])
def test_createPR_poisson(matching):
    """Poisson(1.3 L) / L matrices, 150 x 150, the reference's default n_thresh, with and without GTsoft."""
    for L in (3, 5, 7, 10):
        for seed in range(8):
            rng = np.random.default_rng(100 * L + seed)
            S = rng.poisson(1.3 * L, size=(150, 150)).astype(f32) / f32(L)
            GT = random_gt(rng, 150, 150, density=0.02)
            check_pr(S, GT, 100, matching)
            if seed < 2:
                check_pr(S, GT, 100, matching, GTsoft=GT | np.roll(GT, 1, axis=0) | np.roll(GT, -2, axis=0))


@gpu
@pytest.mark.parametrize("matching", ["single", "multi"])
def test_createPR_constant_and_denormal(matching):
    """A constant matrix (max == min: step 0) and the values {0, 1e-45}, whose float32 step underflows to 0 and
    takes numpy's denormal branch (y_i = i / (n - 1) * delta + start)."""
    rng = np.random.default_rng(5)
    const = np.full((6, 50), 2.5, f32)
    den = np.where(rng.random((8, 64)) < 0.5, f32(0), f32(1e-45)).astype(f32)
    den[:, :10] = 0
    # the branch matters: without it every threshold but the last would be 1e-45
    assert (np.linspace(den.max(), den.min(), 101)[:-1] == 0).any()
    for S in (const, den, -den):
        GT = random_gt(rng, *S.shape)
        for n in (2, 3, 100, 101):
            check_pr(S, GT, n, matching)


@gpu
def test_createPR_single_first_maximum():
    """matching='single' takes the FIRST row of a tied column maximum (np.argmax): columns where a positive and a
    negative row share the maximum, in both orders."""
    rng = np.random.default_rng(6)
    S = rng.integers(0, 3, size=(6, 500)).astype(f32)
    GT = rng.random((6, 500)) < 0.5
    top = S == S.max(0)
    mixed = (top & GT).any(0) & (top & ~GT).any(0)
    assert mixed.sum() > 100
    for n in (2, 3, 100, 101):
        check_pr(S, GT, n, "single")


@gpu
def test_createPR_single_query_count_limits():
    """One query, and Qo = 8192 (all of the kernel's shared memory)."""
    rng = np.random.default_rng(7)
    for Po, Qo in ((50, 1), (3, 8192)):
        S = rng.integers(0, 41, size=(Po, Qo)).astype(f32) / f32(7)
        GT = random_gt(rng, Po, Qo)
        if Qo == 1:
            GT[rng.integers(Po), 0] = True
        for n in (2, 3, 100, 101):
            check_pr(S, GT, n, "single")


@gpu
def test_createPR_multi_slices():
    """'multi' with the count kernel on 1 slice (65 535 thresholds) and on 64 slices over an element count that is
    not a multiple of 64, large enough that the min/max kernel strides over the grid."""
    rng = np.random.default_rng(8)
    S = rng.integers(0, 30, size=(37, 53)).astype(f32) / f32(10)
    GT = random_gt(rng, 37, 53)
    check_pr(S, GT, 65535, "multi")
    Po, Qo = 2053, 2029
    n = Po * Qo
    assert n > 63 * 65536 and n % 64 != 0 and n > 148 * 8 * 256
    S = rng.poisson(1.3 * 7, size=(Po, Qo)).astype(f32) / f32(7)
    GT = random_gt(rng, Po, Qo, density=0.01)
    check_pr(S, GT, 100, "multi")


@gpu
@pytest.mark.parametrize("matching", ["single", "multi"])
def test_createPR_float64_and_integer_input(matching):
    """float64, integer and bool matrices take numpy's float64 thresholds (values representable in float32)."""
    rng = np.random.default_rng(9)
    K = rng.integers(-20, 60, size=(40, 90))
    GT = random_gt(rng, 40, 90)
    for S in (K.astype(np.float64) / 4, K.astype(np.float64), K, K.astype(np.int32), (K % 50).astype(np.uint8),
              K > 10):
        for n in (2, 3, 100, 101):
            check_pr(S, GT, n, matching)


# --------------------------------------------------------------------------- B. lens_recall
def recall_loop(ti, Po, ns, gt_dense=None, gt_center=None, tol=0):
    """metrics.py:213-224 over given top-N lists: hits[i] = queries with a positive among their first ns[i]
    entries (-1 = empty slot), n_valid = queries with any positive."""
    B, Qo, N = ti.shape
    hits, nv = np.zeros(len(ns), np.int64), 0
    for b in range(B):
        for q in range(Qo):
            if gt_dense is not None:
                g = gt_dense[b] if gt_dense.ndim == 3 else gt_dense
                valid = bool(g[:, q].any())
                pos = [r >= 0 and bool(g[r, q]) for r in ti[b, q]]
            else:
                c = int(gt_center[b, q])
                valid = c >= 0
                pos = [r >= 0 and abs(int(r) - c) <= tol for r in ti[b, q]]
            if not valid:
                continue
            nv += 1
            first = pos.index(True) if True in pos else N
            for i, k in enumerate(ns):
                hits[i] += first < k
    return hits, nv


def random_lists(rng, B, Qo, N, Po):
    ti = rng.integers(0, Po, size=(B, Qo, N)).astype(np.int32)
    ti[rng.random((B, Qo, N)) < 0.2] = -1                     # empty slots anywhere
    ti[:, ::7, N // 2:] = -1                                   # and empty tails (N > Po)
    return ti


NS8 = (1, 2, 5, 10, 25, 32, 63, 64)


@gpu
def test_recall_dense_gt():
    """Shared 2-D and per-stream 3-D ground truth, ns of length 8 up to N = 64 and of length 1, B * Qo = 300."""
    from lens_b200 import ops
    rng = np.random.default_rng(10)
    B, Qo, Po, N = 3, 100, 200, 64
    ti = random_lists(rng, B, Qo, N, Po)
    gt3 = rng.random((B, Po, Qo)) < 0.01
    gt3[:, :, :9] = False
    for gt in (gt3[1], gt3):
        for ns in (NS8, (7,), (64,)):
            want_h, want_n = recall_loop(ti, Po, ns, gt_dense=gt)
            assert 0 < want_n < B * Qo and 0 < want_h[-1]
            h, n = ops.recall_counts(cuda(ti), Po, gt_dense=cuda(gt.astype(np.uint8)), ns=ns)
            assert h.tolist() == want_h.tolist() and int(n.item()) == want_n, (gt.ndim, ns)


@gpu
@pytest.mark.parametrize("tol", [0, 3])
def test_recall_band_gt(tol):
    """Band ground truth through gt_center: -1 (no match), centres at 0 and Po - 1, hits planted near the centre."""
    from lens_b200 import ops
    rng = np.random.default_rng(11 + tol)
    B, Qo, Po, N = 3, 100, 200, 64
    ti = random_lists(rng, B, Qo, N, Po)
    c = rng.integers(0, Po, size=(B, Qo)).astype(np.int32)
    c[:, ::5], c[:, 1::5], c[:, 2::9] = 0, Po - 1, -1
    for b in range(B):
        for q in range(Qo):
            if rng.random() < 0.7:
                ti[b, q, rng.integers(N)] = np.clip(c[b, q] + rng.integers(-4, 5), 0, Po - 1)
    for ns in (NS8, (10,)):
        want_h, want_n = recall_loop(ti, Po, ns, gt_center=c, tol=tol)
        h, n = ops.recall_counts(cuda(ti), Po, gt_center=cuda(c), gt_tol=tol, ns=ns)
        assert h.tolist() == want_h.tolist() and int(n.item()) == want_n, ns


@gpu
def test_recall_counters_accumulate():
    """hits / n_valid are accumulated over calls, as the header promises."""
    from lens_b200 import ops
    rng = np.random.default_rng(12)
    B, Qo, Po, N = 2, 77, 50, 25
    gt = rng.random((Po, Qo)) < 0.05
    ti1, ti2 = random_lists(rng, B, Qo, N, Po), random_lists(rng, B, Qo, N, Po)
    ns = (1, 5, 10, 15, 20, 25)
    h, n = ops.recall_counts(cuda(ti1), Po, gt_dense=cuda(gt.astype(np.uint8)), ns=ns)
    h, n = ops.recall_counts(cuda(ti2), Po, gt_dense=cuda(gt.astype(np.uint8)), ns=ns, hits=h, n_valid=n)
    (h1, n1), (h2, n2) = recall_loop(ti1, Po, ns, gt_dense=gt), recall_loop(ti2, Po, ns, gt_dense=gt)
    assert h.tolist() == (h1 + h2).tolist() and int(n.item()) == n1 + n2


@gpu
def test_recall_end_to_end_equals_stable_argsort():
    """seqmatch_topk(L = 1) then recall_counts == O.recall_at_k(kind='stable') on a tie-heavy matrix."""
    from lens_b200 import ops
    rng = np.random.default_rng(13)
    Po, Qo = 300, 211
    D = rng.integers(0, 6, size=(Po, Qo)).astype(f32)
    GT = rng.random((Po, Qo)) < 0.02
    ns = (1, 5, 10, 15, 20, 25)
    _, ti, _ = ops.seqmatch_topk(cuda(D.T)[None], 1, 25)
    h, n = ops.recall_counts(ti, Po, gt_dense=cuda(GT.astype(np.uint8)), ns=ns)
    n = int(n.item())
    assert n == GT.any(0).sum()
    for i, K in enumerate(ns):
        assert int(h[i]) / n == O.recall_at_k(D, GT, K=K, kind="stable"), K


# --------------------------------------------------------------------------- C. lens_recall_bounds
def tie_matrix(rng, Po, Qo):
    """Tie-heavy columns (small integer sets of per-column width), some -inf entries, a column without any
    positive and a column where every entry is positive; every other column gets at least one positive."""
    width = rng.integers(1, 12, size=Qo)
    D = (rng.random((Po, Qo)) * width).astype(np.int64).astype(f32)
    D[rng.random((Po, Qo)) < 0.05] = -np.inf
    GT = rng.random((Po, Qo)) < rng.random(Qo) * 0.5
    GT[rng.integers(Po, size=Qo), np.arange(Qo)] = True
    if Qo >= 3:
        GT[:, 0] = False
        GT[:, 1] = True
    return D, GT


def bounds_ns(Po):
    """Ascending K, several inside one tie group, K = Po and K > Po (the column runs out)."""
    ks = sorted({1, 2, 3, 5, max(Po - 1, 1), Po, Po + 1, Po + 7})
    return tuple(ks[-8:])


@gpu
@pytest.mark.parametrize("Qo", [1, 7, 9, 1000])
@pytest.mark.parametrize("Po", [1, 31, 32, 33, 1000])
def test_recall_bounds(Po, Qo):
    from lens_b200 import ops
    rng = np.random.default_rng(Po * 7919 + Qo)
    D, GT = tie_matrix(rng, Po, Qo)
    ns = bounds_ns(Po)
    lo, hi, nv = ops.recall_bounds(cuda(D), cuda(GT.astype(np.uint8)), ns)
    lo, hi, nv = lo.tolist(), hi.tolist(), int(nv.item())
    keep = GT.any(0)
    assert nv == keep.sum() > 0
    for i, K in enumerate(ns):
        wl, wh = O.recall_bounds(D, GT, K)
        assert (lo[i], hi[i]) == (round(wl * nv), round(wh * nv)), K
    if Po > 1 and Qo > 1:
        assert any(a != b for a, b in zip(lo, hi))                # the ties do decide something here
    # any order numpy's default argsort gives the ties lies between the bounds
    for _ in range(20 if Po * Qo <= 100_000 else 3):
        perm = rng.permutation(Po)
        Dp, Gp = D[perm][:, keep], GT[perm][:, keep]
        order = Dp.argsort(0)
        for i, K in enumerate(ns):
            hit = int(np.take_along_axis(Gp, order[-K:], axis=0).any(0).sum())
            assert lo[i] <= hit <= hi[i], K
    # recallAtK: the reference's value, from the kernels where the bounds meet and numpy's tie order elsewhere
    from lens_b200.src.metrics import recallAtK
    for K in [k for k in ns if k <= 64][:4]:
        assert recallAtK(D, GT, K=K) == O.recall_at_k(D, GT, K=K), K


# --------------------------------------------------------------------------- D. batch top-N
def check_topn(S, L, N, want_D=False):
    """ops.seqmatch_topk on S [B, Q, P] == O.seqmatch + O.topk per stream: values, indices, empty slots, D.
    Returns the kernel names the call launched."""
    from lens_b200 import ops
    (tv, ti, D), names = kernels_run(lambda: ops.seqmatch_topk(cuda(S), L, N, want_D=want_D))
    tv, ti = tv.cpu().numpy(), ti.cpu().numpy()
    for b in range(S.shape[0]):
        Do = O.seqmatch(S[b], L)
        io, vo = O.topk(Do, N)
        assert np.array_equal(ti[b], io), b
        assert np.array_equal(tv[b], vo), b
        Po = Do.shape[0]
        if Po < N:
            assert (ti[b][:, Po:] == -1).all() and np.isneginf(tv[b][:, Po:]).all()
        if want_D:
            assert np.array_equal(D[b].cpu().numpy(), Do), b
    return names


@gpu
@pytest.mark.parametrize("S_kind", ["constant", "poisson"])
@pytest.mark.parametrize("P,N,L", [(20000, 1, 10), (20000, 16, 1), (20000, 25, 10), (20000, 32, 10),
                                   (70000, 32, 10), (70000, 32, 1)])
def test_topn_segmented(P, N, L, S_kind):
    """Few queries against many places: the places are split into segments (70 000 places at N = 32: as many as
    512 / N lists fit the merge) and topn_merge_kernel merges them.  A constant S ties everything, so the answer is
    the N largest indices, all in the last, partial segment; Poisson(0.3) gives tie plateaus across segments."""
    B, Q = 1, L + 2
    S = np.ones((B, Q, P), f32) if S_kind == "constant" else \
        np.random.default_rng(P + N + L).poisson(0.3, size=(B, Q, P)).astype(f32)
    names = check_topn(S, L, N, want_D=(N != 16))
    assert ran(names, "seqmatch_topk_warp_kernel<true>") and ran(names, "topn_merge_kernel"), names
    assert not ran(names, "seqmatch_topk_warp_kernel<false>"), names


@gpu
@pytest.mark.parametrize("N", [33, 64])
def test_topn_cta_kernel(N):
    """32 < N <= 64: fewer places than N (the tail is -inf / -1), and a plateau of ties across the 2048-place
    chunk boundary of the CTA kernel."""
    rng = np.random.default_rng(N)
    L = 10
    small = rng.poisson(1.3, size=(2, L + 3, L - 1 + 31)).astype(f32)            # Po = 31 < N
    names = check_topn(small, L, N, want_D=True)
    assert ran(names, "seqmatch_topk_kernel"), names
    L = 4
    S = np.minimum(rng.poisson(0.3, size=(2, L + 2, 5000)), 3).astype(f32)
    S[:, :, 2000:2110] = 5                                                       # D = 5 for r in [2000, 2107)
    names = check_topn(S, L, N)
    assert ran(names, "seqmatch_topk_kernel"), names
    check_topn(np.ones((1, L + 1, 4500), f32), L, N)


@gpu
def test_topn_warp_kernel():
    """N = 32 on the one-warp-per-query kernel, Po = 998 (not a multiple of the 128 places a warp loads at once)."""
    S = np.random.default_rng(14).poisson(1.3, size=(4, 12, 1000)).astype(f32)
    for N in (32, 7):
        names = check_topn(S, 3, N, want_D=True)
        assert ran(names, "seqmatch_topk_warp_kernel<false>") and not ran(names, "topn_merge_kernel"), names


# --------------------------------------------------------------------------- E. SAD
def sad_both_paths(a, b):
    """lens_sad_matrix on aligned copies (16-byte loads when npix % 16 == 0) and on contiguous views offset by
    one byte (the byte-wise path)."""
    from lens_b200 import ops
    out = [ops.sad_matrix(cuda(a), cuda(b))]
    views = []
    for x in (a, b):
        buf = torch.empty(x.size + 1, dtype=torch.uint8, device="cuda")
        buf[1:] = cuda(x.ravel())
        v = buf[1:].view(x.shape)
        assert v.is_contiguous() and v.data_ptr() % 16 != 0
        views.append(v)
    out.append(ops.sad_matrix(*views))
    return [o.cpu().numpy() for o in out]


@gpu
@pytest.mark.parametrize("npix", [1, 15, 16, 17, 6400, 65792, 65793])
def test_sad_matrix(npix):
    rng = np.random.default_rng(npix)
    a = rng.integers(0, 256, size=(5, npix), dtype=np.uint8)
    b = rng.integers(0, 256, size=(7, npix), dtype=np.uint8)
    a[0], b[0] = 0, 255                                                    # the largest sum: npix * 255
    want = np.abs(a[:, None, :].astype(np.int64) - b[None, :, :].astype(np.int64)).sum(-1)
    assert want[0, 0] == npix * 255
    if npix == 65793:
        assert want[0, 0] == 2 ** 24 - 1
    for got in sad_both_paths(a, b):
        assert got.dtype == np.float32 and np.array_equal(got, want.astype(f32))


@gpu
def test_reciprocal():
    from lens_b200 import ops
    rng = np.random.default_rng(15)
    x = np.concatenate([np.array([0.0, -0.0, 1.0, 3.0, 7.0, -2.5, 1e-45, 1e-38, 3e38, -3e38, np.inf, -np.inf], f32),
                        rng.integers(0, 2 ** 24, size=1000).astype(f32),
                        (rng.standard_normal(333) * 10.0 ** rng.integers(-40, 38, size=333)).astype(f32)])
    with np.errstate(divide="ignore", over="ignore"):
        want = f32(1) / x
    got = ops.reciprocal(cuda(x)).cpu().numpy()
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))


# --------------------------------------------------------------------------- F. lens_online_match
def online_match_gpu(seq, L):
    """lens_online_match through the C ABI: seq i32 [R, P] -> (result f64 [P, R], argmax i32 [R])."""
    from lens_b200._lib import lib, check, ptr, stream_ptr
    R, P = seq.shape
    d = cuda(seq.astype(np.int32))
    res = torch.empty((P, R), dtype=torch.float64, device="cuda")
    am = torch.empty((R,), dtype=torch.int32, device="cuda")
    check(lib().lens_online_match(ptr(d), R, P, L, ptr(res), ptr(am), stream_ptr()), "lens_online_match")
    return res.cpu().numpy(), am.cpu().numpy()


@gpu
@pytest.mark.parametrize("R,P,L", [(4, 300, 2), (4, 300, 3), (4, 37, 9), (6, 5, 9), (64, 300, 4), (64, 40, 7),
                                   (3, 20, 64)])
def test_online_match(R, P, L):
    """Even and odd L, L > R, L > P, R = 64; small counts so that column maxima tie across threads."""
    seq = np.random.default_rng(R * P + L).integers(0, 4, size=(R, P))
    res, am = online_match_gpu(seq, L)
    want_res, want_am = O.online_match(seq, L)
    assert np.array_equal(res, want_res)
    assert np.array_equal(am, want_am)


@gpu
def test_online_match_first_maximum_across_threads():
    """Two equal maxima per column, 295 places apart (owned by different threads): the first one wins."""
    R, P, L = 8, 1000, 3
    seq = np.zeros((R, P), np.int64)
    rr = np.arange(R)
    seq[rr, rr + 1] = 9                  # diagonal lines: column r peaks at p = r + 1 and p = r + 296
    seq[rr, rr + 296] = 9
    res, am = online_match_gpu(seq, L)
    want_res, want_am = O.online_match(seq, L)
    assert res[5, 4] == res[300, 4] == res[:, 4].max()
    assert np.array_equal(want_am, rr + 1)
    assert np.array_equal(res, want_res) and np.array_equal(am, want_am)
