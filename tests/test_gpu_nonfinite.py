"""The evaluation kernels of csrc/match.cu on infinite, NaN and signed-zero similarities, against plain numpy.

recallAtK, createPR and run_sad take any matrix a caller passes, and the SAD baseline itself makes +inf (1 / 0 for
a zero distance).  numpy's rule is the reference: np.sort puts every NaN last (one class above +inf, whatever its
sign or payload), -0.0 == +0.0, np.argmax / np.max / np.min return the first NaN / NaN.  Each case first asserts
that it contains what it exists for.  Top-N lists are compared with indices, bounds and PR counts exactly."""
import struct
import zlib

import numpy as np
import pytest
import torch

from oracle import oracle as O
from test_gpu_metrics import kernels_run, ran

gpu = pytest.mark.gpu
f32 = np.float32
FMAX = np.finfo(f32).max
TINY = f32(1e-45)                                              # the smallest subnormal
# numpy's nan, the NaN of x86 inf - inf / 0 * inf, a signalling one and a negative one with another payload
NAN_BITS = (0x7fc00000, 0xffc00000, 0x7f800001, 0xffbfffff)
NANS = np.array(NAN_BITS, np.uint32).view(f32)
SPECIAL = np.array([np.inf, -np.inf, 0.0, -0.0, FMAX, -FMAX, TINY, -TINY], f32)
PALETTE = np.concatenate([NANS, SPECIAL, np.array([1.0, 2.0, -3.5], f32)])


def cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def bits(a):
    return np.ascontiguousarray(a, f32).view(np.uint32)


def neg_zero(a):
    return (a == 0) & np.signbit(a)


def palette_matrix(rng, Po, Qo, palette=PALETTE):
    """[Po, Qo] f32, every column drawn from 2-5 palette values (tie-heavy); column 0 only NaNs of mixed payloads,
    column 1 only +-inf, column 2 only +-0 (when Qo > 3)."""
    D = np.empty((Po, Qo), f32)
    for q in range(Qo):
        vals = rng.choice(palette, size=rng.integers(2, 6), replace=False)
        D[:, q] = vals[rng.integers(0, len(vals), Po)]
    if Qo > 3:
        D[:, 0] = NANS[rng.integers(0, len(NANS), Po)]
        D[:, 1] = np.array([np.inf, -np.inf], f32)[rng.integers(0, 2, Po)]
        D[:, 2] = np.array([0.0, -0.0], f32)[rng.integers(0, 2, Po)]
    return D


def palette_gt(rng, D, density=0.15):
    """Positives at random, at least one per column but the last (a column without a positive is dropped)."""
    Po, Qo = D.shape
    GT = rng.random((Po, Qo)) < density
    GT[rng.integers(0, Po, Qo), np.arange(Qo)] = True
    GT[:, -1] = False
    return GT


def assert_covers(D, GT):
    """The palette case is not vacuous: positives sit on each kind of special value, below a NaN or a +inf and
    above a -inf of the same column."""
    pos = GT
    for name, m in (("NaN", np.isnan(D)), ("+inf", D == np.inf), ("-inf", D == -np.inf), ("-0", neg_zero(D)),
                    ("+0", (D == 0) & ~np.signbit(D)), ("FLT_MAX", np.abs(D) == FMAX),
                    ("subnormal", np.abs(D) == TINY)):
        assert (m & pos).any(), f"no positive on {name}"
    nan = np.isnan(D)
    assert (nan.any(0) & (pos & ~nan).any(0)).any(), "no positive below a NaN"
    assert ((D == np.inf).any(0) & (pos & (D < np.inf)).any(0)).any(), "no positive below a +inf"
    assert ((D == -np.inf).any(0) & (pos & (D != -np.inf)).any(0)).any(), "no positive above a -inf"
    assert (np.isnan(D).all(0)).any() and (np.isinf(D).all(0)).any(), "no all-NaN or all-inf column"


# --------------------------------------------------------------------------- top-N with indices
def stable_topn(D, N):
    """np.argsort(col, kind='stable')[-N:][::-1] of every column of D [Po, Qo] -> idx i32 [Qo, N] (-1 past Po) and
    the values at them (-inf past Po), payloads as they are in D."""
    Po, Qo = D.shape
    n = min(N, Po)
    top = np.argsort(D, axis=0, kind="stable")[::-1][:n]
    idx = np.full((Qo, N), -1, np.int32)
    val = np.full((Qo, N), -np.inf, f32)
    idx[:, :n] = top.T
    val[:, :n] = np.take_along_axis(D, top, 0).T
    return idx, val


def check_seqmatch_topn(S, L, N):
    """ops.seqmatch_topk on S [B, Q, P] == stable_topn of O.seqmatch per stream (D too, NaN == NaN).  Returns the
    kernel names the call launched."""
    from lens_b200 import ops
    (tv, ti, D), names = kernels_run(lambda: ops.seqmatch_topk(cuda(S), L, N, want_D=True))
    tv, ti, D = tv.cpu().numpy(), ti.cpu().numpy(), D.cpu().numpy()
    for b in range(S.shape[0]):
        with np.errstate(invalid="ignore", over="ignore"):
            Do = O.seqmatch(S[b], L)
        assert np.array_equal(D[b], Do, equal_nan=True), b
        idx, val = stable_topn(Do, N)
        assert np.array_equal(ti[b], idx), b
        assert np.array_equal(tv[b], val, equal_nan=True), b
    return names


def topn_input(rng, B, Q, P):
    """Query-major S [B, Q, P] from the palette (column = one query row of S at L = 1)."""
    return np.stack([palette_matrix(rng, P, Q).T for _ in range(B)])


@gpu
@pytest.mark.parametrize("N", [1, 7, 32])
def test_topn_warp_kernel_nonfinite(N):
    rng = np.random.default_rng(N)
    S = topn_input(rng, 2, 40, 300)
    assert np.isnan(S).any() and np.isinf(S).any() and neg_zero(S).any()
    names = check_seqmatch_topn(S, 1, N)
    assert ran(names, "seqmatch_topk_warp_kernel<false>") and not ran(names, "topn_merge_kernel"), names


@gpu
@pytest.mark.parametrize("N", [33, 64])
def test_topn_cta_kernel_nonfinite(N):
    """32 < N <= 64, with Po = 20 < N (the tail is -inf / -1) and Po = 2500 (two chunks of the CTA kernel)."""
    rng = np.random.default_rng(N)
    for P in (20, 2500):
        S = topn_input(rng, 2, 9, P)
        assert np.isnan(S).any() and np.isinf(S).any() and neg_zero(S).any()
        names = check_seqmatch_topn(S, 1, N)
        assert ran(names, "seqmatch_topk_kernel"), names


@gpu
@pytest.mark.parametrize("N", [1, 25])
def test_topn_segmented_nonfinite(N):
    """Few queries against 20 000 places: per-segment lists merged by topn_merge_kernel.  NaNs and +inf sit in
    several segments, so the merge decides among them."""
    rng = np.random.default_rng(100 + N)
    S = topn_input(rng, 1, 5, 20000)
    S[0, 3, ::997] = NANS[1]                          # x86's NaN in every segment of query 3
    S[0, 4, ::1500] = np.inf
    assert np.isnan(S[0, 3, :8192]).any() and np.isnan(S[0, 3, 12000:]).any()
    names = check_seqmatch_topn(S, 1, N)
    assert ran(names, "seqmatch_topk_warp_kernel<true>") and ran(names, "topn_merge_kernel"), names


@gpu
@pytest.mark.parametrize("N,P", [(7, 300), (40, 300), (16, 20000)])
def test_topn_sequences_make_nan(N, P):
    """L = 3 on S without any NaN: a diagonal that holds both +inf and -inf sums to NaN inside the kernel, one
    with FLT_MAX twice overflows to +inf, -1e-45 alone divides to -0.0 next to +0.0; all three paths."""
    rng = np.random.default_rng(N + P)
    L = 3
    pal = np.array([np.inf, -np.inf, 0.0, -0.0, FMAX, 1.0, 2.0, -TINY], f32)
    S = pal[rng.integers(0, len(pal), (2, 6 + L - 1, P))]
    with np.errstate(invalid="ignore", over="ignore"):
        D = np.stack([O.seqmatch(S[b], L) for b in range(2)])
    assert not np.isnan(S).any() and np.isnan(D).any() and (D == np.inf).any() and (D == -np.inf).any()
    assert neg_zero(D).any()                          # -1e-45 / 3 rounds to -0.0
    names = check_seqmatch_topn(S, L, N)
    kernel = "seqmatch_topk_kernel" if N > 32 else \
        "seqmatch_topk_warp_kernel<true>" if P >= 8192 else "seqmatch_topk_warp_kernel<false>"
    assert ran(names, kernel), names


def merge_case(rng, case, Po, Qo):
    if case == "neg_nan":
        D = np.array([NANS[1], NANS[0], -np.inf, 1.0], f32)[rng.integers(0, 4, (Po, Qo))]
    elif case == "signed_zero":
        D = np.array([0.0, -0.0, -1.0], f32)[rng.integers(0, 3, (Po, Qo))]
    else:
        D = palette_matrix(rng, Po, Qo)
    return D


@gpu
@pytest.mark.parametrize("case", ["neg_nan", "signed_zero", "palette"])
@pytest.mark.parametrize("W,N", [(4, 25), (8, 64), (3, 1)])
def test_topn_merge_nonfinite(case, W, N):
    """lens_topn_merge of per-shard lists (place-sharded database) holding raw values: x86's NaN 0xffc00000,
    -0.0 next to +0.0, the palette.  The merged list is the stable top-N of the whole column."""
    from lens_b200 import ops
    rng = np.random.default_rng(W * N)
    chunk, Qo = 40, 30
    D = merge_case(rng, case, W * chunk, Qo)
    vals = np.empty((W, 1, Qo, N), f32)
    idx = np.empty((W, 1, Qo, N), np.int32)
    for w in range(W):
        i, v = stable_topn(D[w * chunk:(w + 1) * chunk], N)
        idx[w, 0], vals[w, 0] = np.where(i >= 0, i + w * chunk, -1), v
    if case == "neg_nan":
        assert (bits(vals) == 0xffc00000).any() and (bits(vals) == 0x7fc00000).any()
    if case == "signed_zero":
        assert neg_zero(vals).any() and ((vals == 0) & ~np.signbit(vals)).any()
    ov, oi = ops.topn_merge(cuda(vals), cuda(idx))
    want_i, want_v = stable_topn(D, N)
    assert np.array_equal(oi[0].cpu().numpy(), want_i)
    assert np.array_equal(ov[0].cpu().numpy(), want_v, equal_nan=True)


# --------------------------------------------------------------------------- lens_recall_bounds
def bounds_column(col, pos, K):
    """(lo, hi) of one column by brute force over its tie classes from the top: all NaNs are one class above +inf,
    then the distinct values (-0.0 and +0.0 one class).  Certain hit: a positive strictly above the class of the
    K-th entry, or the ties cannot all be negatives; possible: a positive above or among the ties."""
    nan = np.isnan(col)
    classes = [nan] + [~nan & (col == v) for v in sorted(set(col[~nan].tolist()), reverse=True)]
    g, gpos = 0, False
    for cls in classes:
        c, cpos = int(cls.sum()), int((cls & pos).sum())
        if c == 0:
            continue
        if g + c >= K:
            if gpos:
                return 1, 1
            return int(cpos > 0 and c - cpos < K - g), int(cpos > 0)
        g, gpos = g + c, gpos or cpos > 0
    return int(gpos), int(gpos)                           # K > Po: every entry is in the top K


def bounds_ref(D, GT, ns):
    keep = GT.any(0)
    lo, hi = np.zeros(len(ns), np.int64), np.zeros(len(ns), np.int64)
    for q in np.nonzero(keep)[0]:
        for i, K in enumerate(ns):
            a, b = bounds_column(D[:, q], GT[:, q], K)
            lo[i] += a
            hi[i] += b
    return lo.tolist(), hi.tolist(), int(keep.sum())


def check_bounds(D, GT, ns):
    from lens_b200 import ops
    lo, hi, nv = ops.recall_bounds(cuda(D), cuda(GT.astype(np.uint8)), ns)
    got = (lo.tolist(), hi.tolist(), int(nv.item()))
    assert got == bounds_ref(D, GT, ns), ns
    return got


@gpu
def test_recall_bounds_top_class():
    """The top class is counted: one +inf positive above a finite distractor (certain hit at K = 1), two tied +inf
    of which one is positive (possible, not certain), the same with NaN, and NaNs of different payloads tied."""
    cols = [([1.0, np.inf, 0.5], 1, (1, 1)), ([np.inf, np.inf, 0.5], 1, (0, 1)), ([1.0, np.nan, np.inf], 1, (1, 1)),
            ([NANS[0], NANS[1], np.inf], 0, (0, 1)), ([NANS[3], -np.inf, 2.0], 0, (1, 1))]
    D = np.array([c[0] for c in cols], f32).T.copy()
    GT = np.zeros(D.shape, bool)
    GT[[c[1] for c in cols], np.arange(len(cols))] = True
    for q, (_, _, want) in enumerate(cols):
        assert bounds_column(D[:, q], GT[:, q], 1) == want, q
    lo, hi, nv = check_bounds(D, GT, (1, 2, 3, 4))
    assert (lo[0], hi[0], nv) == (3, 5, 5)


def bounds_ns(Po):
    """Ascending K, several inside one tie class, K = Po and K > Po."""
    return tuple(sorted({1, 2, 3, 5, max(Po - 1, 1), Po, Po + 1, Po + 7})[-8:])


@gpu
@pytest.mark.parametrize("Po,Qo", [(1, 9), (5, 40), (33, 64), (300, 64)])
def test_recall_bounds_nonfinite(Po, Qo):
    rng = np.random.default_rng(Po * 100 + Qo)
    D = palette_matrix(rng, Po, Qo)
    GT = palette_gt(rng, D)
    if Po >= 33:
        assert_covers(D, GT)
    ns = bounds_ns(Po)
    lo, hi, nv = check_bounds(D, GT, ns)
    if Po > 1:
        assert any(a != b for a, b in zip(lo, hi))
    # numpy's default argsort lands inside the bounds whatever the row order
    keep = GT.any(0)
    for _ in range(10):
        perm = rng.permutation(Po)
        Dp, Gp = D[perm][:, keep], GT[perm][:, keep]
        order = Dp.argsort(0)
        for i, K in enumerate(ns):
            hit = int(np.take_along_axis(Gp, order[-K:], axis=0).any(0).sum())
            assert lo[i] <= hit <= hi[i], K


# --------------------------------------------------------------------------- createPR
def pr_case(rng, case):
    """[Po, Qo] f32 matrices for createPR; the assertions in test_createPR_nonfinite say what each one holds."""
    S = rng.integers(-3, 8, size=(30, 50)).astype(f32) / f32(4)
    if case == "nan":
        S[rng.integers(0, 30), rng.integers(0, 50)] = NANS[1]
    elif case == "np_nan":
        S[rng.integers(0, 30), rng.integers(0, 50)] = np.nan       # positive: the largest of the bit-pattern keys
    elif case == "nan_column":
        S[:, 7] = NANS[rng.integers(0, 4, 30)]
    elif case == "inf_max":
        S[rng.random(S.shape) < 0.05] = np.inf
    elif case == "inf_column":
        S[:, 3] = np.array([np.inf, -np.inf], f32)[rng.integers(0, 2, 30)]
    elif case == "neg_inf_min":
        S[rng.random(S.shape) < 0.05] = -np.inf
        S[:, 5] = -np.inf
    elif case == "zeros_subnormals":
        S = np.array([0.0, -0.0, TINY, -TINY, 3 * TINY], f32)[rng.integers(0, 5, (30, 50))]
    elif case == "flt_max":
        S[rng.random(S.shape) < 0.05] = FMAX
        S[rng.random(S.shape) < 0.05] = -FMAX
    return S


PR_CASES = ["nan", "nan_column", "inf_max", "inf_column", "neg_inf_min", "zeros_subnormals", "flt_max", "np_nan"]


@gpu
@pytest.mark.parametrize("dtype", ["float32", "float64"])
@pytest.mark.parametrize("matching", ["single", "multi"])
@pytest.mark.parametrize("case", PR_CASES)
def test_createPR_nonfinite(case, matching, dtype):
    """Both matching modes, float32 thresholds (float32 S) and float64 ones (float64 S), against the reference's
    createPR (O.create_pr), NaN == NaN."""
    from lens_b200.src.metrics import createPR
    rng = np.random.default_rng(PR_CASES.index(case))
    GT = rng.random((30, 50)) < 0.1
    GT[:, -1] = False
    with np.errstate(invalid="ignore", over="ignore"):
        S = pr_case(rng, case).astype(dtype)
        Pw, Rw = O.create_pr(S, GT, n_thresh=100, matching=matching)
        val = S if matching == "multi" else S.max(0)
        thresh = np.linspace(val.max(), val.min(), 100)
    assert thresh.dtype == S.dtype
    if case in ("nan", "np_nan", "nan_column"):
        assert np.isnan(val).any() and np.isnan(Pw[1:]).all() and not np.any(Rw)
    if case in ("inf_max", "inf_column"):
        assert val.max() == np.inf and not np.isnan(val).any() and np.isnan(thresh[:-1]).all()
    if case == "neg_inf_min":
        assert val.min() == -np.inf and np.isfinite(val.max())
    if case == "zeros_subnormals":
        assert neg_zero(S).any() and (np.abs(S) == TINY).any()
    if case == "flt_max":
        assert val.max() == FMAX and (matching == "single" or val.min() == -FMAX)
    P, R = createPR(S, GT, None, matching=matching, n_thresh=100)
    assert np.array_equal(np.array(P, np.float64), np.array(Pw, np.float64), equal_nan=True)
    assert np.array_equal(np.array(R, np.float64), np.array(Rw, np.float64), equal_nan=True)


# --------------------------------------------------------------------------- end to end
@gpu
@pytest.mark.parametrize("seed", [0, 1, 2])
def test_recallAtK_nonfinite(seed):
    """recallAtK == the reference's own call (numpy's default argsort) on palette matrices."""
    from lens_b200.src.metrics import recallAtK
    rng = np.random.default_rng(seed)
    D = palette_matrix(rng, 120, 64)
    GT = palette_gt(rng, D)
    assert_covers(D, GT)
    for K in (1, 2, 5, 25, 64):
        assert recallAtK(D, GT, K=K) == O.recall_at_k(D, GT, K=K), K


# 48 places x 8 queries: '0'-'3' finite (never positive), 'i' +inf, 'P' +inf and positive.  Every column ties a
# few positive +inf with a negative one at its highest index, so the tie order decides R@1 (bounds 0 and 1 per
# column): the deterministic rule of the top-N kernel misses everywhere, numpy's default argsort (quicksort, with
# or without its AVX2 / AVX-512 sorts) hits in some columns.  A bounds walk that skips +inf reports lo == hi and
# recallAtK would return the deterministic 0.0 instead of the reference's value.
INF_TIES = [
    "0131i3i30321130PPPP2iPii3P02P0P000iiPP10i201i3i0",
    "00i22P1i0ii3PP1i2iii1102iP33PP0i1PiiPiPPPi0031i3",
    "3i33P03Pi00iiPiPPi211PP12P20PP2ii3PPi1P30P2PPi00",
    "PP212i20i0PPi0P30PPP31iPiP0P300i1P0P3PP2P213Pi21",
    "22333123ii12ii10P113P3301i03Pi30i2iPPiP121i3Pi23",
    "2P103PP1i311Piii0Pi032i2iii0P221333i3P21112PiPii",
    "Pi01PPPii3ii3Pi10Pii2303iPPPP11iii312i23i1Pi102i",
    "ii232i3100102i00i0P11P32230iii200P23PP2PP30i20Pi",
]


@gpu
def test_recallAtK_inf_ties():
    from lens_b200.src.metrics import recall_detail, recallAtK
    D = np.array([[np.inf if c in "iP" else float(c) for c in col] for col in INF_TIES], f32).T.copy()
    GT = np.array([[c == "P" for c in col] for col in INF_TIES]).T.copy()
    assert bounds_ref(D, GT, (1,)) == ([0], [8], 8)
    assert O.recall_at_k(D, GT, K=1, kind="stable") == 0.0
    d = recall_detail(D, GT, (1,))
    assert (d["lo"], d["hi"], d["ties_decided"]) == ([0.0], [1.0], [1])
    assert recallAtK(D, GT, K=1) == O.recall_at_k(D, GT, K=1)


def write_png_gray(path, img):
    """8-bit greyscale PNG, written with zlib alone."""
    def chunk(kind, data):
        return struct.pack(">I", len(data)) + kind + data + struct.pack(">I", zlib.crc32(kind + data))
    h, w = img.shape
    raw = b"".join(b"\x00" + img[r].tobytes() for r in range(h))
    with open(path, "wb") as f:
        f.write(b"\x89PNG\r\n\x1a\n" + chunk(b"IHDR", struct.pack(">IIBBBBB", w, h, 8, 0, 0, 0, 0))
                + chunk(b"IDAT", zlib.compress(raw)) + chunk(b"IEND", b""))


@gpu
def test_run_sad_zero_distance(tmp_path):
    """run_sad on a PNG tree with repeated frame runs, so that sequence distances are 0 and similarities +inf:
    query frames 2-5 equal reference frames 4-7 and 0-3 (two tied +inf in queries 2 and 3, one of them positive),
    and both traverses hold a run of empty frames.  Against the reference restated in numpy: SAD distances,
    O.seqmatch, 1 / D, O.create_pr, O.recall_at_k."""
    from lens_b200.src.sad import RECALL_NS, run_sad
    rng = np.random.default_rng(7)
    L, Q, R = 3, 10, 30
    ref = rng.integers(0, 256, size=(R, 6, 6), dtype=np.uint8)
    qry = rng.integers(0, 256, size=(Q, 6, 6), dtype=np.uint8)
    ref[0:4] = ref[4:8]
    qry[2:6] = ref[4:8]
    qry[7:10] = 0
    ref[20:23] = 0
    for name, frames in (("ref", ref), ("qry", qry)):
        (tmp_path / name).mkdir()
        for i, fr in enumerate(frames):
            write_png_gray(str(tmp_path / name / f"frame_{i}.png"), fr)
    GT = rng.random((R - L + 1, Q - L + 1)) < 0.1
    GT[[4, 5, 20], [2, 3, 7]] = True                 # zero distances: q = 2, 3 at r = q + 2, and the empty runs
    GT[[0, 1], [2, 3]] = False                       # their tied twins at r = q - 2 are negatives
    dist = np.abs(qry.reshape(Q, 1, -1).astype(np.int64) - ref.reshape(1, R, -1).astype(np.int64)).sum(-1)
    D = O.seqmatch(dist.astype(f32), L)
    with np.errstate(divide="ignore"):
        sim = f32(1) / D
    assert sim[4, 2] == sim[0, 2] == sim[5, 3] == sim[1, 3] == np.inf and sim[20, 7] == np.inf
    Pw, Rw = O.create_pr(sim, GT, n_thresh=100, matching="single")
    want_recall = [round(O.recall_at_k(sim, GT, K=n), 2) for n in RECALL_NS]
    PR, recall = run_sad(str(tmp_path / "ref"), str(tmp_path / "qry"), GT, None, L)
    assert np.array_equal(np.array(PR["Precision"], np.float64), np.array(Pw, np.float64), equal_nan=True)
    assert np.array_equal(np.array(PR["Recall"], np.float64), np.array(Rw, np.float64), equal_nan=True)
    assert recall == want_recall
