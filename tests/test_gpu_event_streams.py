"""Many independent event streams in one binning call (lens_bin_event_streams) and the pipeline entry points
built on it (InferencePipeline.step_events / step_event_groups).

Every binning case compares each stream's frames, pooled pixels and window counts with ops.bin_events on an
aligned copy of that stream's events and with the CPU oracle, and checks with torch.profiler that the intended
kernel ran.  The pipeline cases compare with step(pooled=...) on per-stream bin_events output bit for bit."""
import ctypes as C
import re

import numpy as np
import pytest
import torch

from conftest import synth_weights
from oracle import oracle as O

gpu = pytest.mark.gpu
W_US = 1000


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
    return any(re.search("::%s[(<]" % kernel, n) for n in names)


def host_streams(seed, Q, sensor, hot_xy, lead=5, trail=3):
    """Streams of every length residue mod 8 (and an empty one, one entirely before t0, one entirely after the
    last window, one with a hot pixel that collects > 255 events in a window), concatenated in stream order
    between `lead` and `trail` events that belong to no stream.  -> (t u32, x u16, y u16, offsets i64, t0 u32)."""
    rng = np.random.default_rng(seed)
    lens = [8 * 40 + r for r in range(8)] + [1, 7, 1003, 4097] + [0, 200, 150, 2000]
    kinds = ["normal"] * 12 + ["empty", "before", "after", "hot"]
    ts, xs, ys, t0s, offsets = [], [], [], [], [lead]
    for kind, n in zip(kinds, lens):
        t0 = int(rng.integers(W_US // 4, 3 * W_US))
        lo, hi = t0 - W_US // 4, t0 + Q * W_US + W_US // 4
        if kind == "before":
            lo, hi = 0, t0
        elif kind == "after":
            lo, hi = t0 + Q * W_US, t0 + (Q + 2) * W_US
        t = np.sort(rng.integers(lo, hi, n))
        x, y = rng.integers(0, sensor, n), rng.integers(0, sensor, n)
        if kind == "hot":
            t = np.sort(rng.integers(t0, t0 + W_US, n))           # all in window 0
            m = rng.random(n) < 0.5
            x[m], y[m] = hot_xy
        ts.append(t); xs.append(x); ys.append(y); t0s.append(t0)
        offsets.append(offsets[-1] + n)
    junk = lambda k: rng.integers(0, 1 << 20, k)                   # noqa: E731  (events outside every stream)
    t = np.concatenate([np.sort(junk(lead))] + ts + [np.sort(junk(trail))]).astype(np.uint32)
    x = np.concatenate([junk(lead) % sensor] + xs + [junk(trail) % sensor]).astype(np.uint16)
    y = np.concatenate([junk(lead) % sensor] + ys + [junk(trail) % sensor]).astype(np.uint16)
    return t, x, y, np.array(offsets, np.int64), np.array(t0s, np.uint32)


def dev_events(t, x, y):
    return cuda(t.view(np.int32)), cuda(x.view(np.int16)), cuda(y.view(np.int16))


def per_stream_bin_events(t, x, y, offsets, t0, Q, roi, k, **kw):
    """ops.bin_events on an aligned copy of every stream -> list of (frames, pooled, counts) on the host."""
    from lens_b200 import ops
    out = []
    for b in range(len(t0)):
        s = slice(int(offsets[b]), int(offsets[b + 1]))
        tb, xb, yb = dev_events(t[s], x[s], y[s])
        f, p, c = ops.bin_events(tb, xb, yb, int(t0[b]), W_US, Q, roi, k, **kw)
        out.append((f.cpu().numpy(), p.cpu().numpy(), c.cpu().numpy()))
    return out


BIN_CASES = {   # name: (sensor, roi, k, roi_x0, roi_y0, index_shift, wrap_u8, kernel, hot pixel)
    "pow2": (64, 64, 4, 0, 0, 1, True, "bin_pow2_kernel", (17, 9)),
    "pow2_shift0_saturate": (64, 64, 4, 0, 0, 0, False, "bin_pow2_kernel", (17, 9)),
    "speck_crop": (128, 80, 8, 23, 0, 1, True, "bin_kernel", (23 + 19, 11)),
    "speck_crop_shift0_saturate": (128, 80, 8, 23, 0, 0, False, "bin_kernel", (23 + 19, 11)),
    "banded_roi200": (256, 200, 8, 0, 0, 1, True, "bin_kernel", (3, 195)),
    "k1": (40, 24, 1, 4, 6, 1, True, "bin_kernel", (10, 10)),
}


@gpu
@pytest.mark.parametrize("case", sorted(BIN_CASES))
def test_bin_event_streams_equal_per_stream_binning(case):
    from lens_b200 import ops
    sensor, roi, k, x0, y0, shift, wrap, kernel, hot = BIN_CASES[case]
    Q = 4
    t, x, y, offsets, t0 = host_streams(len(case), Q, sensor, hot)
    kw = dict(roi_x0=x0, roi_y0=y0, index_shift=shift, wrap_u8=wrap)
    td, xd, yd = dev_events(t, x, y)
    (f, p, c), names = kernels_run(lambda: ops.bin_event_streams(td, xd, yd, cuda(offsets), cuda(t0.view(np.int32)),
                                                                 W_US, Q, roi, k, want_frames=True, **kw))
    assert ran(names, kernel) and not ran(names, {"bin_kernel": "bin_pow2_kernel"}.get(kernel, "bin_kernel")), names
    f, p, c = f.cpu().numpy(), p.cpu().numpy(), c.cpu().numpy()
    dims = roi // k
    assert f.shape == (len(t0), Q, roi, roi) and p.shape == (len(t0), Q, dims * dims) and c.shape == (len(t0), Q)
    want = per_stream_bin_events(t, x, y, offsets, t0, Q, roi, k, **kw)
    for b in range(len(t0)):
        s = slice(int(offsets[b]), int(offsets[b + 1]))
        of, op, oc = O.bin_events(t[s], x[s], y[s], int(t0[b]), W_US, Q, roi, k, **kw)
        for got, mine, ref in zip((f[b], p[b], c[b]), want[b], (of, op, oc)):
            assert np.array_equal(got, mine), (case, b)
            assert np.array_equal(got, ref), (case, b)
    # the conditions the special streams exist for
    lens = np.diff(offsets)
    assert set(lens % 8) == set(range(8))
    assert (c[lens == 0] == 0).all() and (c[-3] == 0).all() and (c[-2] == 0).all()   # empty, before, after
    hx, hy = hot
    s = slice(int(offsets[-2]), int(offsets[-1]))
    n_hot = int(((x[s] == hx) & (y[s] == hy) & (t[s] < t0[-1] + W_US)).sum())
    assert n_hot > 255
    # want_frames=False: the same pooled pixels and counts
    _, p2, c2 = ops.bin_event_streams(td, xd, yd, cuda(offsets), cuda(t0.view(np.int32)), W_US, Q, roi, k, **kw)
    assert np.array_equal(p2.cpu().numpy(), p) and np.array_equal(c2.cpu().numpy(), c)


@gpu
def test_single_stream_equals_bin_events_and_launch_count_is_independent_of_B():
    from lens_b200 import ops, _lib
    rng = np.random.default_rng(4)
    n, Q, roi, k = 50_003, 7, 80, 8
    t = np.sort(rng.integers(0, 9 * W_US, n)).astype(np.uint32)
    x, y = rng.integers(0, 128, n).astype(np.uint16), rng.integers(0, 128, n).astype(np.uint16)
    td, xd, yd = dev_events(t, x, y)
    for t0 in (0, 333):
        want = ops.bin_events(td, xd, yd, t0, W_US, Q, roi, k, roi_x0=23)
        got = ops.bin_event_streams(td, xd, yd, cuda(np.array([0, n], np.int64)), cuda(np.array([t0], np.int32)),
                                    W_US, Q, roi, k, roi_x0=23, want_frames=True)
        for a, b in zip(got, want):
            assert np.array_equal(a.cpu().numpy()[0], b.cpu().numpy())
    launches = []
    for B in (1, 256):
        offsets = cuda(np.linspace(0, n, B + 1).astype(np.int64))
        t0 = cuda(np.zeros(B, np.int32))
        torch.cuda.synchronize()
        l0 = _lib.launch_count()
        ops.bin_event_streams(td, xd, yd, offsets, t0, W_US, 2, roi, k, roi_x0=23)
        launches.append(_lib.launch_count() - l0)
    assert launches[0] == launches[1] == 2
    # B = 0 and Q = 0 launch nothing
    l0 = _lib.launch_count()
    _, p, c = ops.bin_event_streams(td, xd, yd, cuda(np.array([0], np.int64)), cuda(np.zeros(0, np.int32)),
                                    W_US, 3, roi, k)
    _, p2, c2 = ops.bin_event_streams(td, xd, yd, offsets, t0, W_US, 0, roi, k)
    assert _lib.launch_count() == l0 and p.shape == (0, 3, 100) and c2.shape == (256, 0)


@gpu
def test_check_sorted():
    from lens_b200 import ops, _lib
    t, x, y, offsets, t0 = host_streams(8, 3, 64, (1, 1))
    starts = offsets[1:-1][np.diff(offsets)[1:] > 0]
    assert (t[starts] < t[starts - 1]).any()                       # the stream starts do descend
    args = lambda t_, off: (*dev_events(t_, x, y), cuda(off), cuda(t0.view(np.int32)), W_US, 3, 64, 4)  # noqa: E731
    _, p, _ = ops.bin_event_streams(*args(t, offsets), check_sorted=True)
    bad_t = t.copy()
    i = int(offsets[1]) + 10                                      # inside stream 1
    bad_t[i], bad_t[i + 1] = bad_t[i + 1], bad_t[i] - 1
    with pytest.raises(ValueError):
        ops.bin_event_streams(*args(bad_t, offsets), check_sorted=True)
    for off in (offsets[::-1].copy(),                              # decreasing
                np.concatenate([[-1], offsets[1:]]),               # before the arrays
                np.concatenate([offsets[:-1], [len(t) + 1]]),      # past the end
                np.concatenate([offsets[:3], [10 ** 15], offsets[4:]])):
        a = args(t, off)
        torch.cuda.synchronize()
        l0 = _lib.launch_count()
        with pytest.raises(ValueError):
            ops.bin_event_streams(*a, check_sorted=True)
        assert _lib.launch_count() - l0 == 1                       # the check only: nothing was binned
    assert (np.diff(offsets) == 0).any()       # the accepted streams include an empty one


def pipeline(Wf, Wo, T, L, B, roi=80, k=8):
    from lens_b200.pipeline import InferencePipeline
    return InferencePipeline(torch.from_numpy(Wf), torch.from_numpy(Wo), roi=roi, k=k, T=T, L=L, max_streams=B)


def assert_same_step(a, b):
    for key in ("S", "top_val", "top_idx", "hits", "n_valid", "overflow"):
        assert (a[key] is None and b[key] is None) or torch.equal(a[key], b[key]), key


def device_streams(B, Q, epw, seed):
    from lens_b200 import synth
    return synth.event_streams_device(B, Q, window_us=W_US * 250, events_per_window=epw, seed=seed)


@gpu
@pytest.mark.parametrize("path", ["tensor_core", "cuda_core"])
def test_step_events_equals_step_on_binned_pooled(path):
    from lens_b200 import synth
    B, Q, L, T, F = (64, 4, 2, 30, 160) if path == "tensor_core" else (6, 5, 2, 30, 160)
    P = 1024 if path == "tensor_core" else 300
    Wf, Wo = synth_weights(100, F, P, seed=3)
    t, x, y, off, t0 = device_streams(B, Q, 131_072 if path == "tensor_core" else 60_000, seed=21)
    gt = cuda(synth.gt_centers(B, Q - L + 1, P - L + 1, seed=5))
    pa, pb = pipeline(Wf, Wo, T, L, B), pipeline(Wf, Wo, T, L, B)
    oh, th = off.cpu().numpy(), t0.cpu().numpy()
    pooled = []
    for b in range(B):
        s = slice(int(oh[b]), int(oh[b + 1]))
        _, p, _ = ops_bin(t[s].clone(), x[s].clone(), y[s].clone(), int(th[b]), Q)
        pooled.append(p)
    pooled = torch.stack(pooled)
    for _ in range(2):                                             # state carries over between calls
        got, names = kernels_run(lambda: pa.step_events(t, x, y, off, t0, W_US * 250, Q, roi_x0=23, gt_center=gt,
                                                        gt_tol=1))
        want = pb.step(pooled=pooled, gt_center=gt, gt_tol=1)
        assert_same_step(got, want)
        assert ran(names, "bin_kernel")
        assert ran(names, "output_tc_kernel") == (path == "tensor_core"), names
        assert ran(names, "output_simt_kernel") == (path == "cuda_core"), names
    assert got["events_per_window"].shape == (B, Q) and int(got["events_per_window"].min()) > 0
    assert float(got["S"].sum()) > 0


def ops_bin(t, x, y, t0, Q):
    from lens_b200 import ops
    return ops.bin_events(t, x, y, t0, W_US * 250, Q, 80, 8, roi_x0=23)


@gpu
def test_step_events_small_case_equals_oracle():
    B, Q, L, T, F, P = 3, 5, 2, 40, 96, 200
    Wf, Wo = synth_weights(100, F, P, seed=9)
    t, x, y, off, t0 = device_streams(B, Q, 70_000, seed=4)
    out = pipeline(Wf, Wo, T, L, B).step_events(t, x, y, off, t0, W_US * 250, Q, roi_x0=23)
    th, xh, yh, oh, t0h = (a.cpu().numpy() for a in (t, x, y, off, t0))
    pooled, counts = [], []
    for b in range(B):
        s = slice(int(oh[b]), int(oh[b + 1]))
        _, p, c = O.bin_events(th[s].view(np.uint32), xh[s].view(np.uint16), yh[s].view(np.uint16), int(t0h[b]),
                               W_US * 250, Q, 80, 8, roi_x0=23)
        pooled.append(p); counts.append(c)
    assert np.array_equal(out["events_per_window"].cpu().numpy(), np.stack(counts))
    onet = O.OracleSNN(Wf, Wo, O.raster_uniforms(T, 80, 8), T, n_streams=B)
    So = onet.run_streams(np.stack(pooled))
    assert np.array_equal(out["S"].cpu().numpy(), So)
    assert So.sum() > 0
    for b in range(B):
        io, vo = O.topk(O.seqmatch(So[b], L), 25)
        assert np.array_equal(out["top_idx"][b].cpu().numpy(), io)
        assert np.array_equal(out["top_val"][b].cpu().numpy(), vo)


def groups_of(t, x, y, off, t0, sizes):
    """(b0, t, x, y, offsets, t0) per group of consecutive streams, each group's events in its own (aligned)
    arrays with offsets relative to them."""
    oh = off.cpu().numpy()
    b0 = 0
    for n in sizes:
        e0, e1 = int(oh[b0]), int(oh[b0 + n])
        yield b0, t[e0:e1].clone(), x[e0:e1].clone(), y[e0:e1].clone(), off[b0:b0 + n + 1] - e0, t0[b0:b0 + n].clone()
        b0 += n


@gpu
def test_step_event_groups_equals_step_events():
    from lens_b200 import synth
    from lens_b200._lib import LensError
    B, Q, L, T, F, P = 13, 4, 3, 30, 128, 400
    Wf, Wo = synth_weights(100, F, P, seed=5)
    t, x, y, off, t0 = device_streams(B, Q, 50_000, seed=8)
    gt = cuda(synth.gt_centers(B, Q - L + 1, P - L + 1, seed=2))
    pa, pb = pipeline(Wf, Wo, T, L, B), pipeline(Wf, Wo, T, L, B)
    for _ in range(2):
        want = pa.step_events(t, x, y, off, t0, W_US * 250, Q, roi_x0=23, gt_center=gt, gt_tol=1)
        got = pb.step_event_groups(groups_of(t, x, y, off, t0, [4, 2, 6, 1]), B, Q, W_US * 250, roi_x0=23,
                                   gt_center=gt, gt_tol=1)
        assert_same_step(got, want)
        assert torch.equal(got["events_per_window"], want["events_per_window"])
    with pytest.raises(LensError):
        pb.step_event_groups(groups_of(t, x, y, off, t0, [3, 10]), B, Q, W_US * 250, roi_x0=23)


@gpu
def test_empty_windows_stay_queries():
    from lens_b200 import synth
    B, Q, L, T, F, P = 4, 5, 2, 30, 96, 150
    Wf, Wo = synth_weights(100, F, P, seed=6)
    t, x, y, off, t0 = (a.cpu().numpy() for a in device_streams(B, Q, 40_000, seed=12))
    # stream 1 loses every event of windows 1 and 3
    s = slice(int(off[1]), int(off[2]))
    rel = (t[s].astype(np.int64) - int(t0[1])) // (W_US * 250)
    keep = np.ones(len(t), bool)
    keep[s] = (rel != 1) & (rel != 3)
    t, x, y = t[keep], x[keep], y[keep]
    off = off.copy()
    off[2:] -= int((~keep).sum())
    args = (cuda(t), cuda(x), cuda(y), cuda(off), cuda(t0), W_US * 250, Q)
    out = pipeline(Wf, Wo, T, L, B).step_events(*args, roi_x0=23)
    from lens_b200 import ops
    _, pooled, n_ev = ops.bin_event_streams(*args[:7], 80, 8, roi_x0=23)
    ev = out["events_per_window"].cpu().numpy()
    assert np.array_equal(ev, n_ev.cpu().numpy())
    assert (ev[1, [1, 3]] == 0).all() and (ev[:, [0, 2, 4]] > 0).all() and (ev[[0, 2, 3]] > 0).all()
    assert (pooled[1, [1, 3]] == 0).all()
    want = pipeline(Wf, Wo, T, L, B).step(pooled=pooled)
    assert_same_step(out, want)


def test_argument_validation_without_a_gpu():
    from lens_b200 import _lib
    L = _lib.lib()
    a = C.c_void_p(0x10000)                                        # never dereferenced: checks come first

    def call(B=2, Q=3, window=1000, x=a, n=16, roi=80, k=8):
        return L.lens_bin_event_streams(a, x, a, n, a, a, B, Q, window, 0, 0, roi, k, 1, 1, None, a, a, a, None)
    for kw, word in ((dict(B=-1), b"negative"), (dict(Q=-2), b"negative"), (dict(window=0), b"window_us"),
                     (dict(x=C.c_void_p(0x10002)), b"aligned"), (dict(B=1 << 16, Q=1 << 16), b"too many"),
                     (dict(k=0), b"roi")):
        assert call(**kw) == -1, kw
        assert word in L.lens_last_error(), (kw, L.lens_last_error())
    assert L.lens_bin_event_streams(a, a, a, 16, None, a, 2, 3, 1000, 0, 0, 80, 8, 1, 1, None, a, a, a, None) == -1
    assert b"offsets" in L.lens_last_error()
    assert L.lens_check_sorted_segments_u32(a, 16, a, -1, a, None) == -1
    assert L.lens_check_sorted_segments_u32(a, 16, None, 2, a, None) == -1
    assert L.lens_check_sorted_segments_u32(C.c_void_p(0x10004), 16, a, 2, a, None) == -1
