"""Every kernel variant of the spiking network against the CPU oracle, bit for bit.

forward_common (snn.cu) picks the hidden-layer kernel (tensor-core, raster or generic feature_kernel) and the
output-layer kernel (tensor-core or CUDA-core) from the shape, the IAF parameters, the mode and whether
per-step debug buffers are requested, and the tensor-core kernel has one template instantiation per
(threshold 1 / v_min -1, debug, K steps, layer).  Each case below targets one of these and checks with the
profiler that it actually ran, so a later dispatch change cannot turn it into a test of another kernel;
each also first asserts, on the oracle's results, the condition it exists for (multi-spike steps, overflow,
6-plane tiles, ...), so it cannot become vacuous.  Compared: spike counts, all three membrane potentials and
the overflow counter after each of two calls (state carry-over), plus every step where the debug path runs.
All weights are exact on the fixed-point grid (n_inexact == 0) and per-query counts stay far below 2^24.
"""
import math

import numpy as np
import pytest
import torch

from conftest import synth_weights, synth_pooled
from oracle import oracle as O

pytestmark = pytest.mark.gpu

MAX_SPIKE = 127      # LENS_MAX_SPIKE


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


def assert_ran(names, *kernels):
    for k in kernels:
        k = "".join(k.split())
        assert any(k in n for n in names), f"{k} did not run; kernels: {sorted(names)}"


def tidy(W, floor=2.0 ** -12):
    """Zero the weights below `floor`: keeps every row within the fixed-point grid's 46 bits."""
    return np.where(np.abs(W) < floor, 0.0, W).astype(np.float32)


def row_planes(W):
    """Radix-256 digit planes the tensor-core kernel needs per row of W (snn.cu weights_to_fixed_kernel +
    snn_tc.cu planes_kernel): row weights as integers over the row's lowest set bit, balanced digits."""
    out = []
    for row in np.asarray(W, np.float32):
        nz = [float(w) for w in row if w != 0.0]
        if not nz:
            out.append(0)
            continue
        ints = [(int(m * 2 ** 53), e - 53) for m, e in (math.frexp(w) for w in nz)]   # w = m * 2^e exactly
        lsb = min(e + ((m & -m).bit_length() - 1) for m, e in ints)
        top = 0
        for m, e in ints:
            m = m << (e - lsb) if e >= lsb else m >> (lsb - e)      # exact: lsb is at or below m's lowest bit
            for j in range(6):
                d = ((m + 128) & 255) - 128
                if d:
                    top = max(top, j + 1)
                m = (m - d) >> 8
            assert m == 0, "row needs more than 6 digit planes"
        out.append(top)
    return np.array(out)


def tile_planes(W):
    p = row_planes(W)
    return np.array([max(5, p[i:i + 128].max()) for i in range(0, len(p), 128)])


class Oracle:
    """The oracle's results for `pooled` split into `calls` consecutive calls (always with every step)."""

    def __init__(self, Wf, Wo, T, pooled, thr=1.0, vmin=-1.0, calls=2):
        self.Wf, self.Wo, self.T, self.pooled, self.thr, self.vmin = Wf, Wo, T, pooled, thr, vmin
        B, Q, I = pooled.shape
        self.dims = math.isqrt(I)
        assert self.dims ** 2 == I
        self.U = O.raster_uniforms(T, self.dims, 1)
        self.parts = np.array_split(np.arange(Q), calls)
        net = O.OracleSNN(Wf, Wo, self.U, T, thr=thr, v_min=vmin, n_streams=B)
        self.calls = []
        for part in self.parts:
            c, h, o = net.run_streams(pooled[:, part], want_steps=True)
            self.calls.append(dict(counts=c, hidden=h, out=o, state=net.state(), overflow=net.overflow()))
        self.counts = np.concatenate([c["counts"] for c in self.calls], 1)
        self.hidden = np.concatenate([c["hidden"] for c in self.calls], 1)
        self.out = np.concatenate([c["out"] for c in self.calls], 1)
        self.overflow = self.calls[-1]["overflow"]

    def check_gpu(self, mode, want_steps):
        """Run the same calls on the GPU, compare everything, return the kernels that ran."""
        from lens_b200.network import B200Network
        B = self.pooled.shape[0]
        net = B200Network(torch.from_numpy(self.Wf), torch.from_numpy(self.Wo), roi=self.dims, k=1,
                          num_timesteps=self.T, spike_threshold=self.thr, min_v_mem=self.vmin, max_streams=B,
                          U=torch.from_numpy(self.U))
        assert net.n_inexact == 0
        names = set()
        for part, want in zip(self.parts, self.calls):
            r, n = kernels_run(lambda: net.run_streams(pooled=cuda(self.pooled[:, part]), mode=mode,
                                                       want_steps=want_steps))
            names |= n
            c = r[0] if want_steps else r
            assert np.array_equal(c.cpu().numpy(), want["counts"]), "spike counts differ"
            if want_steps:
                # the GPU reports the hidden spike count it transported (clipped to LENS_MAX_SPIKE, int8); the
                # oracle's debug byte is the unclipped count saturated at 255
                assert np.array_equal(r[1].cpu().numpy(), np.minimum(want["hidden"], MAX_SPIKE)), "hidden spikes differ"
                assert np.array_equal(r[2].cpu().numpy(), want["out"]), "output spikes differ"
            for name, a, b in zip(("v0", "v1", "v2"), want["state"], net.state()):
                assert np.array_equal(b.cpu().numpy(), a), f"membrane potential {name} differs"
            assert net.overflow() == want["overflow"], "overflow counter differs"
        return names


def dense_pooled(B, Q, I, seed):
    """Pixels spread over 0..255 (every input fires in about half the steps): busy hidden layers at small I."""
    rng = np.random.default_rng(seed)
    p = rng.integers(0, 256, (B, Q, I)).astype(np.uint8)
    p[rng.random((B, Q, I)) < 0.3] = 0
    return p


# ------------------------------------------------------------------------ hidden layer on tensor cores
@pytest.mark.parametrize("want_steps", [False, True])
@pytest.mark.parametrize("B,T", [(3, 45), (6, 32)])       # odd last stream / a block with a lone last pair
@pytest.mark.parametrize("I,F,P,K", [(16, 40, 130, 0), (49, 63, 200, 2), (81, 200, 150, 0), (196, 224, 260, 0)])
def test_hidden_tc_kernels(I, F, P, K, B, T, want_steps):
    """Ip = 32 / 64 / 96 / 224: the K = 2 and generic K = 0 instantiations of the hidden-layer kernel."""
    Wf, Wo = synth_weights(I, F, P, seed=I + F)
    Wf = tidy(Wf)
    o = Oracle(Wf, Wo, T, dense_pooled(B, 4, I, seed=I), calls=2)
    assert o.hidden.sum() > 0 and o.counts.sum() > 0 and o.overflow == 0
    names = o.check_gpu(mode=2, want_steps=want_steps)
    assert_ran(names, f"output_tc_kernel<true, {str(want_steps).lower()}, {K}, true>")


# ------------------------------------------------------------------------ 5- and 6-plane tiles in one launch
def mixed_plane_rows(W, six, rng):
    """Rows in `six` get one weight 2^-20 below the row maximum with a full 24-bit significand (> 40 significant
    bits: 6 digit planes); the others keep only weights within 2^-10 of their maximum (5 planes)."""
    W = W.copy()
    for r in range(W.shape[0]):
        m = np.abs(W[r]).max()
        if six[r]:
            j = rng.integers(0, W.shape[1])
            W[r, j] = np.float32(m * 2.0 ** -20 * (1 + (rng.integers(1, 2 ** 23) | 1) * 2.0 ** -23))
        else:
            W[r, np.abs(W[r]) < m * 2.0 ** -10] = 0.0
    return W


@pytest.mark.parametrize("want_steps", [False, True])
def test_mixed_digit_planes(want_steps):
    """Place tiles alternate 5 and 6 planes (and so do the two feature tiles of F = 200); with 400 streams the
    super-items outnumber the SMs several times, so every CTA moves between both kinds of tile."""
    I, F, P, T, B = 100, 200, 5 * 128 + 37, 32, 400
    rng = np.random.default_rng(11)
    Wf, Wo = synth_weights(I, F, P, seed=3)
    Wf = mixed_plane_rows(tidy(Wf), np.arange(F) < 128, rng)
    Wo = mixed_plane_rows(Wo, (np.arange(P) // 128) % 2 == 0, rng)
    assert tile_planes(Wo).tolist() == [6, 5, 6, 5, 6, 5] and tile_planes(Wf).tolist() == [6, 5]
    o = Oracle(Wf, Wo, T, synth_pooled(B, 2, I, seed=4), calls=2)
    for tile in range(6):
        assert o.counts[..., tile * 128:(tile + 1) * 128].sum() > 0
    assert o.hidden[..., :128].sum() > 0 and o.hidden[..., 128:].sum() > 0
    names = o.check_gpu(mode=2, want_steps=want_steps)
    d = str(want_steps).lower()
    assert_ran(names, f"output_tc_kernel<true, {d}, 7, false>", f"output_tc_kernel<true, {d}, 4, true>")


# ------------------------------------------------------------------------ multi-spike steps in the output scan
@pytest.mark.parametrize("want_steps", [False, True])
def test_output_multi_spike_tiles(want_steps):
    """W_out scaled by 16 (exactly) on place tiles 1 and 3 only: those tiles fire several spikes in some steps and
    leave the fast scan, their neighbours in the same stream pair and chunk stay on it."""
    I, F, P, T, B = 100, 200, 5 * 128, 32, 4
    Wf, Wo = synth_weights(I, F, P, seed=5)
    Wf = tidy(Wf)
    scaled = np.zeros(P, bool)
    scaled[128:256] = scaled[384:512] = True
    Wo[scaled] *= 16.0
    o = Oracle(Wf, Wo, T, synth_pooled(B, 4, I, seed=6), calls=2)
    # per (stream pair, chunk, place tile): the largest output step count
    m = o.out.reshape(B // 2, 2, -1, 32, P // 128, 128).max(axis=(1, 3, 5))
    assert m[..., ~scaled[::128]].max() == 1 and (m[..., scaled[::128]] >= 2).any()
    both = (m[..., scaled[::128]].max(-1) >= 2) & (m[..., ~scaled[::128]].min(-1) == 1)
    assert both.any(), "no pair and chunk in which a redone tile has fast neighbours"
    assert (m == 2).any(), "no tile whose largest step is exactly two spikes"
    names = o.check_gpu(mode=2, want_steps=want_steps)
    assert_ran(names, f"output_tc_kernel<true, {str(want_steps).lower()}, 7, false>")


# ------------------------------------------------------------------------ hidden spikes beyond LENS_MAX_SPIKE
def single_step_input(U, half):
    """(input, pixel) such that the raster fires that input in exactly one step of the 32, in half `half`."""
    Uq = np.array([[np.searchsorted(np.float32(np.arange(1, 256)) / np.float32(255.0), u, side="right")
                    for u in row] for row in U[:32]])            # pixel > Uq[t, i]  <=>  U[t, i] < pixel / 255
    for i in range(U.shape[1]):
        t = np.argmin(Uq[:, i])
        if (Uq[:, i] == Uq[t, i]).sum() == 1 and t // 16 == half and Uq[t, i] < 255:
            return i, int(Uq[t, i]) + 1
    raise AssertionError("no input fires in a single step")


@pytest.mark.parametrize("want_steps", [False, True])
@pytest.mark.parametrize("mode", [1, 2])
def test_hidden_overflow(mode, want_steps):
    """Two hidden neurons receive 200 per input spike from one input each, which fires in a single step of the
    first (resp. second) 16-step half of the chunk: > 127 spikes, clipped and counted.  Streams 0 (first pair),
    3 (second pair, other half) and 4 (odd last pair) overflow; their pair partners do not."""
    I, F, P, T, B = 100, 200, 300, 32, 5
    Wf, Wo = synth_weights(I, F, P, seed=7)
    Wf = tidy(Wf)
    pooled = synth_pooled(B, 4, I, seed=8)
    U = O.raster_uniforms(T, 10, 1)
    (ia, va), (ib, vb) = single_step_input(U, 0), single_step_input(U, 1)
    fa, fb = 17, 150
    Wf[[fa, fb]] = 0.0
    Wf[fa, ia] = Wf[fb, ib] = 200.0
    pooled[:, :, [ia, ib]] = 0
    pooled[0, :, ia] = va
    pooled[3, :, ib] = vb
    pooled[4, :, ia] = va
    o = Oracle(Wf, Wo, T, pooled, calls=2)
    over = (o.hidden > MAX_SPIKE).any(axis=(1, 2))
    assert o.overflow > 0 and over.tolist() == [True, False, False, True, True]
    names = o.check_gpu(mode=mode, want_steps=want_steps)
    if mode == 1:
        assert_ran(names, f"feature_raster_kernel<{str(want_steps).lower()}>", "output_simt_kernel")
    else:
        assert_ran(names, f"output_tc_kernel<true, {str(want_steps).lower()}, 4, true>")


def test_input_overflow_float_seam():
    """`net(x)` with x >= 128 at some inputs: IAF#0 of feature_kernel fires more than 127 spikes in one step."""
    from lens_b200.network import B200Network
    from lens_b200._lib import LensError
    I, F, P, T, Bp, dims = 100, 120, 90, 20, 3, 10
    Wf, Wo = synth_weights(I, F, P, seed=9)
    Wf = tidy(Wf)
    rng = np.random.default_rng(10)
    x = (rng.random((Bp, T, I)) < 0.05).astype(np.float32)
    x[1, 3, [5, 40]] = [130.0, 200.5]
    x[2, 17, 77] = 128.0
    onet = O.OracleSNN(Wf, Wo, None, T, n_streams=Bp)
    want = [onet.forward_float(x)]
    state1, over1 = onet.state(), onet.overflow()
    want.append(onet.forward_float(x))
    assert over1 >= 3 and onet.overflow() > over1
    gnet = B200Network(torch.from_numpy(Wf), torch.from_numpy(Wo), roi=dims, k=1, num_timesteps=T)
    gnet.check_overflow = False
    xg = cuda(x.reshape(Bp * T, 1, dims, dims))
    got, names = kernels_run(lambda: gnet(xg))
    assert np.array_equal(got.cpu().numpy(), want[0].reshape(Bp * T, P))
    for a, b in zip(state1, gnet.state()):
        assert np.array_equal(b.cpu().numpy(), a)
    assert gnet.overflow() == over1
    assert np.array_equal(gnet(xg).cpu().numpy(), want[1].reshape(Bp * T, P))
    for a, b in zip(onet.state(), gnet.state()):
        assert np.array_equal(b.cpu().numpy(), a)
    assert gnet.overflow() == onet.overflow()
    assert_ran(names, "feature_kernel(", "output_simt_kernel")
    gnet.check_overflow = True
    with pytest.raises(LensError, match="more than 127 spikes"):
        gnet(xg)


# ------------------------------------------------------------------------ spike_threshold / min_v_mem
@pytest.mark.parametrize("want_steps", [False, True])
@pytest.mark.parametrize("mode", [1, 2])
@pytest.mark.parametrize("thr,vmin", [(1, -0.5), (1, -3), (0.5, -1), (2, -1), (0.75, -0.25), (1, 0.5), (1, 1)])
def test_iaf_parameters(thr, vmin, mode, want_steps):
    """Other thresholds and floors than the reference's 1 / -1: the generic output scans, feature_kernel on
    pooled input, and the raster kernel with v_min != -1.  With v_min > 0 IAF#0 leaves rest by itself."""
    I, F, P, T, B = 100, 100, 200, 40, 3
    Wf, Wo = synth_weights(I, F, P, seed=12)
    Wf = tidy(Wf)
    o = Oracle(Wf, Wo, T, dense_pooled(B, 4, I, seed=13), thr=thr, vmin=vmin, calls=2)
    assert o.hidden.sum() > 0 and o.counts.sum() > 0
    if vmin > 0:
        assert (o.calls[-1]["state"][0] != 0).any()      # IAF#0 left rest without input
    names = o.check_gpu(mode=mode, want_steps=want_steps)
    d = str(want_steps).lower()
    if thr == 1 and vmin <= 0:
        assert_ran(names, f"feature_raster_kernel<{d}>")
    else:
        assert_ran(names, "feature_kernel(")
    assert_ran(names, "output_simt_kernel" if mode == 1 else f"output_tc_kernel<false, {d}, 0, false>")


# ------------------------------------------------------------------------ the advertised size limits
@pytest.mark.parametrize("I,F", [(196, 392), (324, 200), (400, 800), (1024, 992)])
def test_size_limits(I, F):
    """Shapes up to I = 1024, F = 992 run on the CUDA-core kernels (they need more than 48 KB of shared
    memory); F = 392 is the reference's --dims 14 with its default --feature_multiplier 2."""
    from lens_b200._lib import LensError
    P, T, B = 60, 20, 3
    Wf, Wo = synth_weights(I, F, P, seed=I + F)
    Wf = tidy(Wf)
    o = Oracle(Wf, Wo, T, synth_pooled(B, 2, I, seed=14), calls=2)
    assert o.hidden.sum() > 0 and o.counts.sum() > 0
    assert_ran(o.check_gpu(mode=1, want_steps=False), "feature_kernel(", "output_simt_kernel")
    o.check_gpu(mode=0, want_steps=True)
    if F > 224:
        with pytest.raises(LensError, match="tensor-core mode unavailable"):
            o.check_gpu(mode=2, want_steps=False)
    else:
        assert_ran(o.check_gpu(mode=2, want_steps=False), "feature_kernel(", "output_tc_kernel<true, false, 7, false>")


@pytest.mark.parametrize("F", [224, 225])
def test_largest_tensor_core_shape(F):
    """F = 224 is the largest hidden layer the tensor-core output kernel takes; F = 225 must be refused in
    tensor-core mode and run everywhere else."""
    from lens_b200._lib import LensError
    I, P, T, B = 100, 300, 32, 4
    Wf, Wo = synth_weights(I, F, P, seed=F)
    Wf = tidy(Wf)
    o = Oracle(Wf, Wo, T, synth_pooled(B, 2, I, seed=15), calls=2)
    assert o.counts.sum() > 0
    assert_ran(o.check_gpu(mode=1, want_steps=False), "output_simt_kernel")
    o.check_gpu(mode=0, want_steps=False)
    if F == 224:
        assert_ran(o.check_gpu(mode=2, want_steps=False), "output_tc_kernel<true, false, 7, false>")
    else:
        with pytest.raises(LensError, match="tensor-core mode unavailable"):
            o.check_gpu(mode=2, want_steps=False)


def test_forward_float_largest_input():
    """The operator seam at I = 1024 (32 x 32 pooled pixels), F = 992."""
    from lens_b200.network import B200Network
    I, F, P, T, Bp, dims = 1024, 992, 50, 10, 2, 32
    Wf, Wo = synth_weights(I, F, P, seed=16)
    Wf = tidy(Wf)
    rng = np.random.default_rng(17)
    x = (rng.random((Bp, T, I)) < 0.03).astype(np.float32)
    onet = O.OracleSNN(Wf, Wo, None, T, n_streams=Bp)
    want = onet.forward_float(x)
    assert want.sum() > 0
    gnet = B200Network(torch.from_numpy(Wf), torch.from_numpy(Wo), roi=dims, k=1, num_timesteps=T)
    assert gnet.n_inexact == 0
    got, names = kernels_run(lambda: gnet(cuda(x.reshape(Bp * T, 1, dims, dims))))
    assert np.array_equal(got.cpu().numpy(), want.reshape(Bp * T, P))
    for a, b in zip(onet.state(), gnet.state()):
        assert np.array_equal(b.cpu().numpy(), a)
    assert_ran(names, "feature_kernel(", "output_simt_kernel")
