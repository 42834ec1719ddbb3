"""GPU parity tests: the CUDA path, called through the C ABI, against the CPU oracle.

Bar: bit-exact for binned frames, pooled pixels, hidden / output spikes, spike counts,
membrane potentials (the exact-contraction contract makes even those bit-exact), the
sequence-matched matrix and the top-N indices.  Sizes are ones the oracle finishes in
seconds; full-size configurations are covered by the property tests in test_gpu_scale.py.
"""
import numpy as np
import pytest
import torch

from conftest import synth_weights, synth_pooled
from oracle import oracle as O

pytestmark = pytest.mark.gpu


def cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


# ------------------------------------------------------------------------------- K1
def make_events(rng, n, sensor, n_win, window, hot=True):
    t = np.sort(rng.integers(0, n_win * window, n)).astype(np.uint32)
    x = rng.integers(0, sensor, n).astype(np.uint16)
    y = rng.integers(0, sensor, n).astype(np.uint16)
    if hot:   # a few hot pixels at a very high rate: exercises u8 wrap and atomic contention
        m = rng.random(n) < 0.3
        x[m] = rng.choice([0, 5, sensor - 1], m.sum())
        y[m] = rng.choice([0, 7, sensor - 1], m.sum())
    return t, x, y


@pytest.mark.parametrize("sensor,roi,k,x0,y0,shift,wrap", [
    (128, 80, 8, 23, 0, 1, True),     # Speck ROI of the reference
    (128, 128, 8, 0, 0, 1, True),     # config 4: no crop
    (32, 32, 1, 0, 0, 0, False),      # k = 1, saturating
    (346, 260, 10, 40, 0, 1, True),   # DAVIS346-sized frame: multi-band histogram
    (16, 7, 1, 3, 2, 1, True),        # odd roi (unaligned frame rows)
    (128, 64, 8, 0, 0, 1, True),      # power-of-two fast path with events outside the roi
    (256, 256, 16, 0, 0, 1, False),   # largest fast-path roi, saturating
])
def test_bin_events(sensor, roi, k, x0, y0, shift, wrap):
    from lens_b200 import ops
    rng = np.random.default_rng(sensor * 1000 + roi)
    n_win, window = 9, 1000
    t, x, y = make_events(rng, 60000, sensor, n_win, window)
    t[(t >= 3000) & (t < 4000)] = 4000            # window 3 is empty
    t.sort()
    fo, po, co = O.bin_events(t, x, y, 0, window, n_win, roi, k, x0, y0, shift, wrap)
    f, p, c = ops.bin_events(cuda(t.view(np.int32)), cuda(x.view(np.int16)), cuda(y.view(np.int16)),
                             0, window, n_win, roi, k, x0, y0, shift, wrap)
    assert np.array_equal(f.cpu().numpy(), fo)
    assert np.array_equal(p.cpu().numpy(), po)
    assert np.array_equal(c.cpu().numpy(), co)
    assert co[3] == 0 and not fo[3].any()                # window 3 is empty
    # some pixel saw more than 255 events in one window: wrapping and saturating frames differ there
    fs, _, _ = O.bin_events(t, x, y, 0, window, n_win, roi, k, x0, y0, shift, False)
    assert (fs != fo).any() if wrap else fo.max() == 255


def test_bin_events_edges():
    from lens_b200 import ops
    # no events at all; events before t0 and after the last window are dropped
    z32, z16 = torch.zeros(0, dtype=torch.int32).cuda(), torch.zeros(0, dtype=torch.int16).cuda()
    f, p, c = ops.bin_events(z32, z16, z16, 0, 100, 3, 8, 2)
    assert f.sum().item() == 0 and c.sum().item() == 0
    t = np.array([5, 50, 150, 151, 399, 400, 1000], dtype=np.uint32)
    x = np.array([1, 1, 2, 2, 0, 3, 3], dtype=np.uint16)
    y = np.array([1, 1, 2, 2, 0, 3, 3], dtype=np.uint16)
    fo, po, co = O.bin_events(t, x, y, 100, 100, 3, 8, 2)
    f, p, c = ops.bin_events(cuda(t.view(np.int32)), cuda(x.view(np.int16)), cuda(y.view(np.int16)),
                             100, 100, 3, 8, 2)
    assert np.array_equal(f.cpu().numpy(), fo) and np.array_equal(c.cpu().numpy(), co)
    assert co.tolist() == [2, 0, 1] and fo[2, 7, 7] == 1   # (0,0) wraps to the last row / column


def test_pool_frames():
    from lens_b200 import ops
    rng = np.random.default_rng(1)
    for roi, k in [(80, 8), (7, 1), (12, 3), (128, 8)]:
        fr = rng.integers(0, 256, (11, roi, roi)).astype(np.uint8)
        assert np.array_equal(ops.pool_frames(cuda(fr), k).cpu().numpy(), O.pool(fr, k))


# -------------------------------------------------------------------------- K2 + K3
def run_both(Wf, Wo, U, T, pooled, roi, k, mode, calls=1, want_steps=True):
    """want_steps=False runs the production kernels (the debug buffers select other instantiations):
    spike counts, membrane potentials and the overflow counter are compared; True adds every step."""
    from lens_b200.network import B200Network
    B, Q, I = pooled.shape
    onet = O.OracleSNN(Wf, Wo, U, T, n_streams=B)
    gnet = B200Network(torch.from_numpy(Wf), torch.from_numpy(Wo), roi=roi, k=k, num_timesteps=T,
                       max_streams=B, U=torch.from_numpy(U))
    assert gnet.n_inexact == 0
    res = []
    for part in np.array_split(np.arange(Q), calls):
        if want_steps:
            oc, oh, oo = onet.run_streams(pooled[:, part], want_steps=True)
            gc, gh, go = gnet.run_streams(pooled=cuda(pooled[:, part]), mode=mode, want_steps=True)
            res.append((oc, oh, oo, gc.cpu().numpy(), gh.cpu().numpy(), go.cpu().numpy()))
        else:
            oc = onet.run_streams(pooled[:, part])
            gc = gnet.run_streams(pooled=cuda(pooled[:, part]), mode=mode)
            res.append((oc, None, None, gc.cpu().numpy(), None, None))
    ov = onet.state()
    gv = [v.cpu().numpy() for v in gnet.state()]
    assert gnet.overflow() == onet.overflow()
    return res, ov, gv


# (mode, want_steps): the per-step debug buffers select other instantiations of the kernels than a production
# run does (with want_steps=False the tensor-core kernels take their fast scans), so both are compared
SNN_MODES = [pytest.param(1, True, id="1"), pytest.param(2, True, id="2"),
             pytest.param(1, False, id="1-production"), pytest.param(2, False, id="2-production")]


def assert_same(res, ov, gv):
    for oc, oh, oo, gc, gh, go in res:
        if oh is not None:
            assert np.array_equal(gh, oh), "hidden spikes differ"
            assert np.array_equal(go, oo), "output spikes differ"
        assert np.array_equal(gc, oc), "spike counts differ"
    for a, b in zip(ov, gv):
        assert np.array_equal(a, b), "membrane potentials differ"


@pytest.mark.parametrize("mode,want_steps", SNN_MODES)
def test_snn_config1_golden(golden, mode, want_steps):
    """Bundled model + data: GPU == oracle bit for bit, and == the reference's own output."""
    g = golden("config1")
    roi, dims, T = int(g["roi_dim"]), int(g["dims"]), int(g["timebin"])
    k = roi // dims
    U = O.raster_uniforms(T, roi, k)
    pooled = O.pool(g["frames"], k)[None]
    res, ov, gv = run_both(g["W_feat"], g["W_out"], U, T, pooled, roi, k, mode, want_steps=want_steps)
    assert_same(res, ov, gv)
    assert np.array_equal(res[0][3][0], g["S"].astype(np.float32))   # reference similarity matrix
    assert np.abs(gv[2][0] - g["v2"]).max() < 1e-5 and np.abs(gv[1][0] - g["v1"]).max() < 1e-5


@pytest.mark.parametrize("mode,want_steps", SNN_MODES)
def test_snn_brisevent_golden_prefix(golden, mode, want_steps):
    """Second bundled model (k = 1, P = 641, multi-spike outputs): first 60 queries."""
    g = golden("brisevent")
    roi, dims, T = int(g["roi_dim"]), int(g["dims"]), int(g["timebin"])
    k = roi // dims
    U = O.raster_uniforms(T, roi, k)
    pooled = O.pool(g["frames"][:60], k)[None]
    res, ov, gv = run_both(g["W_feat"], g["W_out"], U, T, pooled, roi, k, mode, want_steps=want_steps)
    assert_same(res, ov, gv)
    S = g["S"][:60].astype(np.float32)
    assert (res[0][3][0] != S).sum() <= 2


@pytest.mark.parametrize("I_dims,F,P,T,B,Q,calls", [
    (10, 200, 100, 250, 3, 2, 1),     # LENS default sizes, three streams
    (10, 200, 1000, 50, 4, 3, 3),     # config-2 places, state carried across three calls
    (7, 63, 641, 20, 2, 4, 2),        # brisevent sizes
    (4, 40, 130, 33, 5, 2, 1),        # ragged: P not a multiple of the place tile, T odd
    (3, 9, 5, 7, 1, 1, 1),            # tiny
])
@pytest.mark.parametrize("mode,want_steps", SNN_MODES)
def test_snn_synthetic(I_dims, F, P, T, B, Q, calls, mode, want_steps):
    I = I_dims * I_dims
    Wf, Wo = synth_weights(I, F, P, seed=F + P)
    k = 2
    roi = I_dims * k
    U = O.raster_uniforms(T, roi, k)
    pooled = synth_pooled(B, Q, I, seed=B * 7 + Q)
    pooled[0, 0, :] = 255          # saturated frame: every input fires every step
    if B > 1:
        pooled[1, :, :] = 0        # empty frames
    res, ov, gv = run_both(Wf, Wo, U, T, pooled, roi, k, mode, calls=calls, want_steps=want_steps)
    assert_same(res, ov, gv)


def test_snn_float_seam_matches_oracle(golden):
    """`net(x)` with x f32 [T*B', 1, roi, roi] (lens/run_model.py:238), incl. non-binary input."""
    from lens_b200.network import B200Network
    g = golden("config1")
    roi, T, k = 80, 20, 8
    rng = np.random.default_rng(9)
    Bp = 2
    x = (rng.random((Bp * T, 1, roi, roi)) < 0.05).astype(np.float32)
    x[:, :, 3::8, 3::8] *= rng.choice([0.0, 0.5, 1.0, 2.5], (Bp * T, 1, 10, 10)).astype(np.float32)
    gnet = B200Network(torch.from_numpy(g["W_feat"]), torch.from_numpy(g["W_out"]), roi=roi, k=k,
                       num_timesteps=T)
    onet = O.OracleSNN(g["W_feat"], g["W_out"], None, T, n_streams=Bp)
    xp = x[:, 0, 3::8, 3::8].reshape(Bp, T, 100)
    for _ in range(2):   # second call continues from the carried-over state
        got = gnet(cuda(x)).cpu().numpy()
        want = onet.forward_float(xp).reshape(Bp * T, -1)
        assert np.array_equal(got, want)
    gnet.reset_states()
    onet.reset_states()
    assert np.array_equal(gnet(cuda(x)).cpu().numpy(), onet.forward_float(xp).reshape(Bp * T, -1))


def test_inexact_weights_are_reported():
    from lens_b200.network import B200Network
    Wf, Wo = synth_weights(4, 8, 6, seed=1)
    Wo[0, 0] = 1.0
    Wo[0, 1] = 2.0 ** -60        # 60 bits below the row maximum: cannot be exact
    net = B200Network(torch.from_numpy(Wf), torch.from_numpy(Wo), roi=2, k=1, num_timesteps=4)
    assert net.n_inexact == 1


# ------------------------------------------------------------------------------- K4
@pytest.mark.parametrize("B,Q,P,L,N", [
    (1, 100, 100, 2, 25), (3, 16, 1000, 2, 25), (2, 10, 3000, 10, 25), (2, 5, 12, 4, 25),
    (1, 7, 9, 1, 5), (1, 4, 5000, 3, 64),
])
def test_seqmatch_topk(B, Q, P, L, N):
    from lens_b200 import ops
    rng = np.random.default_rng(B + Q + P + L)
    S = rng.poisson(1.3, (B, Q, P)).astype(np.float32)      # spike counts: many ties
    tv, ti, D = ops.seqmatch_topk(cuda(S), L, N, want_D=True)
    tv, ti, D = tv.cpu().numpy(), ti.cpu().numpy(), D.cpu().numpy()
    for b in range(B):
        Do = O.seqmatch(S[b], L)
        io, vo = O.topk(Do, N)
        assert np.array_equal(D[b], Do)
        assert np.array_equal(ti[b], io)
        assert np.array_equal(tv[b], vo)


def test_recall_dense_and_band(golden):
    from lens_b200 import ops
    g = golden("config1")
    D, GT = g["D"], g["GTtol"]
    S = g["S"].astype(np.float32)[None]
    tv, ti, Dg = ops.seqmatch_topk(cuda(S), int(g["sequence_length"]), 25, want_D=True)
    assert np.array_equal(Dg[0].cpu().numpy(), D)
    hits, nv = ops.recall_counts(ti, D.shape[0], gt_dense=cuda(GT.astype(np.uint8)))
    hits, nv = hits.cpu().numpy(), int(nv.item())
    for i, n in enumerate(ops.RECALL_NS):
        want = O.recall_at_k(D, GT, K=n, kind="stable")
        assert abs(hits[i] / nv - want) < 1e-12
        lo, hi = O.recall_bounds(D, GT, n)
        assert lo - 1e-12 <= hits[i] / nv <= hi + 1e-12
    # band ground truth == the equivalent dense matrix
    Po, Qo = D.shape
    centre = np.arange(Qo, dtype=np.int32)[None]
    centre[0, 5] = -1
    dense = (np.abs(np.arange(Po)[:, None] - centre[0][None, :]) <= 2).astype(np.uint8)
    dense[:, 5] = 0
    h1, n1 = ops.recall_counts(ti, Po, gt_dense=cuda(dense))
    h2, n2 = ops.recall_counts(ti, Po, gt_center=cuda(centre), gt_tol=2)
    assert torch.equal(h1, h2) and torch.equal(n1, n2) and int(n1.item()) == Qo - 1
