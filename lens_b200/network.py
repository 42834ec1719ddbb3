"""B200Network: the object that stands where `self.sinabs_model` stands.

Reference seam: lens/run_model.py:151-156 builds `sinabs.from_model(Sequential(conv,
ReLU, Flatten, feature_layer.w, ReLU, output_layer.w), input_shape=(1, roi, roi),
num_timesteps=T, add_spiking_output=True)` and :238 calls it as
`net(x: f32[T*B', 1, roi, roi]) -> f32[T*B', P]`, stateful across calls.  This class
keeps that call signature (`__call__`, `reset_states`) and adds the batched fast path
`run_streams` that `LENS.evaluate` uses instead of the per-query python loop.
"""
import ctypes as C

import torch

from . import _lib
from ._lib import check, ptr, stream_ptr, require_cuda, LensError
from .ops import pool_geometry, pool_frames

MODE_AUTO, MODE_SIMT, MODE_TC = 0, 1, 2
MAX_SPIKES_PER_STEP = 127     # LENS_MAX_SPIKE: hidden spikes travel as int8 (sinabs' MultiSpike is unbounded)


def _on_device(fn):
    """Run a method with the network's device current, so the handle's launches, allocations and the
    stream passed to the C ABI belong to that device whatever the caller's current device is."""
    import functools

    @functools.wraps(fn)
    def wrapped(self, *a, **kw):
        with torch.cuda.device(self.device):
            return fn(self, *a, **kw)
    return wrapped


def raster_uniforms(T, roi, k, device):
    """U[T, I]: the columns of the reference's seed-50 `torch.rand(T, roi*roi)` that survive pooling.

    lens/src/dataset.py:120-121 re-seeds torch's CPU generator with 50 for EVERY image, so one
    matrix serves all queries; only the pixels the one-hot conv keeps (run_model.py:130-137) matter.
    Drawing from torch's CPU MT19937 stream is the definition of these numbers (host plumbing).
    """
    g = torch.Generator(device="cpu")
    g.manual_seed(50)
    U = torch.rand(T, roi * roi, generator=g)
    dims, c = pool_geometry(roi, k)
    ii = k * torch.arange(dims) + c
    cols = (ii[:, None] * roi + ii[None, :]).reshape(-1)
    return U[:, cols].contiguous().to(device)


class B200Network:
    """IAF -> Linear(I->F) -> IAF -> Linear(F->P) -> IAF on hand-written sm_100a kernels."""

    def __init__(self, W_feat, W_out, roi, k, num_timesteps, spike_threshold=1.0, min_v_mem=-1.0,
                 max_streams=1, device=None, U=None):
        if not torch.cuda.is_available():
            raise LensError("B200Network needs a CUDA device; there is no CPU fallback")
        self.device = torch.device(device if device is not None else "cuda")
        if self.device.type != "cuda":
            raise LensError(f"B200Network lives on a CUDA device, not on '{self.device}'")
        self.roi, self.k, self.T = int(roi), int(k), int(num_timesteps)
        self.dims, self.c = pool_geometry(self.roi, self.k)
        self.W_feat = W_feat.detach().to(self.device, torch.float32).contiguous()
        self.W_out = W_out.detach().to(self.device, torch.float32).contiguous()
        self.F, self.I = self.W_feat.shape
        self.P = self.W_out.shape[0]
        if self.I != self.dims * self.dims or self.W_out.shape[1] != self.F:
            raise LensError(f"weight shapes {tuple(W_feat.shape)} / {tuple(W_out.shape)} do not match "
                            f"dims={self.dims}")
        self.thr, self.v_min = float(spike_threshold), float(min_v_mem)
        self.U = (U.to(self.device, torch.float32).contiguous() if U is not None
                  else raster_uniforms(self.T, self.roi, self.k, self.device))
        self.max_streams = 0
        self._h = C.c_void_p()
        self.n_inexact = 0
        self.check_overflow = True     # __call__ raises when a hidden neuron exceeded MAX_SPIKES_PER_STEP
        self._create(max_streams)

    # -- handle management ---------------------------------------------------------
    def _create(self, max_streams):
        self._destroy()
        n_inexact = C.c_int64(0)
        with torch.cuda.device(self.device):
            check(_lib.lib().lens_snn_create(self.I, self.F, self.P, self.T, self.thr, self.v_min,
                                             ptr(self.W_feat), ptr(self.W_out), ptr(self.U),
                                             int(max_streams), C.byref(self._h), C.byref(n_inexact),
                                             stream_ptr()), "lens_snn_create")
        self.max_streams = int(max_streams)
        self.n_inexact = int(n_inexact.value)

    @_on_device
    def _destroy(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            _lib.lib().lens_snn_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self._destroy()
        except Exception:
            pass

    def _ensure_streams(self, B):
        # sinabs re-creates (zeroes) its state when the batch shape changes
        if B != self.max_streams:
            self._create(B)

    # -- sinabs-compatible surface ---------------------------------------------------
    @_on_device
    def reset_states(self):
        check(_lib.lib().lens_snn_reset(self._h, stream_ptr()), "lens_snn_reset")

    @_on_device
    def reset_streams(self, mask):
        """reset_states() for the streams with mask[b] != 0 only (mask u8 / bool [max_streams] on the device);
        the other streams' state and the overflow counter are untouched."""
        require_cuda(mask)
        if mask.dtype not in (torch.uint8, torch.bool) or mask.shape != (self.max_streams,):
            raise LensError(f"mask must be u8 / bool [{self.max_streams}], got {mask.dtype} {tuple(mask.shape)}")
        check(_lib.lib().lens_snn_reset_streams(self._h, ptr(mask), stream_ptr()), "lens_snn_reset_streams")

    def eval(self):
        return self

    def to(self, device):
        if torch.device(device).type != "cuda":
            raise LensError("B200Network lives on a CUDA device")
        return self

    @_on_device
    def __call__(self, x):
        """x f32 [T*B', 1, roi, roi] -> output spikes f32 [T*B', P] (lens/run_model.py:238)."""
        require_cuda(x)
        if x.dim() != 4 or x.shape[1] != 1 or x.shape[2] != self.roi or x.shape[3] != self.roi:
            raise LensError(f"expected [T*B, 1, {self.roi}, {self.roi}], got {tuple(x.shape)}")
        n = x.shape[0]
        if n % self.T != 0:
            raise LensError(f"leading dimension {n} is not a multiple of num_timesteps={self.T}")
        Bp = n // self.T
        self._ensure_streams(Bp)
        # the one-hot strided conv keeps pixel (k*i+c, k*j+c): a strided view, made contiguous
        xp = x[:, 0, self.c::self.k, self.c::self.k][:, :self.dims, :self.dims]
        xp = xp.reshape(Bp, self.T, self.I).to(torch.float32).contiguous()
        out = torch.empty((Bp, self.T, self.P), dtype=torch.float32, device=x.device)
        check(_lib.lib().lens_snn_forward_float(self._h, ptr(xp), Bp, self.T, ptr(out), stream_ptr()),
              "lens_snn_forward_float")
        if self.check_overflow:
            self.raise_on_overflow()
        return out.reshape(n, self.P)

    forward = __call__

    # -- batched fast path -------------------------------------------------------------
    @_on_device
    def run_streams(self, frames=None, pooled=None, mode=MODE_AUTO, want_steps=False):
        """Spike-count rows for B independent streams of Q queries.

        frames u8 [B, Q, roi, roi] or pooled u8 [B, Q, I] -> counts f32 [B, Q, P]
        (the rows lens/run_model.py:239-246 stacks into the similarity matrix).  State
        carries over from previous calls, as in the reference.
        """
        if (frames is None) == (pooled is None):
            raise LensError("give exactly one of frames / pooled")
        if pooled is None:
            require_cuda(frames)
            B, Q = frames.shape[:2]
            pooled = pool_frames(frames.reshape(B * Q, self.roi, self.roi), self.k).reshape(B, Q, self.I)
        require_cuda(pooled)
        if pooled.dtype != torch.uint8 or pooled.dim() != 3 or pooled.shape[2] != self.I:
            raise LensError(f"pooled must be u8 [B, Q, {self.I}]")
        B, Q, _ = pooled.shape
        self._ensure_streams(B)
        dev = pooled.device
        counts = torch.empty((B, Q, self.P), dtype=torch.float32, device=dev)
        hid = torch.empty((B, Q * self.T, self.F), dtype=torch.uint8, device=dev) if want_steps else None
        out = torch.empty((B, Q * self.T, self.P), dtype=torch.uint8, device=dev) if want_steps else None
        check(_lib.lib().lens_snn_forward(self._h, ptr(pooled), B, Q, ptr(counts), ptr(hid), ptr(out),
                                          int(mode), stream_ptr()), "lens_snn_forward")
        return (counts, hid, out) if want_steps else counts

    @_on_device
    def run_streams_range(self, pooled, b0, counts, mode=MODE_AUTO):
        """Streams [b0, b0 + nb) only: pooled u8 [nb, Q, I] -> counts f32 [nb, Q, P] (pre-allocated).

        Used to overlap the host->device copy of one group of streams with the compute of another;
        the handle must already be sized for all streams (`ensure_streams`)."""
        require_cuda(pooled, counts)
        nb, Q, _ = pooled.shape
        check(_lib.lib().lens_snn_forward_range(self._h, ptr(pooled), int(b0), int(nb), int(Q), ptr(counts),
                                                None, None, int(mode), stream_ptr()), "lens_snn_forward_range")
        return counts

    @_on_device
    def run_streams_ids(self, pooled, ids, mode=MODE_AUTO):
        """`run_streams` for the streams ids of the handle only, in any order: pooled u8 [n, Q, I] -> counts f32
        [n, Q, P], row i = stream ids[i] (i32 [n] on the device, distinct, in [0, max_streams)).  Each of them
        advances from its own state; every other stream's state is untouched, and the handle is never resized."""
        require_cuda(pooled, ids)
        if pooled.dtype != torch.uint8 or pooled.dim() != 3 or pooled.shape[2] != self.I:
            raise LensError(f"pooled must be u8 [n, Q, {self.I}]")
        n, Q, _ = pooled.shape
        if ids.dtype != torch.int32 or tuple(ids.shape) != (n,):
            raise LensError(f"ids must be i32 [{n}]")
        counts = torch.empty((n, Q, self.P), dtype=torch.float32, device=pooled.device)
        check(_lib.lib().lens_snn_forward_streams(self._h, ptr(pooled), ptr(ids), n, Q, ptr(counts), int(mode),
                                                  stream_ptr()), "lens_snn_forward_streams")
        return counts

    def ensure_streams(self, B):
        self._ensure_streams(B)

    @_on_device
    def state(self):
        """(v0 [B, I], v1 [B, F], v2 [B, P]) membrane potentials."""
        B = self.max_streams
        v0 = torch.empty((B, self.I), dtype=torch.float32, device=self.device)
        v1 = torch.empty((B, self.F), dtype=torch.float32, device=self.device)
        v2 = torch.empty((B, self.P), dtype=torch.float32, device=self.device)
        check(_lib.lib().lens_snn_get_state(self._h, ptr(v0), ptr(v1), ptr(v2), stream_ptr()),
              "lens_snn_get_state")
        return v0, v1, v2

    @_on_device
    def set_timing(self, enable=True):
        check(_lib.lib().lens_snn_set_timing(self._h, int(enable)), "lens_snn_set_timing")

    @_on_device
    def get_timing(self):
        """-> dict(feature_ms, output_ms, n_feature, n_output) accumulated since the last call."""
        f, o = C.c_float(0), C.c_float(0)
        nf, no = C.c_int64(0), C.c_int64(0)
        check(_lib.lib().lens_snn_get_timing(self._h, C.byref(f), C.byref(o), C.byref(nf), C.byref(no)),
              "lens_snn_get_timing")
        return dict(feature_ms=f.value, output_ms=o.value, n_feature=nf.value, n_output=no.value)

    @_on_device
    def overflow_tensor(self):
        """The overflow counter as a device tensor i64 [1] (stream-ordered copy, no synchronisation)."""
        o = torch.zeros((1,), dtype=torch.int64, device=self.device)
        check(_lib.lib().lens_snn_get_overflow(self._h, ptr(o), stream_ptr()), "lens_snn_get_overflow")
        return o

    @_on_device
    def overflow(self):
        """Hidden-neuron steps whose spike count exceeded MAX_SPIKES_PER_STEP since the last reset
        (clipped there; the reference's MultiSpike is unbounded, so a non-zero value means the spike
        counts of this run are not the reference's).  Synchronises."""
        o = torch.zeros((1,), dtype=torch.int64, device=self.device)
        check(_lib.lib().lens_snn_get_overflow(self._h, ptr(o), stream_ptr()), "lens_snn_get_overflow")
        return int(o.item())

    def raise_on_overflow(self):
        n = self.overflow()
        if n:
            raise LensError(f"{n} hidden-neuron steps fired more than {MAX_SPIKES_PER_STEP} spikes in one "
                            "timestep and were clipped (int8 spike transport): results would differ from the "
                            "reference; call reset_states() and rescale the input")
