"""Seeded synthetic workloads of the shapes BASELINE.json names (SURVEY.md 8d).

No datasets or checkpoints are reachable from the GPU box, so benchmarks and scale tests use
random weights with the statistics of the trained LENS models and random count frames / event
streams with the statistics of the bundled Speck recordings.  The small generators run on the
host with numpy (deterministic per seed) and the caller moves their output to the device; the
*_device ones draw full-size workloads on the GPU.
"""
import numpy as np


def weights(I, F, P, seed=1):
    """W_feat [F, I], W_out [P, F] f32 mimicking trained statistics.

    W_feat: ~30 % positive (mean +0.147), ~53 % negative (mean -0.089), ~17 % zero, clipped to
    [-4.7, 1.05]; W_out: dense N(0, 0.0143) clipped to [-0.11, 0.055] with |w| >= 1e-6 (the trainer's
    clamp, lens/src/blitnet.py:234-235 of the reference).
    """
    rng = np.random.default_rng(seed)
    kind = rng.random((F, I))
    Wf = np.where(kind < 0.30, rng.exponential(0.147, (F, I)),
                  np.where(kind < 0.83, -rng.exponential(0.089, (F, I)), 0.0))
    Wf = np.clip(Wf, -4.7, 1.05).astype(np.float32)
    Wo = np.clip(rng.normal(0.0, 0.0143, (P, F)), -0.11, 0.055)
    Wo = np.where(np.abs(Wo) < 1e-6, 1e-6, Wo).astype(np.float32)
    return Wf, Wo


def pixel_counts(shape, seed=2):
    """u8 event counts per pixel: geometric with mean ~8, ~43 % zeros, wrapped modulo 256."""
    rng = np.random.default_rng(seed)
    v = rng.geometric(1.0 / 15.0, shape) - 1
    v = np.where(rng.random(shape) < 0.40, 0, v)
    return (v % 256).astype(np.uint8)


def frames(B, Q, roi=80, seed=2):
    """Count frames u8 [B, Q, roi, roi] of 'Speck resolution' (80x80 ROI of the 128x128 sensor)."""
    return pixel_counts((B, Q, roi, roi), seed)


def events(n_events, sensor=128, window_us=250_000, events_per_window=131_072, seed=5,
           hot_pixels=16, hot_rate=100.0):
    """SoA DVS stream (t_us u32 sorted, x u16, y u16) with hot pixels (SURVEY.md 8d, config 4).

    Uniform inter-arrival times (mean window_us / events_per_window); x, y uniform over the sensor
    except `hot_pixels` pixels that fire `hot_rate` times more often than the rest.
    """
    rng = np.random.default_rng(seed)
    n_win = int(np.ceil(n_events / events_per_window))
    t = np.sort(rng.integers(0, n_win * window_us, n_events, dtype=np.int64)).astype(np.uint32)
    x = rng.integers(0, sensor, n_events).astype(np.uint16)
    y = rng.integers(0, sensor, n_events).astype(np.uint16)
    if hot_pixels:
        p_hot = hot_pixels * hot_rate / (sensor * sensor + hot_pixels * (hot_rate - 1))
        m = rng.random(n_events) < p_hot
        hx = rng.integers(0, sensor, hot_pixels).astype(np.uint16)
        hy = rng.integers(0, sensor, hot_pixels).astype(np.uint16)
        pick = rng.integers(0, hot_pixels, int(m.sum()))
        x[m] = hx[pick]
        y[m] = hy[pick]
    return t, x, y, n_win


def gt_centers(B, Qo, Po, seed=7):
    """Synthetic ground truth: query q of stream b shows place (offset_b + q) (i32 [B, Qo])."""
    rng = np.random.default_rng(seed)
    off = rng.integers(0, max(1, Po - Qo + 1), B)
    return (off[:, None] + np.arange(Qo)[None, :]).astype(np.int32)


# ---- device-side generators for the full-size configurations (host numpy would take minutes) ----------
def frames_device(B, Q, roi=80, seed=2, device="cuda", chunk_streams=2048):
    """Count frames u8 [B, Q, roi, roi] with the statistics of `pixel_counts`, drawn on the device
    (torch CUDA generator, deterministic per seed and device type) in chunks of streams."""
    import torch
    g = torch.Generator(device=device).manual_seed(int(seed))
    out = torch.empty((B, Q, roi, roi), dtype=torch.uint8, device=device)
    for b0 in range(0, B, chunk_streams):
        n = min(chunk_streams, B - b0)
        shape = (n, Q, roi, roi)
        v = torch.empty(shape, dtype=torch.float32, device=device).geometric_(1.0 / 15.0, generator=g) - 1.0
        zero = torch.rand(shape, device=device, generator=g) < 0.40
        v = torch.where(zero, torch.zeros_like(v), v)
        out[b0:b0 + n] = v.to(torch.int32).remainder_(256).to(torch.uint8)
    return out


def events_device(n_events, sensor=128, window_us=250_000, events_per_window=131_072, seed=5,
                  hot_pixels=16, hot_rate=100.0, device="cuda", chunk_windows=512):
    """The event stream of `events` drawn on the device: (t_us i32 sorted, x i16, y i16, n_windows).

    Timestamps are uniform inside consecutive spans of `chunk_windows` windows (sorted per span), so
    every window holds events_per_window events on average; x, y uniform with `hot_pixels` pixels
    firing `hot_rate` times more often."""
    import torch
    g = torch.Generator(device=device).manual_seed(int(seed))
    n_win = -(-n_events // events_per_window)
    t = torch.empty(n_events, dtype=torch.int32, device=device)
    per_chunk = chunk_windows * events_per_window
    for c0 in range(0, n_events, per_chunk):
        n = min(per_chunk, n_events - c0)
        wins = -(-n // events_per_window)
        base = (c0 // events_per_window) * window_us
        tt = torch.randint(0, wins * window_us, (n,), dtype=torch.int32, device=device, generator=g)
        t[c0:c0 + n] = torch.sort(tt).values + base
    assert n_win * window_us < 2 ** 31
    x, y = _pixels_device(n_events, sensor, hot_pixels, hot_rate, g, device)
    return t, x, y, int(n_win)


def _pixels_device(n_events, sensor, hot_pixels, hot_rate, g, device):
    """x, y i16 [n_events] uniform over the sensor, `hot_pixels` pixels firing `hot_rate` times more often."""
    import torch
    x = torch.randint(0, sensor, (n_events,), dtype=torch.int16, device=device, generator=g)
    y = torch.randint(0, sensor, (n_events,), dtype=torch.int16, device=device, generator=g)
    if hot_pixels:
        p_hot = hot_pixels * hot_rate / (sensor * sensor + hot_pixels * (hot_rate - 1))
        hx = torch.randint(0, sensor, (hot_pixels,), dtype=torch.int16, device=device, generator=g)
        hy = torch.randint(0, sensor, (hot_pixels,), dtype=torch.int16, device=device, generator=g)
        step = 1 << 26
        for c0 in range(0, n_events, step):
            n = min(step, n_events - c0)
            m = torch.rand(n, device=device, generator=g) < p_hot
            pick = torch.randint(0, hot_pixels, (n,), device=device, generator=g)
            x[c0:c0 + n] = torch.where(m, hx[pick], x[c0:c0 + n])
            y[c0:c0 + n] = torch.where(m, hy[pick], y[c0:c0 + n])
    return x, y


def event_streams_device(B, Q, window_us=250_000, events_per_window=131_072, sensor=128, seed=11, hot_pixels=16,
                         hot_rate=100.0, device="cuda", chunk_events=1 << 26):
    """B independent DVS streams of Q windows each (the query streams of BASELINE configs 2 and 3), drawn
    on the device: (t_us i32, x i16, y i16, offsets i64 [B + 1], t0_us i32 [B]); stream b is events
    [offsets[b], offsets[b+1]), its window q is [t0_us[b] + q * window_us, + window_us).

    Timestamps are relative to each stream (all below 2^31) and ascending within it.  t0_us[b] is uniform in
    [window_us / 4, window_us); fewer than 64 events per stream fall before it.  Window q holds
    events_per_window +- 1/16 events at uniform times, so stream and window starts fall anywhere relative to
    16-byte boundaries.  x, y as in `events_device`: at the default density 8 events per sensor pixel and
    window, the mean count of `frames`.  Deterministic per seed and device type."""
    import torch
    assert (Q + 1) * window_us < 2 ** 31
    g = torch.Generator(device=device).manual_seed(int(seed))
    i64 = dict(dtype=torch.int64, device=device)
    t0 = torch.randint(window_us // 4, window_us, (B,), generator=g, **i64)
    jit = events_per_window // 16
    counts = torch.randint(events_per_window - jit, events_per_window + jit + 1, (B, Q), generator=g, **i64)
    pre = torch.randint(0, 64, (B, 1), generator=g, **i64)
    seg_len = torch.cat([pre, counts], 1)                         # [B, Q + 1]: before t0, then the Q windows
    seg_t0 = torch.cat([torch.zeros((B, 1), **i64), t0[:, None] + window_us * torch.arange(Q, **i64)], 1)
    seg_span = torch.cat([t0[:, None], torch.full((B, Q), window_us, **i64)], 1)
    offsets = torch.zeros(B + 1, **i64)
    offsets[1:] = torch.cumsum(seg_len.sum(1), 0)
    n = int(offsets[-1])
    t = torch.empty(n, dtype=torch.int32, device=device)
    bits = int(window_us).bit_length()
    off_host = offsets.cpu()
    b0 = 0
    while b0 < B:                                                 # whole streams, about chunk_events at a time
        b1 = int(torch.searchsorted(off_host, off_host[b0] + chunk_events, right=True)) - 1
        b1 = min(max(b1, b0 + 1), B)
        lens = seg_len[b0:b1].reshape(-1)
        seg = torch.repeat_interleave(torch.arange(lens.numel(), **i64), lens)
        span = seg_span[b0:b1].reshape(-1)[seg]
        local = torch.minimum((torch.rand(seg.numel(), device=device, generator=g, dtype=torch.float64)
                               * span).to(torch.int64), span - 1)
        del span
        key = torch.sort((seg << bits) | local).values            # sorted inside each segment
        seg = key >> bits
        t[int(off_host[b0]):int(off_host[b1])] = (seg_t0[b0:b1].reshape(-1)[seg] + (key & ((1 << bits) - 1))).to(torch.int32)
        del seg, local, key
        b0 = b1
    x, y = _pixels_device(n, sensor, hot_pixels, hot_rate, g, device)
    return t, x, y, offsets, t0.to(torch.int32)
