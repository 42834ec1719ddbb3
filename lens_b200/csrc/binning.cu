// K1: DVS event stream -> count frames (+ pooled pixels).
//
// Replaces lens/collect_data.py:186-202 (per-event `frame[y-1, x-1] += 1` on an
// int64 tensor, `.astype(np.uint8)`) and the one-hot strided pooling conv of
// lens/run_model.py:130-137.  HBM-bound integer work: the event arrays are read
// exactly once with 16-byte loads, one CTA owns one (window, row-band) and keeps
// that band's histogram private in shared memory, so there are no global atomics
// and every output byte is written once.
//
// Layout: events SoA (t_us u32 | x u16 | y u16), sorted by time.  Because of the
// ordering a window is a contiguous index range; a first tiny kernel finds the
// range boundaries by binary search on t_us (one thread per boundary), after which
// the time array is never touched again.
//
// Many streams in one call (lens_bin_event_streams): stream b owns the index range
// [offsets[b], offsets[b+1]) and its own t0_us[b]; its Q windows are windows
// b*Q .. b*Q+Q-1 of the grid.  The boundaries are stored per stream, Q + 1 of them
// ([B][Q + 1]), so window w reads its range at win_offsets[w + w / Q] and the entry
// after it.  A single stream (lens_bin_events) is the case B = 1, Q = n_win,
// offsets = {0, n_events}.
#include "common.cuh"

#include <algorithm>

namespace lens {

// grid covers B * (Q + 1) boundaries.  offsets == nullptr means one stream [0, n_events) starting at t0_us;
// otherwise stream b searches [offsets[b], offsets[b+1]] clamped into [0, n_events] from t0s[b], so every
// boundary lies inside the event arrays whatever offsets holds.
__global__ void window_offsets_kernel(const uint32_t *__restrict__ t_us, int64_t n_events,
                                      const int64_t *__restrict__ offsets, const uint32_t *__restrict__ t0s,
                                      uint32_t t0_us, uint32_t window_us, int B, int64_t Q,
                                      int64_t *__restrict__ win_offsets)
{
    const int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (j >= (int64_t)B * (Q + 1)) return;
    const int64_t b = j / (Q + 1), w = j - b * (Q + 1);
    int64_t lo = 0, hi = n_events;                               // lower_bound(t >= bound) in [lo, hi)
    if (offsets) {
        lo = min(max(offsets[b], (int64_t)0), n_events);
        hi = min(max(offsets[b + 1], lo), n_events);
        t0_us = t0s[b];
    }
    uint64_t bound = (uint64_t)t0_us + (uint64_t)w * window_us;  // first t of window w
    while (lo < hi) {
        int64_t mid = (lo + hi) >> 1;
        if ((uint64_t)__ldg(t_us + mid) < bound) lo = mid + 1;
        else hi = mid;
    }
    win_offsets[j] = lo;
}

// Is the pair (j - 1, j) inside one stream?  `off` [B + 1] need not be valid: every read stays in [0, B].
__device__ __forceinline__ bool inside_one_stream(const int64_t *__restrict__ off, int B, int64_t j)
{
    int lo = 0, hi = B + 1;                      // first s with off[s] > j
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (__ldg(off + mid) <= j) lo = mid + 1;
        else hi = mid;
    }
    const int s = lo - 1;                        // the stream whose range starts at or before j
    return s >= 0 && s < B && __ldg(off + s) < j && j < __ldg(off + s + 1);
}

// Precondition check of lens_bin_events: the window ranges come from a binary search on t_us, which is
// only meaningful for ascending timestamps.  16-byte loads, grid-stride; *unsorted is set to 1 on a descent.
// kStreams (lens_check_sorted_segments_u32): a descent counts only inside one of the B streams of `off`,
// and the offsets themselves must be non-decreasing inside [0, n].  Descents are rare in valid input, so
// the per-descent binary search over the stream starts costs nothing on the streaming loop.
template <bool kStreams>
__global__ void __launch_bounds__(256) sorted_check_u32_kernel(const uint32_t *__restrict__ t, int64_t n,
                                                               const int64_t *__restrict__ off, int B,
                                                               int *__restrict__ unsorted)
{
    const int64_t n4 = n >> 2;
    bool bad = false;
    auto desc = [&](bool d, int64_t j) {         // t[j] < t[j - 1]
        if constexpr (kStreams) { if (d) bad |= inside_one_stream(off, B, j); }
        else bad |= d;
    };
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
        const uint4 v = __ldg(reinterpret_cast<const uint4 *>(t) + i);
        if constexpr (kStreams) {
            desc(v.y < v.x, 4 * i + 1);
            desc(v.z < v.y, 4 * i + 2);
            desc(v.w < v.z, 4 * i + 3);
        } else {
            bad |= v.y < v.x || v.z < v.y || v.w < v.z;
        }
        if (4 * i + 4 < n) desc(__ldg(t + 4 * i + 4) < v.w, 4 * i + 4);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0)
        for (int64_t i = n4 << 2; i + 1 < n; ++i) desc(t[i + 1] < t[i], i + 1);
    if constexpr (kStreams)
        for (int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; s <= B; s += (int64_t)gridDim.x * blockDim.x) {
            const int64_t o = __ldg(off + s);
            bad |= (s == 0 && o < 0) || (s == B && o > n) || (s < B && o > __ldg(off + s + 1));
        }
    if (bad) *unsorted = 1;
}

struct BinParams {
    const uint16_t *x, *y;
    const int64_t *win_offsets;   // [B][Q + 1]
    int Q;                        // windows per stream
    int roi_x0, roi_y0, roi, k, dims, c, index_shift, wrap_u8;
    int band_rows, n_bands;
    uint8_t *frames, *pooled;
    int32_t *win_events;
};

// The reference's (y - shift, x - shift) indexing of a roi x roi tensor (collect_data.py:193-197) after
// the crop offset: every index the reference accepts, i.e. [-roi, roi - 1] with python wrap-around for the
// negative ones (x == roi lands in column roi - 1 for shift 1), is binned; anything else is cropped
// (the reference would raise IndexError).  `kept` counts the binned events (all bands see the same
// events, band 0 reports the count).
__device__ __forceinline__ void bin_one(const BinParams &p, uint32_t *hist, int row0, int row1,
                                        int xe, int ye, int &kept)
{
    int col = xe - p.roi_x0 - p.index_shift, row = ye - p.roi_y0 - p.index_shift;
    if (col < -p.roi || col >= p.roi || row < -p.roi || row >= p.roi) return;
    ++kept;
    col += (col < 0) ? p.roi : 0;   // python negative index: -1 -> last
    row += (row < 0) ? p.roi : 0;
    if (row < row0 || row >= row1) return;
    atomicAdd(&hist[(row - row0) * p.roi + col], 1u);
}

// grid = (n_win, n_bands); dynamic smem = band_rows * roi * 4 bytes.
__global__ void __launch_bounds__(512) bin_kernel(BinParams p)
{
    extern __shared__ uint32_t hist[];
    __shared__ int s_kept;
    const int64_t w = blockIdx.x;
    const int band = blockIdx.y;
    const int row0 = band * p.band_rows;
    const int row1 = min(p.roi, row0 + p.band_rows);
    const int nbins = (row1 - row0) * p.roi;
    for (int i = threadIdx.x; i < nbins; i += blockDim.x) hist[i] = 0u;
    if (threadIdx.x == 0) s_kept = 0;
    __syncthreads();

    const int64_t *wo = p.win_offsets + w + (int)w / p.Q;   // stream b's boundaries start at b * (Q + 1)
    const int64_t e0 = wo[0], e1 = wo[1];
    // head (unaligned) | body (8 events = 16 B of x and of y per thread-iteration) | tail
    int64_t a0 = (e0 + 7) & ~(int64_t)7;
    if (a0 > e1) a0 = e1;
    int64_t a1 = a0 + ((e1 - a0) & ~(int64_t)7);
    int kept = 0;
    for (int64_t e = e0 + threadIdx.x; e < a0; e += blockDim.x) {
        bin_one(p, hist, row0, row1, p.x[e], p.y[e], kept);
    }
    const uint4 *x8 = reinterpret_cast<const uint4 *>(p.x + a0);
    const uint4 *y8 = reinterpret_cast<const uint4 *>(p.y + a0);
    const int64_t n8 = (a1 - a0) >> 3;
    for (int64_t j = threadIdx.x; j < n8; j += blockDim.x) {
        uint4 xv = __ldg(x8 + j), yv = __ldg(y8 + j);
        uint32_t xs[4] = {xv.x, xv.y, xv.z, xv.w}, ys[4] = {yv.x, yv.y, yv.z, yv.w};
#pragma unroll
        for (int h = 0; h < 4; ++h) {
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                int xe = (xs[h] >> (16 * half)) & 0xffff, ye = (ys[h] >> (16 * half)) & 0xffff;
                bin_one(p, hist, row0, row1, xe, ye, kept);
            }
        }
    }
    for (int64_t e = a1 + threadIdx.x; e < e1; e += blockDim.x) {
        bin_one(p, hist, row0, row1, p.x[e], p.y[e], kept);
    }
    if (p.win_events && band == 0) {
        // warp reduce then one shared atomic per warp
        for (int o = 16; o > 0; o >>= 1) kept += __shfl_xor_sync(0xffffffffu, kept, o);
        if ((threadIdx.x & 31) == 0 && kept) atomicAdd(&s_kept, kept);
    }
    __syncthreads();
    if (p.win_events && band == 0 && threadIdx.x == 0) p.win_events[w] = s_kept;

    // write the band of the frame, 4 pixels (one u32) per thread-iteration when roi % 4 == 0
    if (p.frames) {
        uint8_t *f = p.frames + (w * p.roi + row0) * (int64_t)p.roi;
        if ((p.roi & 3) == 0) {
            uint32_t *f4 = reinterpret_cast<uint32_t *>(f);
            for (int i = threadIdx.x; i < (nbins >> 2); i += blockDim.x) {
                uint32_t o = 0;
#pragma unroll
                for (int b = 0; b < 4; ++b) {
                    uint32_t v = hist[4 * i + b];
                    v = p.wrap_u8 ? (v & 255u) : min(v, 255u);
                    o |= v << (8 * b);
                }
                f4[i] = o;
            }
        } else {
            for (int i = threadIdx.x; i < nbins; i += blockDim.x) {
                uint32_t v = hist[i];
                f[i] = (uint8_t)(p.wrap_u8 ? (v & 255u) : min(v, 255u));
            }
        }
    }
    if (p.pooled) {  // y[i][j] = frame[k*i + c][k*j + c] for the picked rows inside this band
        const int I = p.dims * p.dims;
        for (int o = threadIdx.x; o < I; o += blockDim.x) {
            int i = o / p.dims, j = o - i * p.dims;
            int row = p.k * i + p.c, col = p.k * j + p.c;
            if (row >= row0 && row < row1) {
                uint32_t v = hist[(row - row0) * p.roi + col];
                p.pooled[w * I + o] = (uint8_t)(p.wrap_u8 ? (v & 255u) : min(v, 255u));
            }
        }
    }
}

// Fast path: roi is a power of two (<= 256), no crop offset, one band.  Two events are processed per
// 32-bit word of the x / y arrays: (c - shift) mod roi for both halves is (c + roi - shift) & (roi - 1)
// with one add and one mask, the two 16-bit bin indices come from one shift-or, and a word takes the
// per-event path only if one of its events lies outside the roi.  grid = n_win.
__global__ void __launch_bounds__(512) bin_pow2_kernel(BinParams p, int log2roi)
{
    extern __shared__ uint32_t hist[];
    __shared__ int s_kept;
    const int64_t w = blockIdx.x;
    const int roi = p.roi, nbins = roi * roi;
    for (int i = threadIdx.x; i < nbins; i += blockDim.x) hist[i] = 0u;
    if (threadIdx.x == 0) s_kept = 0;
    __syncthreads();
    const uint32_t m2 = (uint32_t)(roi - 1) * 0x00010001u;                  // per-half mask
    const uint32_t add2 = (uint32_t)(roi - p.index_shift) * 0x00010001u;   // per-half (roi - shift)
    const uint32_t oob2 = ~m2;
    const int64_t *wo = p.win_offsets + w + (int)w / p.Q;
    const int64_t e0 = wo[0], e1 = wo[1];
    int64_t a0 = (e0 + 7) & ~(int64_t)7;
    if (a0 > e1) a0 = e1;
    const int64_t a1 = a0 + ((e1 - a0) & ~(int64_t)7);
    int kept = 0;
    for (int64_t e = e0 + threadIdx.x; e < a0; e += blockDim.x) bin_one(p, hist, 0, roi, p.x[e], p.y[e], kept);
    const uint4 *x8 = reinterpret_cast<const uint4 *>(p.x + a0);
    const uint4 *y8 = reinterpret_cast<const uint4 *>(p.y + a0);
    const int64_t n8 = (a1 - a0) >> 3;
    for (int64_t j = threadIdx.x; j < n8; j += blockDim.x) {
        const uint4 xv = __ldg(x8 + j), yv = __ldg(y8 + j);
        const uint32_t xs[4] = {xv.x, xv.y, xv.z, xv.w}, ys[4] = {yv.x, yv.y, yv.z, yv.w};
#pragma unroll
        for (int h = 0; h < 4; ++h) {
            if (((xs[h] | ys[h]) & oob2) == 0u) {            // both events inside the roi
                const uint32_t cx = (xs[h] + add2) & m2, cy = (ys[h] + add2) & m2;
                const uint32_t idx2 = (cy << log2roi) | cx;  // two bin indices, 16 bits each
                atomicAdd(&hist[idx2 & 0xffffu], 1u);
                atomicAdd(&hist[idx2 >> 16], 1u);
                kept += 2;
            } else {
                bin_one(p, hist, 0, roi, xs[h] & 0xffff, ys[h] & 0xffff, kept);
                bin_one(p, hist, 0, roi, xs[h] >> 16, ys[h] >> 16, kept);
            }
        }
    }
    for (int64_t e = a1 + threadIdx.x; e < e1; e += blockDim.x) bin_one(p, hist, 0, roi, p.x[e], p.y[e], kept);
    if (p.win_events) {
        for (int o = 16; o > 0; o >>= 1) kept += __shfl_xor_sync(0xffffffffu, kept, o);
        if ((threadIdx.x & 31) == 0 && kept) atomicAdd(&s_kept, kept);
    }
    __syncthreads();
    if (p.win_events && threadIdx.x == 0) p.win_events[w] = s_kept;
    if (p.frames) {
        uint32_t *f4 = reinterpret_cast<uint32_t *>(p.frames + w * (int64_t)nbins);
        for (int i = threadIdx.x; i < (nbins >> 2); i += blockDim.x) {
            uint32_t o = 0;
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                uint32_t v = hist[4 * i + b];
                v = p.wrap_u8 ? (v & 255u) : min(v, 255u);
                o |= v << (8 * b);
            }
            f4[i] = o;
        }
    }
    if (p.pooled) {
        const int I = p.dims * p.dims;
        for (int o = threadIdx.x; o < I; o += blockDim.x) {
            const int i = o / p.dims, j = o - i * p.dims;
            const uint32_t v = hist[(p.k * i + p.c) * roi + (p.k * j + p.c)];
            p.pooled[w * I + o] = (uint8_t)(p.wrap_u8 ? (v & 255u) : min(v, 255u));
        }
    }
}

__global__ void pool_kernel(const uint8_t *__restrict__ frames, int64_t n, int roi, int k, int dims,
                            int c, uint8_t *__restrict__ pooled)
{
    const int I = dims * dims;
    int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (idx >= n * I) return;
    int64_t f = idx / I;
    int o = (int)(idx - f * I);
    int i = o / dims, j = o - i * dims;
    pooled[idx] = __ldg(frames + (f * roi + (k * i + c)) * (int64_t)roi + (k * j + c));
}

}  // namespace lens

using namespace lens;

namespace {

// K1 for B streams of Q windows: argument checks (all before the first CUDA call), then the boundary search
// and one binning launch over the B * Q windows.  offsets == nullptr: one stream [0, n_events) from t0_us.
int bin_streams(const char *who, const uint32_t *t_us, const uint16_t *x, const uint16_t *y, int64_t n_events,
                const int64_t *offsets, const uint32_t *t0s, uint32_t t0_us, int64_t B, int64_t Q,
                uint32_t window_us, int roi_x0, int roi_y0, int roi, int k, int index_shift, int wrap_u8,
                uint8_t *frames, uint8_t *pooled, int32_t *win_events, int64_t *win_offsets, void *stream)
{
    LENS_CHECK_ARG(n_events >= 0 && B >= 0 && Q >= 0, "%s: negative size", who);
    LENS_CHECK_ARG(n_events == 0 || (t_us && x && y), "%s: NULL event array", who);
    LENS_CHECK_ARG(window_us > 0, "%s: window_us must be > 0", who);
    LENS_CHECK_ARG(roi > 0 && k > 0 && roi >= k, "%s: bad roi=%d k=%d", who, roi, k);
    LENS_CHECK_ARG(index_shift >= 0 && index_shift <= roi, "%s: bad index_shift", who);
    LENS_CHECK_ARG(win_offsets != nullptr, "%s: win_offsets scratch is NULL", who);
    LENS_CHECK_ARG(((uintptr_t)x & 15) == 0 && ((uintptr_t)y & 15) == 0, "%s: x / y must be 16-byte aligned", who);
    LENS_CHECK_ARG(B * Q <= 2147483647LL, "%s: too many windows", who);
    const int64_t n_win = B * Q;
    if (n_win == 0) return 0;
    BinParams p;
    p.x = x; p.y = y; p.win_offsets = win_offsets; p.Q = (int)Q;
    p.roi_x0 = roi_x0; p.roi_y0 = roi_y0; p.roi = roi; p.k = k; p.dims = roi / k;
    p.c = (k / 2) - 1; if (p.c < 0) p.c += k;
    p.index_shift = index_shift; p.wrap_u8 = wrap_u8;
    const int smem_budget = 96 * 1024;  // 2 CTAs / SM
    int band_rows = roi;
    while ((int64_t)band_rows * roi * 4 > smem_budget) band_rows = (band_rows + 1) / 2;
    p.band_rows = band_rows;
    p.n_bands = ceil_div(roi, band_rows);
    LENS_CHECK_ARG(p.n_bands <= 65535, "%s: roi=%d too large", who, roi);
    p.frames = frames; p.pooled = pooled; p.win_events = win_events;
    cudaStream_t st = as_stream(stream);
    {
        int threads = 256;
        int64_t blocks = ceil_div64(B * (Q + 1), threads);
        window_offsets_kernel<<<(unsigned)blocks, threads, 0, st>>>(t_us, n_events, offsets, t0s, t0_us, window_us,
                                                                    (int)B, Q, win_offsets);
        LENS_LAUNCH_CHECK();
    }
    size_t smem = (size_t)band_rows * roi * 4;
    LENS_CUDA(cudaFuncSetAttribute(bin_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   (int)smem));
    const bool pow2 = (roi & (roi - 1)) == 0 && roi >= 4 && roi <= 256;
    if (pow2 && roi_x0 == 0 && roi_y0 == 0 && p.n_bands == 1 && index_shift <= 1) {
        int log2roi = 0;
        while ((1 << log2roi) < roi) ++log2roi;
        LENS_CUDA(cudaFuncSetAttribute(bin_pow2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        bin_pow2_kernel<<<(unsigned)n_win, 512, smem, st>>>(p, log2roi);
    } else {
        dim3 grid((unsigned)n_win, (unsigned)p.n_bands);
        bin_kernel<<<grid, 512, smem, st>>>(p);
    }
    LENS_LAUNCH_CHECK();
    return 0;
}

int check_sorted(const char *who, const uint32_t *t_us, int64_t n, const int64_t *offsets, int B, int *unsorted,
                 void *stream)
{
    LENS_CHECK_ARG(n >= 0 && unsorted, "%s: bad argument", who);
    LENS_CHECK_ARG(n == 0 || t_us, "%s: NULL array", who);
    LENS_CHECK_ARG(((uintptr_t)t_us & 15) == 0, "%s: t_us must be 16-byte aligned", who);
    cudaStream_t st = as_stream(stream);
    LENS_CUDA(cudaMemsetAsync(unsorted, 0, sizeof(int), st));
    if (n > 1 || offsets) {   // with offsets always launched: they are checked even without events
        const int64_t blocks = std::min<int64_t>(ceil_div64(n >> 2, 256) + 1, (int64_t)std::max(sm_count(), 1) * 16);
        if (offsets) sorted_check_u32_kernel<true><<<(unsigned)blocks, 256, 0, st>>>(t_us, n, offsets, B, unsorted);
        else sorted_check_u32_kernel<false><<<(unsigned)blocks, 256, 0, st>>>(t_us, n, nullptr, 0, unsorted);
        LENS_LAUNCH_CHECK();
    }
    return 0;
}

}  // namespace

extern "C" int lens_bin_events(const uint32_t *t_us, const uint16_t *x, const uint16_t *y,
                               int64_t n_events, uint32_t t0_us, uint32_t window_us, int roi_x0,
                               int roi_y0, int roi, int k, int index_shift, int wrap_u8,
                               uint8_t *frames, uint8_t *pooled, int32_t *win_events,
                               int64_t *win_offsets, int64_t n_win, void *stream)
{
    LENS_CHECK_ARG(n_events >= 0 && n_win >= 0, "lens_bin_events: negative size");
    return bin_streams("lens_bin_events", t_us, x, y, n_events, nullptr, nullptr, t0_us, 1, n_win,
                       window_us, roi_x0, roi_y0, roi, k, index_shift, wrap_u8, frames, pooled, win_events,
                       win_offsets, stream);
}

extern "C" int lens_bin_event_streams(const uint32_t *t_us, const uint16_t *x, const uint16_t *y, int64_t n_events,
                                      const int64_t *offsets, const uint32_t *t0_us, int B, int Q, uint32_t window_us,
                                      int roi_x0, int roi_y0, int roi, int k, int index_shift, int wrap_u8,
                                      uint8_t *frames, uint8_t *pooled, int32_t *win_events, int64_t *win_offsets,
                                      void *stream)
{
    LENS_CHECK_ARG(B >= 0 && Q >= 0, "lens_bin_event_streams: negative B=%d or Q=%d", B, Q);
    LENS_CHECK_ARG((int64_t)B * Q == 0 || (offsets && t0_us), "lens_bin_event_streams: NULL offsets / t0_us");
    return bin_streams("lens_bin_event_streams", t_us, x, y, n_events, offsets, t0_us, 0, B, Q, window_us, roi_x0,
                       roi_y0, roi, k, index_shift, wrap_u8, frames, pooled, win_events, win_offsets, stream);
}

extern "C" int lens_check_sorted_u32(const uint32_t *t_us, int64_t n, int *unsorted, void *stream)
{
    return check_sorted("lens_check_sorted_u32", t_us, n, nullptr, 0, unsorted, stream);
}

extern "C" int lens_check_sorted_segments_u32(const uint32_t *t_us, int64_t n, const int64_t *offsets, int B, int *bad,
                                              void *stream)
{
    LENS_CHECK_ARG(B >= 0 && offsets, "lens_check_sorted_segments_u32: bad B=%d or NULL offsets", B);
    return check_sorted("lens_check_sorted_segments_u32", t_us, n, offsets, B, bad, stream);
}

extern "C" int lens_pool_frames(const uint8_t *frames, int64_t n, int roi, int k, uint8_t *pooled,
                                void *stream)
{
    LENS_CHECK_ARG(n >= 0 && roi > 0 && k > 0 && roi >= k, "lens_pool_frames: bad sizes");
    LENS_CHECK_ARG(n == 0 || (frames && pooled), "lens_pool_frames: NULL buffer");
    if (n == 0) return 0;
    int dims = roi / k;
    int c = (k / 2) - 1; if (c < 0) c += k;
    int64_t total = n * dims * dims;
    int threads = 256;
    pool_kernel<<<(unsigned)ceil_div64(total, threads), threads, 0, as_stream(stream)>>>(
        frames, n, roi, k, dims, c, pooled);
    LENS_LAUNCH_CHECK();
    return 0;
}
