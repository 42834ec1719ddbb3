// K2 + K3 (CUDA-core path): the converted sinabs network of lens/run_model.py:139-156
//   IAF#0 -> Linear(I->F) -> IAF#1 -> Linear(F->P) -> IAF#2
// and the per-query loop of lens/run_model.py:229-246, for B independent streams.
//
// Arithmetic contract (DESIGN.md "exact contraction"): both Linear contractions are
// evaluated EXACTLY -- spikes are small integers, weights are converted once to a
// per-row fixed-point grid (w = m * 2^q, |m| < 2^46, lossless for every weight whose
// exponent lies within 22 bits of the row maximum), the products are accumulated in
// int64 and rounded once to fp32 (round-to-nearest-even).  The result is the
// correctly rounded value of sum_k s_k * w_k, independent of summation order, so the
// event-driven kernel below, the tcgen05 digit-plane kernel (snn_tc.cu) and the CPU
// oracle agree bit for bit.  The IAF update itself is elementwise IEEE fp32.
//
// Time is serial per (stream, neuron) because of the membrane recurrence; the
// parallel axes are streams and neurons.  Layers are feed-forward, so the feature
// layer of a stream runs ahead over all its steps (feature_kernel) and leaves the
// hidden spikes as int8 rows in HBM for the output layer (output_simt_kernel here,
// or the tensor-core kernel).  Both kernels keep their membrane potential in a
// register for the whole launch; spikes are sparse (~3 % of inputs, ~4 % of hidden
// units fire per step), so the CUDA-core contraction is event driven: per step the
// active (index, count) pairs are compacted in shared memory and every thread adds
// the matching weight column entries.
#include "snn.cuh"

#include <algorithm>
#include <climits>

namespace lens {

// --------------------------------------------------------------------------------
// weights -> fixed point
// --------------------------------------------------------------------------------
// One CTA per output neuron n.  W [n_out][n_in] f32  ->  fx [n_in][n_out] i64, scale [n_out].
// w = m * 2^q with q = emax - kFxBits (|m| < 2^46), then the trailing zero bits common to the whole
// row are shifted out (q grows by the same amount, the products stay exact): fp32 weights carry 24
// significant bits, so a row whose weights span s binary orders of magnitude needs only 24 + s bits,
// i.e. fewer radix-256 digit planes on the tensor-core path (snn_tc.cu).
__device__ __forceinline__ int64_t weight_to_fixed(float w, int q, bool &inexact)
{
    const uint32_t u = __float_as_uint(w);
    const int ef = (u >> 23) & 255;
    const uint32_t frac = u & 0x7fffffu;
    int64_t m = 0;
    inexact = false;
    if (ef == 255) {
        inexact = true;                                          // inf / nan -> 0, flagged
    } else if (!(ef == 0 && frac == 0)) {
        const int64_t mant = (ef == 0) ? (int64_t)frac : (int64_t)(frac | 0x800000u);
        const int e_ulp = (ef == 0) ? -149 : ef - 150;           // w = mant * 2^e_ulp
        const int sh = e_ulp - q;
        if (sh >= 0) {
            m = mant << sh;                                      // sh <= 22 by construction
        } else {
            const int r = -sh;
            if (r > 26) { m = 0; inexact = true; }
            else {
                int64_t keep = mant >> r;
                const int64_t rem = mant & ((1ll << r) - 1), half = 1ll << (r - 1);
                if (rem > half || (rem == half && (keep & 1))) ++keep;   // RNE
                if (rem) inexact = true;
                m = keep;
            }
        }
        if (u >> 31) m = -m;
    }
    return m;
}

__global__ void __launch_bounds__(256) weights_to_fixed_kernel(const float *__restrict__ W,
                                                               int n_out, int n_in,
                                                               int64_t *__restrict__ fx,
                                                               float *__restrict__ scale,
                                                               int64_t *__restrict__ n_inexact)
{
    __shared__ int s_emax;
    __shared__ unsigned long long s_bits;
    const int n = blockIdx.x;
    if (threadIdx.x == 0) { s_emax = INT_MIN; s_bits = 0ull; }
    __syncthreads();
    int emax = INT_MIN;
    for (int k = threadIdx.x; k < n_in; k += blockDim.x) {
        uint32_t u = __float_as_uint(W[(size_t)n * n_in + k]);
        int ef = (u >> 23) & 255;
        uint32_t frac = u & 0x7fffffu;
        if (ef == 255 || (ef == 0 && frac == 0)) continue;          // inf/nan/zero
        int e = (ef == 0 ? -149 : ef - 150) + 24;                   // |w| < 2^e
        emax = max(emax, e);
    }
    for (int o = 16; o > 0; o >>= 1) emax = max(emax, __shfl_xor_sync(0xffffffffu, emax, o));
    if ((threadIdx.x & 31) == 0) atomicMax(&s_emax, emax);
    __syncthreads();
    emax = s_emax;
    int q = (emax == INT_MIN) ? 0 : emax - kFxBits;
    if (q < -126) q = -126;                                          // keep 2^q a normal float
    // trailing zeros common to the row
    unsigned long long bits = 0ull;
    int64_t bad = 0;
    for (int k = threadIdx.x; k < n_in; k += blockDim.x) {
        bool inexact;
        const int64_t m = weight_to_fixed(W[(size_t)n * n_in + k], q, inexact);
        bits |= (unsigned long long)(m < 0 ? -m : m);
        bad += inexact;
    }
    for (int o = 16; o > 0; o >>= 1) bits |= __shfl_xor_sync(0xffffffffu, bits, o);
    if ((threadIdx.x & 31) == 0 && bits) atomicOr(&s_bits, bits);
    __syncthreads();
    bits = s_bits;
    int tz = bits ? __ffsll((long long)bits) - 1 : 0;
    if (q + tz > 127) tz = 127 - q;
    if (threadIdx.x == 0) scale[n] = __uint_as_float((uint32_t)(q + tz + 127) << 23);
    for (int k = threadIdx.x; k < n_in; k += blockDim.x) {
        bool inexact;
        const int64_t m = weight_to_fixed(W[(size_t)n * n_in + k], q, inexact);
        fx[(size_t)k * n_out + n] = m >> tz;                         // exact: tz zero bits leave
    }
    for (int o = 16; o > 0; o >>= 1) bad += __shfl_xor_sync(0xffffffffu, bad, o);
    if ((threadIdx.x & 31) == 0 && bad) atomicAdd((unsigned long long *)n_inexact, (unsigned long long)bad);
}

// --------------------------------------------------------------------------------
// event list helpers
// --------------------------------------------------------------------------------
// Compact the non-zero entries of `row[0..n)` (one byte per neuron) into (idx, cnt)
// lists; executed by one full warp.  Returns the number of active entries.
__device__ __forceinline__ int warp_compact(const uint8_t *row, int n, uint16_t *idx, uint8_t *cnt)
{
    const int lane = threadIdx.x & 31;
    int base = 0;
    for (int i0 = 0; i0 < n; i0 += 32) {
        int i = i0 + lane;
        uint8_t v = (i < n) ? row[i] : (uint8_t)0;
        unsigned m = __ballot_sync(0xffffffffu, v != 0);
        if (v) {
            int pos = base + __popc(m & ((1u << lane) - 1));
            idx[pos] = (uint16_t)i;
            cnt[pos] = v;
        }
        base += __popc(m);
    }
    return base;
}

// Same, for a row (timestep n) of a hidden-spike tile in the canonical UMMA layout.
__device__ __forceinline__ int warp_compact_tiled(const uint8_t *tile, int n, int F, uint16_t *idx, uint8_t *cnt)
{
    const int lane = threadIdx.x & 31;
    int base = 0;
    for (int i0 = 0; i0 < F; i0 += 32) {
        int i = i0 + lane;
        uint8_t v = (i < F) ? tile[s1_byte_in_half(n, i)] : (uint8_t)0;
        unsigned m = __ballot_sync(0xffffffffu, v != 0);
        if (v) {
            int pos = base + __popc(m & ((1u << lane) - 1));
            idx[pos] = (uint16_t)i;
            cnt[pos] = v;
        }
        base += __popc(m);
    }
    return base;
}

constexpr int kChunk = kTileSteps;   // timesteps per hidden-spike tile (= steps between block syncs)

struct FeatureParams {
    int I, F, Fp, T;
    float thr, vmin;
    const int64_t *Wf_fx;     // [I][F]
    const float *Wf_scale;    // [F]
    const float *U;           // [T][I]
    const uint8_t *pooled;    // [B][Q][I]           (raster mode)
    const float *xin;         // [B][steps][I]       (float mode), exactly one of the two
    int steps;                // per stream (= Q*T in raster mode)
    float *v0, *v1;           // state, already offset to the first stream of this launch
    int8_t *S1;               // [pairs][chunks][Fp/16][2*kTileSteps][16] (pair tiles, see snn.cuh)
    uint8_t *hidden_steps;    // nullable [nb][steps][F]
    int64_t *overflow;
};

// grid = streams, block = round_up(max(I, F), 32) threads.  Thread i < I owns input
// neuron i (IAF#0), thread f < F owns feature neuron f (IAF#1).
__global__ void __launch_bounds__(1024) feature_kernel(FeatureParams p)
{
    extern __shared__ uint8_t smem_raw[];
    const int I = p.I, F = p.F;
    const int Ipad = (I + 31) & ~31;
    uint8_t *s0 = smem_raw;                                    // [kChunk][Ipad] input spikes
    uint16_t *l_idx = reinterpret_cast<uint16_t *>(s0 + kChunk * Ipad);   // [kChunk][Ipad]
    uint8_t *l_cnt = reinterpret_cast<uint8_t *>(l_idx + kChunk * Ipad);  // [kChunk][Ipad]
    int *n_act = reinterpret_cast<int *>(l_cnt + kChunk * Ipad);          // [kChunk]
    uint8_t *tile = reinterpret_cast<uint8_t *>(n_act + kChunk);          // [Fp/16][kChunk][16] this stream's half tile

    const int b = blockIdx.x;
    const int tid = threadIdx.x;
    const int warp = tid >> 5, nwarps = blockDim.x >> 5;
    const float thr = p.thr, vmin = p.vmin;
    const int n_chunks = n_chunks_of(p.steps, p.T);
    float v0 = (tid < I) ? p.v0[(size_t)b * I + tid] : 0.0f;
    float v1 = (tid < F) ? p.v1[(size_t)b * F + tid] : 0.0f;
    const float scale = (tid < F) ? p.Wf_scale[tid] : 0.0f;
    int64_t n_over = 0;
    float prob = 0.0f;

    for (int ch = 0; ch < n_chunks; ++ch) {
        int t0, nc;
        chunk_span(ch, p.steps, p.T, t0, nc);
        // ---- phase A: IAF#0 over the chunk (elementwise, no cross-thread dependency)
        if (tid < I) {
            for (int c = 0; c < nc; ++c) {
                const int step = t0 + c;
                float xin;
                if (p.pooled) {
                    const int q = step / p.T, t = step - q * p.T;
                    if (t == 0 || c == 0)   // lens/src/dataset.py:23  p = u8 / 255 (fp32 division)
                        prob = __fdiv_rn((float)p.pooled[((size_t)b * (p.steps / p.T) + q) * I + tid], 255.0f);
                    xin = (__ldg(p.U + (size_t)t * I + tid) < prob) ? 1.0f : 0.0f;  // dataset.py:121
                } else {
                    xin = p.xin[((size_t)b * p.steps + step) * I + tid];
                }
                float s = iaf_step(v0, xin, thr, vmin);
                if (s > (float)LENS_MAX_SPIKE) { s = (float)LENS_MAX_SPIKE; ++n_over; }
                s0[c * Ipad + tid] = (uint8_t)s;
            }
        }
        __syncthreads();
        // ---- phase B: per-step active lists
        for (int c = warp; c < nc; c += nwarps) {
            int n = warp_compact(s0 + c * Ipad, I, l_idx + c * Ipad, l_cnt + c * Ipad);
            if ((tid & 31) == 0) n_act[c] = n;
        }
        __syncthreads();
        // ---- phase C: exact contraction + IAF#1
        if (tid < F) {
            for (int c = 0; c < nc; ++c) {
                const int n = n_act[c];
                int64_t acc = 0;
                for (int a = 0; a < n; ++a) {
                    const int i = l_idx[c * Ipad + a];
                    const int64_t s = l_cnt[c * Ipad + a];
                    acc += s * __ldg(p.Wf_fx + (size_t)i * F + tid);
                }
                const float x = __fmul_rn(__ll2float_rn(acc), scale);
                float s = iaf_step(v1, x, thr, vmin);
                if (s > (float)LENS_MAX_SPIKE) { s = (float)LENS_MAX_SPIKE; ++n_over; }
                tile[s1_byte_in_half(c, tid)] = (uint8_t)s;
                if (p.hidden_steps) p.hidden_steps[((size_t)b * p.steps + t0 + c) * F + tid] = (uint8_t)s;
            }
            for (int c = nc; c < kChunk; ++c) tile[s1_byte_in_half(c, tid)] = 0;   // ragged last tile
        } else if (tid < p.Fp) {   // K padding
            for (int c = 0; c < kChunk; ++c) tile[s1_byte_in_half(c, tid)] = 0;
        }
        __syncthreads();
        {   // the finished half tile leaves with 16-byte stores into its rows of the pair tile
            uint4 *dst = reinterpret_cast<uint4 *>(p.S1 + ((size_t)(b >> 1) * n_chunks + ch) * s1_tile_bytes(p.Fp));
            const uint4 *src = reinterpret_cast<const uint4 *>(tile);
            const int n16 = p.Fp / 16 * kChunk;
            const int sp = b & 1;
            for (int i = tid; i < n16; i += blockDim.x)
                dst[(i / kChunk) * kTileRows + s1_row(sp, i % kChunk)] = src[i];
        }
    }
    if (tid < I) p.v0[(size_t)b * I + tid] = v0;
    if (tid < F) p.v1[(size_t)b * F + tid] = v1;
    if (n_over) atomicAdd((unsigned long long *)p.overflow, (unsigned long long)n_over);
}

// --------------------------------------------------------------------------------
// raster fast path of the feature layer
// --------------------------------------------------------------------------------
// lens/src/dataset.py:23,121: spike = (U[t][i] < pixel / 255).  pixel / 255 (fp32 division) is
// monotone in the pixel value, so the comparison is equivalent to pixel > Uq[t][i] with
//   Uq[t][i] = (smallest pixel in 1..255 with U[t][i] < pixel/255) - 1,   255 if there is none
// -- one byte per (step, input), built once per handle by exact evaluation of the same fp32 division.
__global__ void raster_thresholds_kernel(const float *__restrict__ U, int n, uint8_t *__restrict__ Uq)
{
    int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n) return;
    const float u = U[idx];
    int lo = 1, hi = 256;                       // first pixel value that spikes, 256 = never
    while (lo < hi) {
        int mid = (lo + hi) >> 1;
        if (u < __fdiv_rn((float)mid, 255.0f)) hi = mid;
        else lo = mid + 1;
    }
    Uq[idx] = (uint8_t)(lo - 1);
}

constexpr int kRasterSlots = 4;      // streams processed concurrently by one CTA

struct RasterParams {
    int I, F, Fp, T, Q, steps, nb;
    float vmin;
    const int64_t *Wf_fx;     // [I][F]
    const float *Wf_scale;    // [F]
    const uint8_t *Uq;        // [T][I]
    const uint8_t *pooled;    // [nb][Q][I]
    float *v1;                // [nb][F] (offset to the first stream of the launch)
    int8_t *S1;               // pair tiles
    uint8_t *hidden_steps;    // nullable [nb][steps][F]
    int64_t *overflow;
};

// Feature layer for binary raster input, threshold 1, IAF#0 at rest (v0 == 0): IAF#0 is then the
// identity (v = 0 + 1 -> one spike -> v = 0), so input spikes come straight from the byte
// comparison above.  Persistent CTAs; each CTA keeps the whole fixed-point W_feat in shared
// memory and runs kRasterSlots streams side by side (slot = blockDim.x / kRasterSlots threads,
// thread f of a slot owns feature neuron f with its membrane potential in a register).
// Per tile of 32 timesteps: (A) every warp compacts the active inputs of some steps into a list of
// weight-row offsets, (C) every thread walks its 32 steps: exact int64 sum over the listed rows,
// IAF#1, spike byte into the slot's tile, (W) the tile leaves for HBM in the pair-tile layout.
// shared-memory accessors on 32-bit shared-window addresses (keeps the hot loop free of
// generic-to-shared address conversions)
__device__ __forceinline__ uint32_t lds_u16(uint32_t a)
{
    uint16_t v;
    asm volatile("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ int64_t lds_s64(uint32_t a)
{
    int64_t v;
    asm volatile("ld.shared.s64 %0, [%1];" : "=l"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ int lds_s32(uint32_t a)
{
    int v;
    asm volatile("ld.shared.s32 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ void sts_u8(uint32_t a, uint32_t v)
{
    asm volatile("st.shared.u8 [%0], %1;" ::"r"(a), "r"(v) : "memory");
}

// slow path of IAF#1: more than one spike in a step (kept out of line so the hot loop stays short);
// returns trunc(vv) and, in the low byte of `packed`, the spike count clipped to LENS_MAX_SPIKE
// (bit 8 set when it had to be clipped)
__device__ __noinline__ float multi_spike(float vv, uint32_t *packed)
{
    const float s = truncf(vv);
    const bool over = s > (float)LENS_MAX_SPIKE;
    *packed = (uint32_t)(over ? (float)LENS_MAX_SPIKE : s) | (over ? 256u : 0u);
    return s;
}

template <bool kDebug>
__global__ void __launch_bounds__(1024, 1) feature_raster_kernel(RasterParams p)
{
    extern __shared__ __align__(16) uint8_t smem_raw[];
    const int I = p.I, F = p.F, Fp = p.Fp;
    const int Ipad = (I + 31) & ~31;
    const int slot_threads = blockDim.x / kRasterSlots;
    const int slot = threadIdx.x / slot_threads;
    const int f = threadIdx.x - slot * slot_threads;
    const int lane = threadIdx.x & 31;
    const int slot_warp = f >> 5, slot_warps = slot_threads >> 5;
    int64_t *sW = reinterpret_cast<int64_t *>(smem_raw);                       // [I][F]
    size_t off = ((size_t)I * F * 8 + 15) & ~(size_t)15;
    uint16_t *sList = reinterpret_cast<uint16_t *>(smem_raw + off) + (size_t)slot * kChunk * Ipad;  // [kChunk][Ipad] i*F
    off += (size_t)kRasterSlots * kChunk * Ipad * 2;
    int *sCnt = reinterpret_cast<int *>(smem_raw + off) + slot * kChunk;       // [kChunk] active inputs per step
    off += (size_t)kRasterSlots * kChunk * 4;
    uint8_t *tile = smem_raw + off + (size_t)slot * kChunk * Fp;               // [Fp/16][kChunk][16]

    for (int i = threadIdx.x; i < I * F; i += blockDim.x) sW[i] = p.Wf_fx[i];
    const float scale = (f < F) ? p.Wf_scale[f] : 0.0f;
    const float vmin = p.vmin;
    const int n_chunks = n_chunks_of(p.steps, p.T);
    const uint32_t a_w = (uint32_t)__cvta_generic_to_shared(sW) + 8u * (uint32_t)(f < F ? f : 0);
    const uint32_t a_list = (uint32_t)__cvta_generic_to_shared(sList);
    const uint32_t a_cnt = (uint32_t)__cvta_generic_to_shared(sCnt);
    const uint32_t a_tile = (uint32_t)__cvta_generic_to_shared(tile) + (uint32_t)((f >> 4) * (kChunk * 16) + (f & 15));
    int64_t n_over = 0;
    __syncthreads();

    const int n_groups = (p.nb + kRasterSlots - 1) / kRasterSlots;
    for (int g = blockIdx.x; g < n_groups; g += gridDim.x) {
        const int b = g * kRasterSlots + slot;
        const bool live = b < p.nb;
        float v1 = (live && f < F) ? p.v1[(size_t)b * F + f] : 0.0f;
        for (int ch = 0; ch < n_chunks; ++ch) {
            int t0, nc;
            chunk_span(ch, p.steps, p.T, t0, nc);
            // ---- (A) active-input lists of this tile's steps (entries = weight-row offsets i * F)
            if (live) {
                for (int c = slot_warp; c < nc; c += slot_warps) {
                    const int step = t0 + c;
                    const int q = step / p.T, t = step - q * p.T;
                    const uint8_t *px = p.pooled + ((size_t)b * p.Q + q) * I;
                    const uint8_t *uq = p.Uq + (size_t)t * I;
                    uint16_t *lst = sList + c * Ipad;
                    int base = 0;
                    for (int i0 = 0; i0 < I; i0 += 32) {
                        const int i = i0 + lane;
                        const bool spike = (i < I) && (__ldg(px + i) > __ldg(uq + i));
                        const unsigned m = __ballot_sync(0xffffffffu, spike);
                        if (spike) lst[base + __popc(m & ((1u << lane) - 1))] = (uint16_t)(i * F);
                        base += __popc(m);
                    }
                    if (lane == 0) sCnt[c] = base;
                }
            }
            __syncthreads();
            // ---- (C) exact contraction over the listed weight rows + IAF#1
            if (live && f < F) {
                uint32_t al = a_list, ac = a_cnt, at = a_tile;
#pragma unroll 1
                for (int c = 0; c < nc; ++c, al += 2 * Ipad, ac += 4, at += 16) {
                    const int n = lds_s32(ac);
                    int64_t acc = 0;
#pragma unroll 1
                    for (uint32_t a = al, ae = al + 2 * n; a != ae; a += 2) acc += lds_s64(a_w + 8u * lds_u16(a));
                    const float x = __fmul_rn(__ll2float_rn(acc), scale);
                    float vv = __fadd_rn(v1, x);                // IAF#1 with thr == 1 (see iaf_step)
                    float s = (vv >= 1.0f) ? 1.0f : 0.0f;
                    uint32_t sb = (vv >= 1.0f) ? 1u : 0u;
                    if (vv >= 2.0f) {                           // rare: several spikes in one step
                        uint32_t packed;
                        s = multi_spike(vv, &packed);
                        sb = packed & 255u;
                        n_over += packed >> 8;
                    }
                    vv = __fsub_rn(vv, s);                      // exact: s is the integer part of vv
                    v1 = __fadd_rn(fmaxf(__fsub_rn(vv, vmin), 0.0f), vmin);
                    sts_u8(at, sb);
                    if (kDebug) p.hidden_steps[((size_t)b * p.steps + t0 + c) * F + f] = (uint8_t)sb;
                }
                for (int c = nc; c < kChunk; ++c) tile[s1_byte_in_half(c, f)] = 0;   // ragged last tile
            } else if (live && f < Fp) {
                for (int c = 0; c < kChunk; ++c) tile[s1_byte_in_half(c, f)] = 0;    // K padding
            }
            __syncthreads();
            // ---- (W) this stream's rows of the pair tile
            if (live) {
                uint4 *dst = reinterpret_cast<uint4 *>(p.S1 + ((size_t)(b >> 1) * n_chunks + ch) * s1_tile_bytes(Fp));
                const uint4 *src = reinterpret_cast<const uint4 *>(tile);
                const int n16 = Fp / 16 * kChunk;
                const int sp = b & 1;
                for (int i = f; i < n16; i += slot_threads)
                    dst[(i / kChunk) * kTileRows + s1_row(sp, i % kChunk)] = src[i];
            }
        }
        if (live && f < F) p.v1[(size_t)b * F + f] = v1;
    }
    if (n_over) atomicAdd((unsigned long long *)p.overflow, (unsigned long long)n_over);
}

static size_t raster_smem_bytes(const SnnHandle *h)
{
    const int Ipad = (h->I + 31) & ~31;
    return (((size_t)h->I * h->F * 8 + 15) & ~(size_t)15) + (size_t)kRasterSlots * kChunk * Ipad * 2 + (size_t)kRasterSlots * kChunk * 4 +
           (size_t)kRasterSlots * kChunk * h->Fp;
}

// IAF#0 stays at rest only for v_min <= 0: with v_min > 0 a step without input lifts it to v_min (and
// v_min >= 1 makes it fire on its own), which feature_kernel computes and this path does not.
static bool raster_path_ok(const SnnHandle *h)
{
    return h->Uq && h->thr == 1.0f && h->vmin <= 0.0f && !h->v0_dirty && (size_t)h->I * h->F <= 65535 &&
           h->Fp * kRasterSlots <= 1024 && raster_smem_bytes(h) <= 227 * 1024;
}

static int launch_feature_raster(SnnHandle *h, const uint8_t *pooled, int b0, int nb, int steps,
                                 uint8_t *hidden_steps, cudaStream_t st)
{
    RasterParams p;
    p.I = h->I; p.F = h->F; p.Fp = h->Fp; p.T = h->T; p.Q = steps / h->T; p.steps = steps; p.nb = nb;
    p.vmin = h->vmin; p.Wf_fx = h->Wf_fx; p.Wf_scale = h->Wf_scale; p.Uq = h->Uq; p.pooled = pooled;
    p.v1 = h->v1 + (size_t)b0 * h->F; p.S1 = h->S1; p.hidden_steps = hidden_steps; p.overflow = h->counters;
    const size_t smem = raster_smem_bytes(h);
    const int threads = kRasterSlots * h->Fp;
    const int grid = std::min(std::max(sm_count(), 1), ceil_div(nb, kRasterSlots));
    LaunchTimer timer(h, st, 0);
    if (hidden_steps) {
        LENS_CUDA(cudaFuncSetAttribute(feature_raster_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        feature_raster_kernel<true><<<grid, threads, smem, st>>>(p);
    } else {
        LENS_CUDA(cudaFuncSetAttribute(feature_raster_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        feature_raster_kernel<false><<<grid, threads, smem, st>>>(p);
    }
    LENS_LAUNCH_CHECK();
    return 0;
}

struct OutputParams {
    int F, Fp, P, T;
    float thr, vmin;
    const int64_t *Wo_fx;    // [F][P]
    const float *Wo_scale;   // [P]
    const int8_t *S1;        // [pairs][chunks][Fp/16][2*kTileSteps][16] (pair tiles)
    int steps;
    float *v2;               // state, offset to first stream of the launch
    float *counts;           // [nb][steps/T][P], nullable
    float *spikes_out;       // [nb][steps][P] f32, nullable (operator seam)
    uint8_t *out_steps;      // [nb][steps][P] u8, nullable (debug)
};

constexpr int kOutThreads = 128;

// grid = (streams, place tiles); block = 128 threads, thread owns one place.
__global__ void __launch_bounds__(kOutThreads) output_simt_kernel(OutputParams p)
{
    extern __shared__ uint8_t smem_raw[];
    const int Fp = p.Fp, F = p.F, P = p.P;
    uint8_t *s1 = smem_raw;                                               // [kChunk][Fp]
    uint16_t *l_idx = reinterpret_cast<uint16_t *>(s1 + kChunk * Fp);     // [kChunk][Fp]
    uint8_t *l_cnt = reinterpret_cast<uint8_t *>(l_idx + kChunk * Fp);    // [kChunk][Fp]
    int *n_act = reinterpret_cast<int *>(l_cnt + kChunk * Fp);            // [kChunk]

    const int b = blockIdx.x;
    const int tid = threadIdx.x;
    const int warp = tid >> 5;
    const int place = blockIdx.y * kOutThreads + tid;
    const bool live = place < P;
    const float thr = p.thr, vmin = p.vmin;
    float v2 = live ? p.v2[(size_t)b * P + place] : 0.0f;
    const float scale = live ? p.Wo_scale[place] : 0.0f;
    const int64_t *wcol = p.Wo_fx + (live ? place : 0);
    float count = 0.0f;
    const int Q = p.steps / p.T;
    const int n_chunks = n_chunks_of(p.steps, p.T);

    for (int ch = 0; ch < n_chunks; ++ch) {
        int t0, nc;
        chunk_span(ch, p.steps, p.T, t0, nc);
        // stage this stream's rows of the pair tile with 16-byte loads
        {
            const uint4 *src = reinterpret_cast<const uint4 *>(p.S1 + ((size_t)(b >> 1) * n_chunks + ch) * s1_tile_bytes(Fp));
            uint4 *dst = reinterpret_cast<uint4 *>(s1);
            const int n16 = Fp / 16 * kChunk;
            const int sp = b & 1;
            for (int i = tid; i < n16; i += kOutThreads)
                dst[i] = __ldg(src + (i / kChunk) * kTileRows + s1_row(sp, i % kChunk));
        }
        __syncthreads();
        for (int c = warp; c < nc; c += kOutThreads / 32) {
            int n = warp_compact_tiled(s1, c, F, l_idx + c * Fp, l_cnt + c * Fp);
            if ((tid & 31) == 0) n_act[c] = n;
        }
        __syncthreads();
        if (live) {
            for (int c = 0; c < nc; ++c) {
                const int n = n_act[c];
                int64_t acc = 0;
                for (int a = 0; a < n; ++a) {
                    const int k = l_idx[c * Fp + a];
                    const int64_t s = l_cnt[c * Fp + a];
                    acc += s * __ldg(wcol + (size_t)k * P);
                }
                const float x = __fmul_rn(__ll2float_rn(acc), scale);
                const float s = iaf_step(v2, x, thr, vmin);
                const int step = t0 + c;
                const size_t row = (size_t)b * p.steps + step;
                if (p.spikes_out) p.spikes_out[row * P + place] = s;
                if (p.out_steps) p.out_steps[row * P + place] = (uint8_t)fminf(s, 255.0f);
                if (p.counts) {
                    count += s;                                   // run_model.py:239 sum over T
                    const int q = step / p.T;
                    if (step - q * p.T == p.T - 1) {
                        p.counts[((size_t)b * Q + q) * P + place] = count;
                        count = 0.0f;
                    }
                }
            }
        }
        __syncthreads();
    }
    if (live) p.v2[(size_t)b * P + place] = v2;
}

static constexpr size_t feature_smem_bytes(int I, int Fp)
{
    return (size_t)kChunk * ((I + 31) & ~31) * 4 + kChunk * sizeof(int) + (size_t)kChunk * Fp;
}

static constexpr size_t output_simt_smem_bytes(int Fp) { return (size_t)kChunk * Fp * 4 + kChunk * sizeof(int); }

// Dynamic shared memory above the default 48 KB needs a per-kernel opt-in.  A handle opts the CUDA-core
// kernels in once, to what the largest shape lens_snn_create accepts needs (I = 1024, F = 992), so handles
// of different sizes never lower each other's limit; shapes that fit 48 KB (the bundled models) never make
// the call.
constexpr size_t kDefaultSmem = 48 * 1024;
constexpr size_t kFeatureSmemMax = feature_smem_bytes(1024, 992), kOutputSmemMax = output_simt_smem_bytes(992);
static_assert(kFeatureSmemMax <= 227 * 1024 && kOutputSmemMax <= 227 * 1024,
              "the CUDA-core kernels must run every shape lens_snn_create accepts");

static int launch_feature(SnnHandle *h, const uint8_t *pooled, const float *xin, int b0, int nb,
                          int steps, uint8_t *hidden_steps, cudaStream_t st)
{
    FeatureParams p;
    p.I = h->I; p.F = h->F; p.Fp = h->Fp; p.T = h->T; p.thr = h->thr; p.vmin = h->vmin;
    p.Wf_fx = h->Wf_fx; p.Wf_scale = h->Wf_scale; p.U = h->U;
    p.pooled = pooled; p.xin = xin; p.steps = steps;
    p.v0 = h->v0 + (size_t)b0 * h->I; p.v1 = h->v1 + (size_t)b0 * h->F;
    p.S1 = h->S1; p.hidden_steps = hidden_steps; p.overflow = h->counters;
    int threads = (std::max(std::max(h->I, h->Fp), 32) + 31) & ~31;
    const size_t smem = feature_smem_bytes(h->I, h->Fp);
    if (smem > kDefaultSmem && !h->feature_smem_optin) {
        LENS_CUDA(cudaFuncSetAttribute(feature_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kFeatureSmemMax));
        h->feature_smem_optin = true;
    }
    LaunchTimer timer(h, st, 0);
    feature_kernel<<<nb, threads, smem, st>>>(p);
    LENS_LAUNCH_CHECK();
    return 0;
}

static int launch_output_simt(SnnHandle *h, int b0, int nb, int steps, float *counts,
                              float *spikes_out, uint8_t *out_steps, cudaStream_t st)
{
    OutputParams p;
    p.F = h->F; p.Fp = h->Fp; p.P = h->P; p.T = h->T; p.thr = h->thr; p.vmin = h->vmin;
    p.Wo_fx = h->Wo_fx; p.Wo_scale = h->Wo_scale; p.S1 = h->S1; p.steps = steps;
    p.v2 = h->v2 + (size_t)b0 * h->P;
    p.counts = counts; p.spikes_out = spikes_out; p.out_steps = out_steps;
    const size_t smem = output_simt_smem_bytes(h->Fp);
    if (smem > kDefaultSmem && !h->output_smem_optin) {
        LENS_CUDA(cudaFuncSetAttribute(output_simt_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kOutputSmemMax));
        h->output_smem_optin = true;
    }
    dim3 grid(nb, ceil_div(h->P, kOutThreads));
    LaunchTimer timer(h, st, 1);
    output_simt_kernel<<<grid, kOutThreads, smem, st>>>(p);
    LENS_LAUNCH_CHECK();
    return 0;
}

static int ensure_scratch(SnnHandle *h, size_t bytes)
{
    if (bytes <= h->S1_cap) return 0;
    if (h->S1) LENS_CUDA(cudaFree(h->S1));
    h->S1 = nullptr; h->S1_cap = 0;
    LENS_CUDA(cudaMalloc(&h->S1, bytes));
    h->S1_cap = bytes;
    return 0;
}

// Streams are processed in groups so the hidden-spike scratch stays bounded.
static size_t scratch_budget() { return (size_t)6 << 30; }

static int forward_common(SnnHandle *h, const uint8_t *pooled, const float *xin, int B, int steps,
                          float *counts, float *spikes_out, uint8_t *hidden_steps,
                          uint8_t *out_steps, int mode, cudaStream_t st, int first_stream = 0)
{
    const size_t per_pair = (size_t)n_chunks_of(steps, h->T) * s1_tile_bytes(h->Fp);
    // streams are processed in groups (even size: a pair tile never straddles two groups)
    int group = (int)std::min<size_t>((size_t)B + (B & 1), 2 * std::max<size_t>((size_t)1, scratch_budget() / std::max<size_t>(per_pair, 1)));
    int rc = ensure_scratch(h, per_pair * (group / 2));
    if (rc) return rc;
    const int Q = steps / h->T;
    bool use_tc = false;
    if (mode == LENS_SNN_TC) use_tc = true;
    else if (mode == LENS_SNN_AUTO) use_tc = snn_tc_supported(h) && !spikes_out && (size_t)B * h->P >= (size_t)64 * 1024;
    if (use_tc) {
        LENS_CHECK_ARG(snn_tc_supported(h) && !spikes_out,
                       "lens_snn_forward: tensor-core mode unavailable for this shape");
        rc = snn_tc_prepare(h, st);
        if (rc) return rc;
    }
    for (int bl = 0; bl < B; bl += group) {
        const int nb = std::min(group, B - bl);
        const int b0 = first_stream + bl;   // index into the handle's state arrays
        uint8_t *hs = hidden_steps ? hidden_steps + (size_t)bl * steps * h->F : nullptr;
        if (pooled && use_tc && snn_tc_hidden_supported(h))
            rc = snn_tc_hidden(h, pooled + (size_t)bl * Q * h->I, nb, b0, steps, hs, st);
        else if (pooled && raster_path_ok(h))
            rc = launch_feature_raster(h, pooled + (size_t)bl * Q * h->I, b0, nb, steps, hs, st);
        else
            rc = launch_feature(h, pooled ? pooled + (size_t)bl * Q * h->I : nullptr,
                                xin ? xin + (size_t)bl * steps * h->I : nullptr, b0, nb, steps, hs, st);
        if (rc) return rc;
        float *c = counts ? counts + (size_t)bl * Q * h->P : nullptr;
        uint8_t *os = out_steps ? out_steps + (size_t)bl * steps * h->P : nullptr;
        if (use_tc)
            rc = snn_tc_output(h, h->S1, nb, b0, steps, c, os, st);
        else
            rc = launch_output_simt(h, b0, nb, steps, c,
                                    spikes_out ? spikes_out + (size_t)bl * steps * h->P : nullptr, os, st);
        if (rc) return rc;
    }
    return 0;
}

// lens_snn_reset_streams: zero the membrane potentials of the masked streams, one CTA per stream at a time.
__global__ void __launch_bounds__(256) reset_streams_kernel(const uint8_t *__restrict__ mask, int maxB, int I, int F,
                                                            int P, float *__restrict__ v0, float *__restrict__ v1,
                                                            float *__restrict__ v2)
{
    for (int b = blockIdx.x; b < maxB; b += gridDim.x) {
        if (!mask[b]) continue;                             // block-uniform
        for (int i = threadIdx.x; i < I; i += blockDim.x) v0[(size_t)b * I + i] = 0.0f;
        for (int i = threadIdx.x; i < F; i += blockDim.x) v1[(size_t)b * F + i] = 0.0f;
        for (int i = threadIdx.x; i < P; i += blockDim.x) v2[(size_t)b * P + i] = 0.0f;
    }
}

// lens_snn_forward_streams: rows ids[i] of v0 / v1 / v2 <-> rows i of the workspace (kScatter: back to the state).
// One CTA per (stream, layer) at a time, 16-byte copies when the rows allow them; ids outside [0, maxB) are skipped.
template <bool kScatter>
__global__ void __launch_bounds__(256) state_rows_kernel(const int32_t *__restrict__ ids, int n, int maxB, int I, int F,
                                                         int P, float *__restrict__ v0, float *__restrict__ v1,
                                                         float *__restrict__ v2, float *__restrict__ ws, int ws_cap)
{
    for (long long w = blockIdx.x; w < 3LL * n; w += gridDim.x) {
        const int layer = (int)(w / n), i = (int)(w - (long long)layer * n);
        const int b = ids[i];
        if ((unsigned)b >= (unsigned)maxB) continue;                // block-uniform
        const int len = layer == 0 ? I : layer == 1 ? F : P;
        float *state = (layer == 0 ? v0 : layer == 1 ? v1 : v2) + (size_t)b * len;
        float *work = ws + (layer == 0 ? 0 : layer == 1 ? (size_t)ws_cap * I : (size_t)ws_cap * (I + F)) +
                      (size_t)i * len;
        const float *src = kScatter ? work : state;
        float *dst = kScatter ? state : work;
        if ((len & 3) == 0 && ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) & 15) == 0) {
            const float4 *s4 = reinterpret_cast<const float4 *>(src);
            float4 *d4 = reinterpret_cast<float4 *>(dst);
            for (int k = threadIdx.x; k < len / 4; k += blockDim.x) d4[k] = s4[k];
        } else {
            for (int k = threadIdx.x; k < len; k += blockDim.x) dst[k] = src[k];
        }
    }
}

}  // namespace lens

using namespace lens;

extern "C" int lens_snn_create(int I, int F, int P, int T, float thr, float v_min,
                               const float *W_feat, const float *W_out, const float *U,
                               int max_streams, void **handle, int64_t *n_inexact, void *stream)
{
    LENS_CHECK_ARG(handle != nullptr, "lens_snn_create: handle is NULL");
    *handle = nullptr;
    LENS_CHECK_ARG(I > 0 && F > 0 && P > 0 && T > 0 && max_streams > 0, "lens_snn_create: bad sizes");
    LENS_CHECK_ARG(I <= 1024 && F <= 992, "lens_snn_create: I=%d F=%d exceed the supported 1024/992", I, F);
    LENS_CHECK_ARG(W_feat && W_out, "lens_snn_create: NULL weights");
    LENS_CHECK_ARG(thr > 0.0f, "lens_snn_create: threshold must be positive");
    cudaStream_t st = as_stream(stream);
    SnnHandle *h = new SnnHandle();
    h->I = I; h->F = F; h->P = P; h->T = T; h->thr = thr; h->vmin = v_min; h->maxB = max_streams;
    h->Fp = (F + kHiddenPad - 1) / kHiddenPad * kHiddenPad;
    cudaGetDevice(&h->device);
#define H_CUDA(call)                                                                   \
    do {                                                                               \
        cudaError_t e__ = (call);                                                      \
        if (e__ != cudaSuccess) {                                                      \
            set_err("lens_snn_create: %s -> %s", #call, cudaGetErrorString(e__));      \
            lens_snn_destroy(h);                                                       \
            return (int)e__;                                                           \
        }                                                                              \
    } while (0)
    H_CUDA(cudaMalloc(&h->Wf_fx, (size_t)I * F * sizeof(int64_t)));
    H_CUDA(cudaMalloc(&h->Wf_scale, (size_t)F * sizeof(float)));
    H_CUDA(cudaMalloc(&h->Wo_fx, (size_t)F * P * sizeof(int64_t)));
    H_CUDA(cudaMalloc(&h->Wo_scale, (size_t)P * sizeof(float)));
    H_CUDA(cudaMalloc(&h->counters, 2 * sizeof(int64_t)));
    H_CUDA(cudaMemsetAsync(h->counters, 0, 2 * sizeof(int64_t), st));
    if (U) {
        H_CUDA(cudaMalloc(&h->U, (size_t)T * I * sizeof(float)));
        H_CUDA(cudaMemcpyAsync(h->U, U, (size_t)T * I * sizeof(float), cudaMemcpyDeviceToDevice, st));
        H_CUDA(cudaMalloc(&h->Uq, (size_t)T * I));
        raster_thresholds_kernel<<<ceil_div(T * I, 256), 256, 0, st>>>(h->U, T * I, h->Uq);
        count_launch();
        H_CUDA(cudaGetLastError());
    }
    H_CUDA(cudaMalloc(&h->v0, (size_t)max_streams * I * sizeof(float)));
    H_CUDA(cudaMalloc(&h->v1, (size_t)max_streams * F * sizeof(float)));
    H_CUDA(cudaMalloc(&h->v2, (size_t)max_streams * P * sizeof(float)));
    H_CUDA(cudaMemsetAsync(h->v0, 0, (size_t)max_streams * I * sizeof(float), st));
    H_CUDA(cudaMemsetAsync(h->v1, 0, (size_t)max_streams * F * sizeof(float), st));
    H_CUDA(cudaMemsetAsync(h->v2, 0, (size_t)max_streams * P * sizeof(float), st));
    weights_to_fixed_kernel<<<F, 256, 0, st>>>(W_feat, F, I, h->Wf_fx, h->Wf_scale, h->counters + 1);
    H_CUDA(cudaGetLastError());
    weights_to_fixed_kernel<<<P, 256, 0, st>>>(W_out, P, F, h->Wo_fx, h->Wo_scale, h->counters + 1);
    H_CUDA(cudaGetLastError());
    if (n_inexact) {   // the one synchronising call of the API (construction time only)
        H_CUDA(cudaMemcpyAsync(n_inexact, h->counters + 1, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
        H_CUDA(cudaStreamSynchronize(st));
    }
#undef H_CUDA
    *handle = h;
    return 0;
}

extern "C" int lens_snn_destroy(void *handle)
{
    if (!handle) return 0;
    SnnHandle *h = static_cast<SnnHandle *>(handle);
    for (auto &t : h->timed) { cudaEventDestroy(t.start); cudaEventDestroy(t.stop); }   // uncollected timings
    h->timed.clear();
    snn_tc_release(h);
    cudaFree(h->Wf_fx); cudaFree(h->Wf_scale); cudaFree(h->Wo_fx); cudaFree(h->Wo_scale);
    cudaFree(h->U); cudaFree(h->Uq); cudaFree(h->v0); cudaFree(h->v1); cudaFree(h->v2);
    cudaFree(h->counters); cudaFree(h->S1); cudaFree(h->ws);
    delete h;
    return 0;
}

extern "C" int lens_snn_reset(void *handle, void *stream)
{
    LENS_CHECK_ARG(handle, "lens_snn_reset: NULL handle");
    SnnHandle *h = static_cast<SnnHandle *>(handle);
    cudaStream_t st = as_stream(stream);
    LENS_CUDA(cudaMemsetAsync(h->v0, 0, (size_t)h->maxB * h->I * sizeof(float), st));
    LENS_CUDA(cudaMemsetAsync(h->v1, 0, (size_t)h->maxB * h->F * sizeof(float), st));
    LENS_CUDA(cudaMemsetAsync(h->v2, 0, (size_t)h->maxB * h->P * sizeof(float), st));
    LENS_CUDA(cudaMemsetAsync(h->counters, 0, sizeof(int64_t), st));
    h->v0_dirty = false;
    return 0;
}

extern "C" int lens_snn_reset_streams(void *handle, const uint8_t *mask, void *stream)
{
    LENS_CHECK_ARG(handle, "lens_snn_reset_streams: NULL handle");
    LENS_CHECK_ARG(mask, "lens_snn_reset_streams: NULL mask");
    SnnHandle *h = static_cast<SnnHandle *>(handle);
    const int blocks = std::min(h->maxB, std::max(sm_count(), 1) * 16);
    reset_streams_kernel<<<blocks, 256, 0, as_stream(stream)>>>(mask, h->maxB, h->I, h->F, h->P, h->v0, h->v1, h->v2);
    LENS_LAUNCH_CHECK();
    return 0;
}

extern "C" int lens_snn_get_state(void *handle, float *v0, float *v1, float *v2, void *stream)
{
    LENS_CHECK_ARG(handle, "lens_snn_get_state: NULL handle");
    SnnHandle *h = static_cast<SnnHandle *>(handle);
    cudaStream_t st = as_stream(stream);
    if (v0) LENS_CUDA(cudaMemcpyAsync(v0, h->v0, (size_t)h->maxB * h->I * sizeof(float), cudaMemcpyDeviceToDevice, st));
    if (v1) LENS_CUDA(cudaMemcpyAsync(v1, h->v1, (size_t)h->maxB * h->F * sizeof(float), cudaMemcpyDeviceToDevice, st));
    if (v2) LENS_CUDA(cudaMemcpyAsync(v2, h->v2, (size_t)h->maxB * h->P * sizeof(float), cudaMemcpyDeviceToDevice, st));
    return 0;
}

extern "C" int lens_snn_get_overflow(void *handle, int64_t *overflow, void *stream)
{
    LENS_CHECK_ARG(handle && overflow, "lens_snn_get_overflow: NULL argument");
    SnnHandle *h = static_cast<SnnHandle *>(handle);
    LENS_CUDA(cudaMemcpyAsync(overflow, h->counters, sizeof(int64_t), cudaMemcpyDeviceToDevice, as_stream(stream)));
    return 0;
}

extern "C" int lens_snn_forward(void *handle, const uint8_t *pooled, int B, int Q, float *counts,
                                uint8_t *hidden_steps, uint8_t *out_steps, int mode, void *stream)
{
    LENS_CHECK_ARG(handle, "lens_snn_forward: NULL handle");
    SnnHandle *h = static_cast<SnnHandle *>(handle);
    LENS_CHECK_ARG(h->U != nullptr, "lens_snn_forward: handle was created without the raster matrix U");
    LENS_CHECK_ARG(B >= 0 && Q >= 0 && B <= h->maxB, "lens_snn_forward: B=%d exceeds max_streams=%d", B, h->maxB);
    LENS_CHECK_ARG(mode >= LENS_SNN_AUTO && mode <= LENS_SNN_TC, "lens_snn_forward: bad mode %d", mode);
    if (B == 0 || Q == 0) return 0;
    LENS_CHECK_ARG(pooled && counts, "lens_snn_forward: NULL buffer");
    LENS_CHECK_ARG((int64_t)Q * h->T <= 2147483647LL, "lens_snn_forward: too many steps");
    return forward_common(h, pooled, nullptr, B, Q * h->T, counts, nullptr, hidden_steps, out_steps,
                          mode, as_stream(stream));
}

extern "C" int lens_snn_forward_range(void *handle, const uint8_t *pooled, int b0, int nb, int Q,
                                      float *counts, uint8_t *hidden_steps, uint8_t *out_steps, int mode,
                                      void *stream)
{
    LENS_CHECK_ARG(handle, "lens_snn_forward_range: NULL handle");
    SnnHandle *h = static_cast<SnnHandle *>(handle);
    LENS_CHECK_ARG(h->U != nullptr, "lens_snn_forward_range: handle was created without the raster matrix U");
    LENS_CHECK_ARG(b0 >= 0 && nb >= 0 && Q >= 0 && b0 + nb <= h->maxB,
                   "lens_snn_forward_range: streams [%d, %d) exceed max_streams=%d", b0, b0 + nb, h->maxB);
    LENS_CHECK_ARG((b0 & 1) == 0, "lens_snn_forward_range: b0 must be even");
    LENS_CHECK_ARG(mode >= LENS_SNN_AUTO && mode <= LENS_SNN_TC, "lens_snn_forward_range: bad mode %d", mode);
    if (nb == 0 || Q == 0) return 0;
    LENS_CHECK_ARG(pooled && counts, "lens_snn_forward_range: NULL buffer");
    LENS_CHECK_ARG((int64_t)Q * h->T <= 2147483647LL, "lens_snn_forward_range: too many steps");
    return forward_common(h, pooled, nullptr, nb, Q * h->T, counts, nullptr, hidden_steps, out_steps, mode,
                          as_stream(stream), b0);
}

extern "C" int lens_snn_forward_streams(void *handle, const uint8_t *pooled, const int32_t *ids, int n, int Q,
                                        float *counts, int mode, void *stream)
{
    LENS_CHECK_ARG(handle, "lens_snn_forward_streams: NULL handle");
    SnnHandle *h = static_cast<SnnHandle *>(handle);
    LENS_CHECK_ARG(h->U != nullptr, "lens_snn_forward_streams: handle was created without the raster matrix U");
    LENS_CHECK_ARG(n >= 0 && Q >= 0, "lens_snn_forward_streams: bad sizes n=%d Q=%d", n, Q);
    LENS_CHECK_ARG(mode >= LENS_SNN_AUTO && mode <= LENS_SNN_TC, "lens_snn_forward_streams: bad mode %d", mode);
    if (n == 0 || Q == 0) return 0;
    LENS_CHECK_ARG(pooled && ids && counts, "lens_snn_forward_streams: NULL buffer");
    LENS_CHECK_ARG((int64_t)Q * h->T <= 2147483647LL, "lens_snn_forward_streams: too many steps");
    cudaStream_t st = as_stream(stream);
    const int need = n + (n & 1);                     // streams are tiled in pairs
    if (need > h->ws_cap) {
        if (h->ws) LENS_CUDA(cudaFree(h->ws));
        h->ws = nullptr; h->ws_cap = 0;
        const size_t bytes = (size_t)need * (h->I + h->F + h->P) * sizeof(float);
        LENS_CUDA(cudaMalloc(&h->ws, bytes));
        LENS_CUDA(cudaMemsetAsync(h->ws, 0, bytes, st));   // the pad row of an odd n is read as a stream's state
        h->ws_cap = need;
    }
    const int blocks = (int)std::min<long long>(3LL * n, (long long)std::max(sm_count(), 1) * 16);
    state_rows_kernel<false><<<blocks, 256, 0, st>>>(ids, n, h->maxB, h->I, h->F, h->P, h->v0, h->v1, h->v2, h->ws,
                                                     h->ws_cap);
    LENS_LAUNCH_CHECK();
    // forward_common reads and writes the state through h->v0 / v1 / v2 (plain kernel parameters): point them at the
    // workspace for the call
    float *v[3] = {h->v0, h->v1, h->v2};
    h->v0 = h->ws;
    h->v1 = h->ws + (size_t)h->ws_cap * h->I;
    h->v2 = h->ws + (size_t)h->ws_cap * (h->I + h->F);
    const int rc = forward_common(h, pooled, nullptr, n, Q * h->T, counts, nullptr, nullptr, nullptr, mode, st);
    h->v0 = v[0]; h->v1 = v[1]; h->v2 = v[2];
    if (rc) return rc;                                // the state is left as it was
    state_rows_kernel<true><<<blocks, 256, 0, st>>>(ids, n, h->maxB, h->I, h->F, h->P, h->v0, h->v1, h->v2, h->ws,
                                                    h->ws_cap);
    LENS_LAUNCH_CHECK();
    return 0;
}

extern "C" int lens_snn_forward_float(void *handle, const float *x, int B, int steps,
                                      float *spikes_out, void *stream)
{
    LENS_CHECK_ARG(handle, "lens_snn_forward_float: NULL handle");
    SnnHandle *h = static_cast<SnnHandle *>(handle);
    LENS_CHECK_ARG(B >= 0 && steps >= 0 && B <= h->maxB, "lens_snn_forward_float: B=%d exceeds max_streams=%d", B, h->maxB);
    if (B == 0 || steps == 0) return 0;
    LENS_CHECK_ARG(x && spikes_out, "lens_snn_forward_float: NULL buffer");
    h->v0_dirty = true;   // arbitrary float input can leave IAF#0 away from rest
    return forward_common(h, nullptr, x, B, steps, nullptr, spikes_out, nullptr, nullptr,
                          LENS_SNN_SIMT, as_stream(stream));
}

extern "C" int lens_snn_set_timing(void *handle, int enable)
{
    LENS_CHECK_ARG(handle, "lens_snn_set_timing: NULL handle");
    SnnHandle *h = static_cast<SnnHandle *>(handle);
    h->timing = enable != 0;
    return 0;
}

extern "C" int lens_snn_get_timing(void *handle, float *feature_ms, float *output_ms,
                                   int64_t *n_feature, int64_t *n_output)
{
    LENS_CHECK_ARG(handle, "lens_snn_get_timing: NULL handle");
    SnnHandle *h = static_cast<SnnHandle *>(handle);
    float ms[2] = {0.f, 0.f};
    int64_t n[2] = {0, 0};
    for (auto &t : h->timed) {
        LENS_CUDA(cudaEventSynchronize(t.stop));
        float e = 0.f;
        LENS_CUDA(cudaEventElapsedTime(&e, t.start, t.stop));
        ms[t.kind] += e; n[t.kind] += 1;
        cudaEventDestroy(t.start); cudaEventDestroy(t.stop);
    }
    h->timed.clear();
    if (feature_ms) *feature_ms = ms[0];
    if (output_ms) *output_ms = ms[1];
    if (n_feature) *n_feature = n[0];
    if (n_output) *n_output = n[1];
    return 0;
}
