// K4: diagonal sequence matching + top-N selection + Recall@N counters.
//
// Replaces lens/run_model.py:248-254 (conv2d(S, eye(L)) / L, transposed) and
// lens/src/metrics.py:213-224 (argsort(0)[-K:] + hit test), called from
// lens/run_model.py:301-302 for N in {1,5,10,15,20,25}.  HBM-bound: every entry of
// the similarity matrix S[B][Q][P] is needed L times, the L reads of a row hit L2
// (one stream's S is Q*P*4 bytes), DRAM sees it once.
//
// D[b][r][q] = (sum_{j<L} S[b][q+j][r+j]) / L : the partial sums are small integers
// (spike counts), exact in fp32 in any order; the one division is IEEE (__fdiv_rn),
// like numpy's float32 / int.  Selection order is (value desc, index desc) -- the
// order np.argsort(kind='stable')[-N:][::-1] produces -- implemented as a 64-bit max
// over keys (rank key(value) << 32 | index), NaN and signed zeros included (f32_rank_key).
#include "common.cuh"

#include <algorithm>
#include <climits>

namespace lens {

constexpr int kMatchThreads = 256;
constexpr int kCandChunk = 2048;
constexpr int kMaxTopN = 64;
constexpr int kUnrollR = 4;       // candidate batches (of 32 places) in flight per warp in the warp-per-query kernel

__device__ __forceinline__ uint32_t f32_orderable(float v)
{
    uint32_t u = __float_as_uint(v);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float f32_from_orderable(uint32_t u)
{
    return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u);
}

// numpy's sort order as a key, for matrices a caller may fill with anything: -0.0 ranks as +0.0 (equal values tie)
// and every NaN, whatever its sign and payload, as one value above +inf (np.sort puts NaNs last).  The key of a NaN
// decodes (f32_from_orderable) to 0x7fffffff; no value has the key 0, which marks an empty top-N slot.  Finite
// non-negative sums (spike counts) get the key f32_orderable gives them.
__device__ __forceinline__ uint32_t f32_rank_key(float v)
{
    return isnan(v) ? 0xffffffffu : f32_orderable(__fadd_rn(v, 0.0f));
}

// One top-N slot from its key (0 = empty slot: -inf / -1).
__device__ __forceinline__ void store_key(unsigned long long k, size_t o, float *__restrict__ top_val,
                                          int32_t *__restrict__ top_idx)
{
    if (k == 0ull) {
        top_val[o] = -INFINITY;
        top_idx[o] = -1;
    } else {
        top_val[o] = f32_from_orderable((uint32_t)(k >> 32));
        top_idx[o] = (int32_t)(uint32_t)(k & 0xffffffffull);
    }
}

// Merges the nr keys of cand (a chunk of places) into the running top-N `best` (descending, 0 = empty slot); all
// arrays in shared memory, called by every thread of the CTA between barriers.
__device__ __forceinline__ void cta_merge_chunk(unsigned long long *cand, unsigned long long *best,
                                                unsigned long long *next_best, unsigned long long *warp_best,
                                                unsigned long long &s_winner, int nr, int N, int tid, int lane,
                                                int warp)
{
    // N rounds of block-wide max over (running best U chunk); keys are unique
    // (distinct place index) so exactly one slot holds the winner.
    for (int n = 0; n < N; ++n) {
        unsigned long long mine = 0ull;
        int mine_pos = -1;
        for (int i = tid; i < N + nr; i += kMatchThreads) {
            const unsigned long long k = (i < N) ? best[i] : cand[i - N];
            if (k > mine) { mine = k; mine_pos = i; }
        }
        unsigned long long wb = mine;
        for (int o = 16; o > 0; o >>= 1) {
            const unsigned long long other = __shfl_xor_sync(0xffffffffu, wb, o);
            wb = other > wb ? other : wb;
        }
        if (lane == 0) warp_best[warp] = wb;
        __syncthreads();
        if (tid == 0) {
            unsigned long long w = 0ull;
            for (int i = 0; i < kMatchThreads / 32; ++i) w = warp_best[i] > w ? warp_best[i] : w;
            s_winner = w;
            next_best[n] = w;
        }
        __syncthreads();
        if (mine != 0ull && mine == s_winner) {
            if (mine_pos < N) best[mine_pos] = 0ull;
            else cand[mine_pos - N] = 0ull;
        }
        __syncthreads();
    }
    for (int i = tid; i < N; i += kMatchThreads) best[i] = next_best[i];
    __syncthreads();
}

// grid = B * Qo.  One CTA scores every database place for one (stream, query).
__global__ void __launch_bounds__(kMatchThreads)
seqmatch_topk_kernel(const float *__restrict__ S, int Q, int P, int L, int N,
                     float *__restrict__ D_out, float *__restrict__ top_val,
                     int32_t *__restrict__ top_idx)
{
    __shared__ unsigned long long cand[kCandChunk];      // keys of the current chunk of places
    __shared__ unsigned long long best[kMaxTopN];        // running top-N (descending)
    __shared__ unsigned long long next_best[kMaxTopN];
    __shared__ unsigned long long warp_best[kMatchThreads / 32];
    __shared__ unsigned long long s_winner;
    const int Qo = Q - L + 1, Po = P - L + 1;
    const int b = blockIdx.x / Qo, q = blockIdx.x - b * Qo;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const float *Sb = S + (size_t)b * Q * P;
    const float fl = (float)L;
    for (int i = tid; i < kMaxTopN; i += kMatchThreads) best[i] = 0ull;   // 0 = empty slot

    for (int r0 = 0; r0 < Po; r0 += kCandChunk) {
        const int nr = min(kCandChunk, Po - r0);
        for (int i = tid; i < nr; i += kMatchThreads) {
            const int r = r0 + i;
            float acc = 0.0f;
            for (int j = 0; j < L; ++j) acc += __ldg(Sb + (size_t)(q + j) * P + (r + j));
            const float d = __fdiv_rn(acc, fl);
            if (D_out) D_out[((size_t)b * Po + r) * Qo + q] = d;
            cand[i] = ((unsigned long long)f32_rank_key(d) << 32) | (uint32_t)r;
        }
        __syncthreads();
        cta_merge_chunk(cand, best, next_best, warp_best, s_winner, nr, N, tid, lane, warp);
    }
    for (int n = tid; n < N; n += kMatchThreads) store_key(best[n], ((size_t)b * Qo + q) * N + n, top_val, top_idx);
}

// ---- warp-per-query variant (N <= 32) ------------------------------------------------------------
// One warp scores one (stream, query): lane i of the warp holds the i-th largest key seen so far.
// Candidates arrive 32 at a time (coalesced loads of the L diagonal terms); a batch is merged only if
// one of its keys beats the current 32nd largest (warp vote), by a 32-element bitonic sort of the batch
// and a bitonic merge with the running list -- shuffles only, no shared memory, no block barriers.
__device__ __forceinline__ unsigned long long shfl_xor_u64(unsigned long long v, int m)
{
    const unsigned lo = __shfl_xor_sync(0xffffffffu, (unsigned)v, m);
    const unsigned hi = __shfl_xor_sync(0xffffffffu, (unsigned)(v >> 32), m);
    return ((unsigned long long)hi << 32) | lo;
}
__device__ __forceinline__ unsigned long long shfl_u64(unsigned long long v, int src)
{
    const unsigned lo = __shfl_sync(0xffffffffu, (unsigned)v, src);
    const unsigned hi = __shfl_sync(0xffffffffu, (unsigned)(v >> 32), src);
    return ((unsigned long long)hi << 32) | lo;
}

// Lane i of `best` holds the i-th largest key of a warp's running list; `key` is one candidate per lane.  Returns the
// top 32 of (list U batch): a bitonic sort of the batch, then a bitonic merge with the list.
__device__ __forceinline__ unsigned long long warp_top32_merge(unsigned long long best, unsigned long long key, int lane)
{
    // bitonic sort of the batch, descending
#pragma unroll
    for (int k = 2; k <= 32; k <<= 1) {
#pragma unroll
        for (int j = k >> 1; j > 0; j >>= 1) {
            const unsigned long long other = shfl_xor_u64(key, j);
            const bool take_max = (((lane & j) == 0) == ((lane & k) == 0));
            key = take_max ? (key > other ? key : other) : (key < other ? key : other);
        }
    }
    // top 32 of (running list U batch): elementwise max against the reversed batch is bitonic
    const unsigned long long rev = shfl_u64(key, 31 - lane);
    unsigned long long c = best > rev ? best : rev;
#pragma unroll
    for (int j = 16; j > 0; j >>= 1) {
        const unsigned long long other = shfl_xor_u64(c, j);
        c = ((lane & j) == 0) ? (c > other ? c : other) : (c < other ? c : other);
    }
    return c;
}

// kSeg = false is the plain one-warp-per-query kernel (40 registers: six CTAs per SM; the segmented instantiation
// needs 48 and would cost the large-batch case a sixth of its resident warps, measured 4.5 -> 7.8 ms on config 3)
template <bool kSeg>
__global__ void __launch_bounds__(256)
seqmatch_topk_warp_kernel(const float *__restrict__ S, long long n_queries, int Q, int P, int L, int N, int n_seg,
                          int seg_len, float *__restrict__ D_out, float *__restrict__ top_val,
                          int32_t *__restrict__ top_idx)
{
    // With n_seg > 1 (few queries, many places) a warp ranks only the places [seg * seg_len, (seg + 1) * seg_len) of
    // its query and writes list `seg` of [n_seg][n_queries][N]; lens_seqmatch_topk merges the lists afterwards.
    const int lane = threadIdx.x & 31;
    const int Qo = Q - L + 1, Po_all = P - L + 1;
    const float fl = (float)L;
    const long long warp0 = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
    const long long n_warps = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long w = warp0; w < (kSeg ? n_queries * n_seg : n_queries); w += n_warps) {
        const int seg = kSeg ? (int)(w / n_queries) : 0;
        const long long g = kSeg ? w - (long long)seg * n_queries : w;
        const int b = (int)(g / Qo), q = (int)(g - (long long)b * Qo);
        const float *Sb = S + ((size_t)b * Q + q) * P;
        const int Po = kSeg ? min(Po_all, (seg + 1) * seg_len) : Po_all;
        unsigned long long best = 0ull;                    // lane i: i-th largest key, 0 = empty
        // kUnrollR batches of 32 candidates per iteration: all their L x kUnrollR loads are issued before
        // the first use, which is what keeps enough bytes in flight per warp to approach the HBM rate
        for (int r0 = kSeg ? seg * seg_len : 0; r0 < Po; r0 += 32 * kUnrollR) {
            float acc[kUnrollR];
#pragma unroll
            for (int u = 0; u < kUnrollR; ++u) acc[u] = 0.0f;
            if (r0 + 32 * kUnrollR <= Po) {
                for (int j = 0; j < L; ++j) {
                    const float *row = Sb + (size_t)j * P + (r0 + lane + j);
#pragma unroll
                    for (int u = 0; u < kUnrollR; ++u) acc[u] += __ldg(row + 32 * u);
                }
            } else {
                for (int j = 0; j < L; ++j) {
                    const float *row = Sb + (size_t)j * P + (r0 + lane + j);
#pragma unroll
                    for (int u = 0; u < kUnrollR; ++u)
                        if (r0 + 32 * u + lane < Po) acc[u] += __ldg(row + 32 * u);
                }
            }
#pragma unroll
            for (int u = 0; u < kUnrollR; ++u) {
                const int r = r0 + 32 * u + lane;
                unsigned long long key = 0ull;
                if (r < Po) {
                    const float d = __fdiv_rn(acc[u], fl);
                    if (D_out) D_out[((size_t)b * Po_all + r) * Qo + q] = d;
                    key = ((unsigned long long)f32_rank_key(d) << 32) | (uint32_t)r;
                }
                const unsigned long long kth = shfl_u64(best, 31);          // current 32nd largest
                if (!__any_sync(0xffffffffu, key > kth)) continue;          // nothing in this batch can enter
                best = warp_top32_merge(best, key, lane);
            }
        }
        if (lane < N) store_key(best, (size_t)w * N + lane, top_val, top_idx);     // w = seg * n_queries + g
    }
}

// ---- streaming K4 (lens_seqmatch_topk_stream) -------------------------------------------------------------------
// New row q of stream b (global row t + q) closes the sequence of rows t + q - L + 1 .. t + q.  Term j of its diagonal
// is new row q - L + 1 + j of S when that is >= 0, else an older row, kept in the stream's ring at slot
// (t + q - L + 1 + j) mod (L - 1).  The choice depends on (q, j) only, so the pointer is warp-uniform per term and
// the loads along the places stay coalesced as in the batch kernels.
struct StreamRows {
    const float *Sq;       // new row q of the stream at position b of S
    const float *ring_b;   // [L-1][P] ring of fleet stream fb
    int n_old;             // terms j < n_old come from the ring
    int slot0;             // ring slot of term 0 (valid rows only: t + q - L + 1 >= 0 there)
    int Lm1, L;
    size_t P;
    __device__ __forceinline__ StreamRows(const float *S, const float *ring, int b, int fb, int Q, int q, int P_, int L_,
                                          long long t)
        : Sq(S + ((size_t)b * Q + q) * P_), ring_b(ring + (size_t)fb * (L_ - 1) * P_), n_old(max(L_ - 1 - q, 0)),
          slot0(L_ > 1 ? (int)((t + q - L_ + 1) % (L_ - 1)) : 0), Lm1(L_ - 1), L(L_), P((size_t)P_) {}
    __device__ __forceinline__ const float *row(int j) const
    {
        if (j < n_old) {
            int s = slot0 + j;
            if (s >= Lm1) s -= Lm1;
            return ring_b + (size_t)s * P;
        }
        return Sq - (size_t)(L - 1 - j) * P;
    }
};

// A row is a sequence end once its stream has seen L rows since its reset (seen saturates at L - 1).
__device__ __forceinline__ bool stream_row_valid(const int32_t *__restrict__ seen, int b, int q, int L)
{
    return __ldg(seen + b) + q + 1 >= L;
}

// Every streaming kernel below serves two kinds of call.  Lockstep (kIdx = false, lens_seqmatch_topk_stream): position
// b of S is fleet stream b and every stream has had t rows.  Indexed (kIdx = true, the *_ids entry points): position b
// is fleet stream fb = ids[b] of n_fleet, with its own row counter rows[fb].  The ring, seen and the place records are
// the fleet's (index fb); S, gt_center, per-push scratch and outputs are by position.  An id outside [0, n_fleet) is
// skipped (-> false).  The lockstep kernels keep their names and code; the indexed ones are separate entry points of
// the same bodies.
template <bool kIdx>
__device__ __forceinline__ bool fleet_stream(const int32_t *__restrict__ ids, const int64_t *__restrict__ rows,
                                             int n_fleet, int b, long long t, int &fb, long long &tb)
{
    fb = b;
    tb = t;
    if (!kIdx) return true;
    fb = __ldg(ids + b);
    if ((unsigned)fb >= (unsigned)n_fleet) return false;
    tb = __ldg(rows + fb);
    return true;
}

// The warp-per-query kernel (N <= 32) over the B * Q new rows, kSeg as in seqmatch_topk_warp_kernel.  A warm-up row
// (not valid) skips the scan and stores an empty list.
template <bool kSeg, bool kIdx>
__device__ __forceinline__ void
stream_warp_topk(const float *__restrict__ S, const float *__restrict__ ring, const int32_t *__restrict__ seen,
                 long long t, const int32_t *__restrict__ ids, const int64_t *__restrict__ rows, int n_fleet,
                 long long n_queries, int Q, int P, int L, int N, int n_seg, int seg_len, float *__restrict__ top_val,
                 int32_t *__restrict__ top_idx)
{
    const int lane = threadIdx.x & 31;
    const int Po_all = P - L + 1;
    const float fl = (float)L;
    const long long warp0 = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
    const long long n_warps = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long w = warp0; w < (kSeg ? n_queries * n_seg : n_queries); w += n_warps) {
        const int seg = kSeg ? (int)(w / n_queries) : 0;
        const long long g = kSeg ? w - (long long)seg * n_queries : w;
        const int b = (int)(g / Q), q = (int)(g - (long long)b * Q);
        const int Po = kSeg ? min(Po_all, (seg + 1) * seg_len) : Po_all;
        unsigned long long best = 0ull;                    // lane i: i-th largest key, 0 = empty
        int fb;
        long long tb;
        if (fleet_stream<kIdx>(ids, rows, n_fleet, b, t, fb, tb) && stream_row_valid(seen, fb, q, L)) {
            const StreamRows rr(S, ring, b, fb, Q, q, P, L, tb);
            for (int r0 = kSeg ? seg * seg_len : 0; r0 < Po; r0 += 32 * kUnrollR) {
                float acc[kUnrollR];
#pragma unroll
                for (int u = 0; u < kUnrollR; ++u) acc[u] = 0.0f;
                if (r0 + 32 * kUnrollR <= Po) {
                    // two diagonal terms per iteration: with one new row per push nearly every load misses L2
                    // (the batch kernel re-reads each row L times from L2), so more bytes must be in flight
#pragma unroll 2
                    for (int j = 0; j < L; ++j) {
                        const float *row = rr.row(j) + (r0 + lane + j);
#pragma unroll
                        for (int u = 0; u < kUnrollR; ++u) acc[u] += __ldg(row + 32 * u);
                    }
                } else {
                    for (int j = 0; j < L; ++j) {
                        const float *row = rr.row(j) + (r0 + lane + j);
#pragma unroll
                        for (int u = 0; u < kUnrollR; ++u)
                            if (r0 + 32 * u + lane < Po) acc[u] += __ldg(row + 32 * u);
                    }
                }
#pragma unroll
                for (int u = 0; u < kUnrollR; ++u) {
                    const int r = r0 + 32 * u + lane;
                    unsigned long long key = 0ull;
                    if (r < Po) key = ((unsigned long long)f32_orderable(__fdiv_rn(acc[u], fl)) << 32) | (uint32_t)r;
                    const unsigned long long kth = shfl_u64(best, 31);
                    if (!__any_sync(0xffffffffu, key > kth)) continue;
                    best = warp_top32_merge(best, key, lane);
                }
            }
        }
        if (lane < N) store_key(best, (size_t)w * N + lane, top_val, top_idx);     // w = seg * n_queries + g
    }
}

template <bool kSeg>
__global__ void __launch_bounds__(256, kSeg ? 1 : 6)
seqmatch_topk_stream_warp_kernel(const float *__restrict__ S, const float *__restrict__ ring,
                                 const int32_t *__restrict__ seen, long long t, long long n_queries, int Q, int P, int L,
                                 int N, int n_seg, int seg_len, float *__restrict__ top_val, int32_t *__restrict__ top_idx)
{
    stream_warp_topk<kSeg, false>(S, ring, seen, t, nullptr, nullptr, 0, n_queries, Q, P, L, N, n_seg, seg_len, top_val,
                                  top_idx);
}

template <bool kSeg>
__global__ void __launch_bounds__(256, kSeg ? 1 : 6)
seqmatch_topk_stream_ids_warp_kernel(const float *__restrict__ S, const float *__restrict__ ring,
                                     const int32_t *__restrict__ seen, const int32_t *__restrict__ ids,
                                     const int64_t *__restrict__ rows, int n_fleet, long long n_queries, int Q, int P,
                                     int L, int N, int n_seg, int seg_len, float *__restrict__ top_val,
                                     int32_t *__restrict__ top_idx)
{
    stream_warp_topk<kSeg, true>(S, ring, seen, 0, ids, rows, n_fleet, n_queries, Q, P, L, N, n_seg, seg_len, top_val,
                                 top_idx);
}

// The CTA-per-query kernel (32 < N <= 64) over the B * Q new rows; grid = B * Q.  (Its name is not pinned, so the
// indexed form is a template argument with ids / rows / n_fleet appended, which the lockstep form never reads.)
template <bool kIdx>
__global__ void __launch_bounds__(kMatchThreads)
seqmatch_topk_stream_kernel(const float *__restrict__ S, const float *__restrict__ ring,
                            const int32_t *__restrict__ seen, long long t, int Q, int P, int L, int N,
                            float *__restrict__ top_val, int32_t *__restrict__ top_idx, const int32_t *__restrict__ ids,
                            const int64_t *__restrict__ rows, int n_fleet)
{
    __shared__ unsigned long long cand[kCandChunk];
    __shared__ unsigned long long best[kMaxTopN];
    __shared__ unsigned long long next_best[kMaxTopN];
    __shared__ unsigned long long warp_best[kMatchThreads / 32];
    __shared__ unsigned long long s_winner;
    const int Po = P - L + 1;
    const int b = blockIdx.x / Q, q = blockIdx.x - b * Q;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const float fl = (float)L;
    for (int i = tid; i < kMaxTopN; i += kMatchThreads) best[i] = 0ull;
    int fb;
    long long tb;
    if (fleet_stream<kIdx>(ids, rows, n_fleet, b, t, fb, tb) && stream_row_valid(seen, fb, q, L)) {   // block-uniform
        const StreamRows rr(S, ring, b, fb, Q, q, P, L, kIdx ? tb : t);
        for (int r0 = 0; r0 < Po; r0 += kCandChunk) {
            const int nr = min(kCandChunk, Po - r0);
            for (int i = tid; i < nr; i += kMatchThreads) {
                const int r = r0 + i;
                float acc = 0.0f;
                for (int j = 0; j < L; ++j) acc += __ldg(rr.row(j) + (r + j));
                cand[i] = ((unsigned long long)f32_orderable(__fdiv_rn(acc, fl)) << 32) | (uint32_t)r;
            }
            __syncthreads();
            cta_merge_chunk(cand, best, next_best, warp_best, s_winner, nr, N, tid, lane, warp);
        }
    }
    for (int n = tid; n < N; n += kMatchThreads) store_key(best[n], ((size_t)b * Q + q) * N + n, top_val, top_idx);
}

// After the match (stream order: it reads the slots this overwrites): the last n_app = min(Q, L - 1) new rows of
// every stream go to their ring slots (t + q) mod (L - 1), and seen advances by Q, saturating at L - 1 (indexed calls:
// in stream_advance_kernel, which runs after every reader of rows).  One CTA per (stream, appended row) at a time,
// 16-byte copies when rows allow them.
template <bool kIdx>
__device__ __forceinline__ void ring_append(const float *__restrict__ S, int B, int Q, int P, int L, long long t,
                                            float *__restrict__ ring, int32_t *__restrict__ seen,
                                            const int32_t *__restrict__ ids, const int64_t *__restrict__ rows,
                                            int n_fleet)
{
    const int Lm1 = L - 1, n_app = min(Q, Lm1);
    const long long n_rows = (long long)B * n_app;
    const bool vec = (P & 3) == 0 && ((reinterpret_cast<uintptr_t>(S) | reinterpret_cast<uintptr_t>(ring)) & 15) == 0;
    for (long long i = blockIdx.x; i < n_rows; i += gridDim.x) {
        const int b = (int)(i / n_app), k = (int)(i - (long long)b * n_app);
        const int q = Q - n_app + k;
        int fb;
        long long tb;
        if (!fleet_stream<kIdx>(ids, rows, n_fleet, b, t, fb, tb)) continue;        // block-uniform
        const float *src = S + ((size_t)b * Q + q) * P;
        float *dst = ring + ((size_t)fb * Lm1 + (int)((tb + q) % Lm1)) * P;
        if (vec) {
            const float4 *s4 = reinterpret_cast<const float4 *>(src);
            float4 *d4 = reinterpret_cast<float4 *>(dst);
            for (int p = threadIdx.x; p < P / 4; p += blockDim.x) d4[p] = __ldg(s4 + p);
        } else {
            for (int p = threadIdx.x; p < P; p += blockDim.x) dst[p] = __ldg(src + p);
        }
        if (!kIdx && k == 0 && threadIdx.x == 0) seen[b] = (int32_t)min((long long)seen[b] + Q, (long long)Lm1);
    }
}

__global__ void __launch_bounds__(256)
ring_append_kernel(const float *__restrict__ S, int B, int Q, int P, int L, long long t, float *__restrict__ ring,
                   int32_t *__restrict__ seen)
{
    ring_append<false>(S, B, Q, P, L, t, ring, seen, nullptr, nullptr, 0);
}

__global__ void __launch_bounds__(256)
ring_append_ids_kernel(const float *__restrict__ S, int B, int Q, int P, int L, float *__restrict__ ring,
                       const int32_t *__restrict__ ids, const int64_t *__restrict__ rows, int n_fleet)
{
    ring_append<true>(S, B, Q, P, L, 0, ring, nullptr, ids, rows, n_fleet);
}

// Indexed calls, last: seen[ids[i]] advances by Q (saturating at L - 1) and rows[ids[i]] by Q.
__global__ void __launch_bounds__(256)
stream_advance_kernel(const int32_t *__restrict__ ids, int n, int n_fleet, int Q, int L, int32_t *__restrict__ seen,
                      int64_t *__restrict__ rows)
{
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int fb = ids[i];
        if ((unsigned)fb >= (unsigned)n_fleet) continue;
        seen[fb] = (int32_t)min((long long)seen[fb] + Q, (long long)(L - 1));
        rows[fb] += Q;
    }
}

// Final merge of per-shard top-N lists (place-sharded database, BASELINE config 5): every rank ranks its own
// range of places, the W lists of a query are all-gathered, and the global top-N is the N best of their
// union under the same order (value desc, place index desc).  One warp per query; the <= W*N candidate keys
// sit in registers (kMergeSlots per lane), N rounds of warp-wide 64-bit max.
constexpr int kMergeSlots = 16;      // W * N <= 32 * kMergeSlots

__global__ void __launch_bounds__(256) topn_merge_kernel(const float *__restrict__ val, const int32_t *__restrict__ idx,
                                                         int W, long long M, int N, float *__restrict__ out_val,
                                                         int32_t *__restrict__ out_idx)
{
    const int lane = threadIdx.x & 31;
    const long long m = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
    if (m >= M) return;
    const int n_cand = W * N;
    unsigned long long key[kMergeSlots];
#pragma unroll
    for (int s = 0; s < kMergeSlots; ++s) {
        const int c = s * 32 + lane;
        key[s] = 0ull;
        if (c < n_cand) {
            const int w = c / N, n = c - w * N;
            const size_t o = ((size_t)w * M + m) * N + n;
            const int32_t i = idx[o];
            if (i >= 0) key[s] = ((unsigned long long)f32_rank_key(val[o]) << 32) | (uint32_t)i;
        }
    }
    for (int n = 0; n < N; ++n) {
        unsigned long long mine = 0ull;
#pragma unroll
        for (int s = 0; s < kMergeSlots; ++s) mine = key[s] > mine ? key[s] : mine;
        unsigned long long best = mine;
        for (int o = 16; o > 0; o >>= 1) {
            const unsigned long long other = shfl_xor_u64(best, o);
            best = other > best ? other : best;
        }
        if (best != 0ull && mine == best) {            // keys are unique (distinct place indices): one owner
#pragma unroll
            for (int s = 0; s < kMergeSlots; ++s)
                if (key[s] == best) key[s] = 0ull;
        }
        if (lane == 0) {
            const size_t o = (size_t)m * N + n;
            out_val[o] = best ? f32_from_orderable((uint32_t)(best >> 32)) : -INFINITY;
            out_idx[o] = best ? (int32_t)(uint32_t)(best & 0xffffffffull) : -1;
        }
    }
}

struct RecallParams {
    const int32_t *top_idx;
    int B, Qo, Po, N;
    const uint8_t *gt_dense;
    int64_t gt_stream_stride;
    const int32_t *gt_center;
    int gt_tol;
    int ns[8];
    int n_ns;
    unsigned long long *hits, *n_valid;
};

// One thread per (stream, query).  metrics.py:214-216 drops queries without any
// positive; :218-224 counts a query as recalled when one of its K best is positive.
__global__ void __launch_bounds__(256) recall_kernel(RecallParams p)
{
    __shared__ unsigned int s_hits[8];
    __shared__ unsigned int s_valid;
    if (threadIdx.x < 8) s_hits[threadIdx.x] = 0;
    if (threadIdx.x == 0) s_valid = 0;
    __syncthreads();
    const int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (g < (int64_t)p.B * p.Qo) {
        const int b = (int)(g / p.Qo), q = (int)(g - (int64_t)b * p.Qo);
        const int32_t *ti = p.top_idx + (size_t)g * p.N;
        bool valid;
        int first_hit = INT_MAX;   // rank of the best-ranked positive among the top N
        if (p.gt_dense) {
            const uint8_t *gt = p.gt_dense + (size_t)b * p.gt_stream_stride;
            valid = false;
            for (int r = 0; r < p.Po; ++r) valid |= gt[(size_t)r * p.Qo + q] != 0;
            if (valid)
                for (int n = 0; n < p.N; ++n) {
                    const int r = ti[n];
                    if (r >= 0 && gt[(size_t)r * p.Qo + q] != 0) { first_hit = n; break; }
                }
        } else {
            const int c = p.gt_center[g];
            valid = c >= 0;
            if (valid)
                for (int n = 0; n < p.N; ++n) {
                    const int r = ti[n];
                    if (r >= 0 && abs(r - c) <= p.gt_tol) { first_hit = n; break; }
                }
        }
        if (valid) {
            atomicAdd(&s_valid, 1u);
            for (int i = 0; i < p.n_ns; ++i)
                if (first_hit < p.ns[i]) atomicAdd(&s_hits[i], 1u);
        }
    }
    __syncthreads();
    if (threadIdx.x < p.n_ns && s_hits[threadIdx.x])
        atomicAdd(p.hits + threadIdx.x, (unsigned long long)s_hits[threadIdx.x]);
    if (threadIdx.x == 0 && s_valid) atomicAdd(p.n_valid, (unsigned long long)s_valid);
}

// Tie-aware bounds of Recall@K (SURVEY H5): lens/src/metrics.py:218 ranks every query column with numpy's
// default argsort, which is free to order equal similarities either way, so the reference's own number
// is only defined up to the choice among ties.  One warp per query column walks the distinct similarity
// values from the top: g = entries strictly above the current value (all of them are in any top-K with
// K > g), c = entries equal to it.  For the K whose K-th entry falls on this value (g < K <= g + c):
//   certain hit  <=> a positive lies strictly above, or the K - g picks among the c ties cannot avoid one
//   possible hit <=> a positive lies strictly above or among the ties.
struct BoundsParams {
    const float *D;            // [Po][Qo]
    const uint8_t *GT;         // [Po][Qo]
    int Po, Qo, n_ns;
    int ns[8];
    unsigned long long *lo, *hi, *n_valid;
};

__global__ void __launch_bounds__(256) recall_bounds_kernel(BoundsParams p)
{
    const int lane = threadIdx.x & 31;
    const int q = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (q >= p.Qo) return;
    int any = 0;
    for (int r = lane; r < p.Po; r += 32) any |= p.GT[(size_t)r * p.Qo + q] != 0;
    if (!__any_sync(0xffffffffu, any)) return;                   // metrics.py:214-216: no positive, dropped
    const int kmax = p.ns[p.n_ns - 1];
    // the levels are the distinct rank keys (f32_rank_key: all NaNs one level above +inf, -0.0 == +0.0), walked
    // from the top; no value has the key 0, so m = 0 below means that no entry is left
    unsigned long long cur = 1ull << 32;                          // above every key
    int g = 0, gpos = 0, next_k = 0;                              // next_k: first K not decided yet
    unsigned lo_mask = 0u, hi_mask = 0u;
    while (next_k < p.n_ns) {
        // largest key strictly below `cur`, its multiplicity and its positives
        unsigned m = 0u;
        for (int r = lane; r < p.Po; r += 32) {
            const unsigned k = f32_rank_key(p.D[(size_t)r * p.Qo + q]);
            if (k < cur) m = max(m, k);
        }
        m = __reduce_max_sync(0xffffffffu, m);
        int c = 0, cpos = 0;
        for (int r = lane; r < p.Po; r += 32) {
            if (f32_rank_key(p.D[(size_t)r * p.Qo + q]) == m) { ++c; cpos += p.GT[(size_t)r * p.Qo + q] != 0; }
        }
        c = __reduce_add_sync(0xffffffffu, c);
        cpos = __reduce_add_sync(0xffffffffu, cpos);
        if (c == 0) {
            // the column is exhausted (K > Po): everything ranked so far is certain
            for (; next_k < p.n_ns; ++next_k)
                if (gpos > 0) { lo_mask |= 1u << next_k; hi_mask |= 1u << next_k; }
            break;
        }
        for (; next_k < p.n_ns && p.ns[next_k] <= g + c; ++next_k) {
            const int room = p.ns[next_k] - g;                    // picks among the c ties
            if (gpos > 0) { lo_mask |= 1u << next_k; hi_mask |= 1u << next_k; }
            else if (cpos > 0) {
                hi_mask |= 1u << next_k;
                if (c - cpos < room) lo_mask |= 1u << next_k;
            }
        }
        g += c; gpos += cpos; cur = m;
        if (g >= kmax) break;
    }
    if (lane == 0) {
        atomicAdd(p.n_valid, 1ull);
        for (int i = 0; i < p.n_ns; ++i) {
            if (lo_mask >> i & 1u) atomicAdd(p.lo + i, 1ull);
            if (hi_mask >> i & 1u) atomicAdd(p.hi + i, 1ull);
        }
    }
}

// Threshold i of np.linspace(start, stop, n) with start = max, stop = min of createPR's values.  numpy (>= 2.0)
// evaluates it in the dtype of those values: float64 for float64, integer and bool matrices (f64 != 0), float32 for
// float32 ones.  Each operation is rounded on its own, like numpy's sequence of array operations, hence the
// explicit intrinsics (no FMA contraction):
//   step = (stop - start) / (n - 1);  y_i = i * step + start,  or, when step underflows to 0 (denormal ranges),
//   y_i = (i / (n - 1)) * (stop - start) + start;  the last element is stop.
// The float32 threshold is returned widened to float64, which is exact, so `(double)v >= t` is the float32
// comparison numpy makes.  The float64 branch never sees step == 0 unless start == stop, where both forms give start.
__device__ __forceinline__ double pr_threshold(int i, int n, float start, float stop, bool f64)
{
    if (f64) {
        const double step = __ddiv_rn(__dsub_rn((double)stop, (double)start), (double)(n - 1));
        return (i == n - 1) ? (double)stop : __dadd_rn(__dmul_rn((double)i, step), (double)start);
    }
    const float div = (float)(n - 1), delta = __fsub_rn(stop, start);
    const float step = __fdiv_rn(delta, div);
    if (i == n - 1) return (double)stop;
    if (step == 0.0f) return (double)__fadd_rn(__fmul_rn(__fdiv_rn((float)i, div), delta), start);
    return (double)__fadd_rn(__fmul_rn((float)i, step), start);
}

// createPR, matching = 'single' (lens/src/metrics.py:21-139): one CTA, columns strided over threads.
// best[q] / hit[q] live in shared memory (Qo <= 8192).
__global__ void __launch_bounds__(256) pr_counts_kernel(const float *__restrict__ S, const uint8_t *__restrict__ GT,
                                                        int Po, int Qo, int n_thresh, int thresh_f64,
                                                        unsigned long long *__restrict__ tp,
                                                        unsigned long long *__restrict__ fp,
                                                        unsigned long long *__restrict__ gtp)
{
    extern __shared__ float s_best[];                       // [Qo] best similarity per query
    uint8_t *s_hit = reinterpret_cast<uint8_t *>(s_best + Qo);   // [Qo] GT at the best match
    __shared__ float s_max[8], s_min[8];
    __shared__ unsigned int s_gtp;
    if (threadIdx.x == 0) s_gtp = 0;
    __syncthreads();
    float vmax = -INFINITY, vmin = INFINITY;
    unsigned int my_gtp = 0;
    bool my_nan = false;
    for (int q = threadIdx.x; q < Qo; q += blockDim.x) {
        float best = -INFINITY;
        int arg = 0;
        bool any = false;
        for (int r = 0; r < Po; ++r) {
            const float v = S[(size_t)r * Qo + q];
            // strict: the first maximum wins, and the first NaN beats everything (np.argmax / np.max)
            if (v > best || (isnan(v) && !isnan(best))) { best = v; arg = r; }
            any |= GT[(size_t)r * Qo + q] != 0;
        }
        s_best[q] = best;
        s_hit[q] = GT[(size_t)arg * Qo + q] != 0;
        my_gtp += any;
        my_nan |= isnan(best);
        vmax = fmaxf(vmax, best); vmin = fminf(vmin, best);
    }
    for (int o = 16; o > 0; o >>= 1) {
        vmax = fmaxf(vmax, __shfl_xor_sync(0xffffffffu, vmax, o));
        vmin = fminf(vmin, __shfl_xor_sync(0xffffffffu, vmin, o));
        my_gtp += __shfl_xor_sync(0xffffffffu, my_gtp, o);
    }
    if ((threadIdx.x & 31) == 0) { s_max[threadIdx.x >> 5] = vmax; s_min[threadIdx.x >> 5] = vmin; atomicAdd(&s_gtp, my_gtp); }
    const bool any_nan = __syncthreads_or(my_nan);
    for (int i = 0; i < 8; ++i) { vmax = fmaxf(vmax, s_max[i]); vmin = fminf(vmin, s_min[i]); }
    if (any_nan) vmax = vmin = __int_as_float(0x7fffffff);     // np.max / np.min of the best values: NaN
    for (int i = threadIdx.x; i < n_thresh; i += blockDim.x) {
        const double t = pr_threshold(i, n_thresh, vmax, vmin, thresh_f64 != 0);
        unsigned long long a = 0, b = 0;
        for (int q = 0; q < Qo; ++q) {
            if ((double)s_best[q] >= t) { if (s_hit[q]) ++a; else ++b; }
        }
        tp[i] = a; fp[i] = b;
    }
    if (threadIdx.x == 0) gtp[0] = s_gtp;
}

// createPR, matching = 'multi' (lens/src/metrics.py:63-91): every entry of the matrix counts.  Pass 1: extreme
// values (as order-preserving integers) and the number of ground-truth positives; pass 2: one CTA per (threshold,
// slice of the matrix) counts the entries >= threshold that are / are not positives.  Thresholds as in the
// 'single' kernel (pr_threshold).
__global__ void __launch_bounds__(256) pr_multi_minmax_kernel(const float *__restrict__ S, const uint8_t *__restrict__ GT,
                                                              long long n, unsigned int *__restrict__ mm,
                                                              unsigned long long *__restrict__ gtp)
{
    unsigned int vmax = 0u, vmin = 0xffffffffu;
    unsigned long long pos = 0;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const unsigned int k = f32_orderable(S[i]);
        vmax = max(vmax, k); vmin = min(vmin, k);
        pos += GT[i] != 0;
    }
    vmax = __reduce_max_sync(0xffffffffu, vmax);
    vmin = __reduce_min_sync(0xffffffffu, vmin);
    for (int o = 16; o > 0; o >>= 1) pos += __shfl_xor_sync(0xffffffffu, pos, o);
    if ((threadIdx.x & 31) == 0) {
        atomicMax(mm, vmax);
        atomicMin(mm + 1, vmin);
        if (pos) atomicAdd(gtp, pos);
    }
}

__global__ void __launch_bounds__(256) pr_multi_counts_kernel(const float *__restrict__ S, const uint8_t *__restrict__ GT,
                                                              long long n, int n_thresh, int thresh_f64,
                                                              const unsigned int *__restrict__ mm,
                                                              unsigned long long *__restrict__ tp,
                                                              unsigned long long *__restrict__ fp)
{
    const int i = blockIdx.x;
    // np.max and np.min are NaN as soon as S holds a NaN.  A NaN is one of the two extremes (above +inf or below -inf by
    // its sign bit); as the minimum it makes every threshold NaN by itself, as the maximum it needs this.
    const float vmax = f32_from_orderable(mm[0]), vmin = isnan(vmax) ? vmax : f32_from_orderable(mm[1]);
    const double t = pr_threshold(i, n_thresh, vmax, vmin, thresh_f64 != 0);
    const long long per = ceil_div64(n, gridDim.y), e0 = per * blockIdx.y, e1 = min(n, e0 + per);
    unsigned long long a = 0, b = 0;
    for (long long e = e0 + threadIdx.x; e < e1; e += blockDim.x)
        if ((double)S[e] >= t) { if (GT[e]) ++a; else ++b; }
    for (int o = 16; o > 0; o >>= 1) {
        a += __shfl_xor_sync(0xffffffffu, a, o);
        b += __shfl_xor_sync(0xffffffffu, b, o);
    }
    if ((threadIdx.x & 31) == 0) {
        if (a) atomicAdd(tp + i, a);
        if (b) atomicAdd(fp + i, b);
    }
}

// ---- fleet precision-recall (lens_seqpr_scan / lens_seqpr_counts) --------------------------------------------
// createPR's counts over the sequence-matched matrices of B streams, recomputed from S as K4 does (D is never
// written).  The columns of the fleet are those of np.concatenate([D_b.T] or [D_b], axis=1): per place (b, p),
// per query (b, q), or every entry (multi).  Scan: one read of S; per-column records, the extremes as
// order-preserving keys {max, ~min} (merged with atomicMax, so groups and ranks combine by max) and gtp.
// Count: the thresholds of the merged extremes in shared memory, every record (or entry, re-read) binned once,
// then prefix sums into tp / fp.
constexpr int kPrPlace = LENS_SEQPR_PLACE, kPrQuery = LENS_SEQPR_QUERY, kPrMulti = LENS_SEQPR_MULTI;
constexpr int kPrTile = 32 * kUnrollR;    // places per warp item
constexpr int kPrMaxThresh = 4096;        // 12 B per threshold of shared memory: table + two histograms

struct SeqPrArgs {
    const float *S;
    int B, Q, P, L, Qo, Po;
    const uint8_t *gt_dense;
    int64_t gt_stride;
    const int32_t *gt_center;
    int gt_tol;
    float *rec_val;                  // per place: [B * Po] best value over the queries
    unsigned long long *rec_key;     // per query: [B * Qo] orderable(best) << 32 | ~place
    uint8_t *rec_flag;               // [B * Po] GT at the first maximum (per place) / [B * Qo] any positive (per query)
    unsigned long long *ext;         // {max key, ~min key}
    unsigned long long *gtp;
    int n_thresh;
    unsigned long long *hist;        // count pass: [2][n_thresh] positives | negatives per bin
};

__device__ __forceinline__ bool seqpr_positive(const SeqPrArgs &a, int b, int p, int q, int center)
{
    if (a.gt_dense) return __ldg(a.gt_dense + (size_t)b * a.gt_stride + (size_t)p * a.Qo + q) != 0;
    return center >= 0 && abs(p - center) <= a.gt_tol;
}

__device__ __forceinline__ int seqpr_center(const SeqPrArgs &a, int b, int q)
{
    return a.gt_dense ? 0 : __ldg(a.gt_center + (size_t)b * a.Qo + q);
}

// D_b[p][q] for the places p0 + 32 u + lane of one tile, as K4 computes it (exact integer partial sums, one IEEE
// division); loads coalesced along the places, four batches of L terms in flight.
__device__ __forceinline__ void seqpr_tile_values(const SeqPrArgs &a, const float *Sb, int q, int p0, int lane,
                                                  float (&d)[kUnrollR])
{
    float acc[kUnrollR];
#pragma unroll
    for (int u = 0; u < kUnrollR; ++u) acc[u] = 0.0f;
    const float *base = Sb + (size_t)q * a.P + p0 + lane;
    if (p0 + kPrTile <= a.Po) {
        for (int j = 0; j < a.L; ++j) {
            const float *row = base + (size_t)j * a.P + j;
#pragma unroll
            for (int u = 0; u < kUnrollR; ++u) acc[u] += __ldg(row + 32 * u);
        }
    } else {
        for (int j = 0; j < a.L; ++j) {
            const float *row = base + (size_t)j * a.P + j;
#pragma unroll
            for (int u = 0; u < kUnrollR; ++u)
                if (p0 + 32 * u + lane < a.Po) acc[u] += __ldg(row + 32 * u);
        }
    }
    const float fl = (float)a.L;
#pragma unroll
    for (int u = 0; u < kUnrollR; ++u) d[u] = __fdiv_rn(acc[u], fl);
}

// Warp-wide merge of a warp's extremes (orderable keys, 0 / ~0 = none) and positives into the caller's totals.
__device__ __forceinline__ void seqpr_merge_extremes(const SeqPrArgs &a, unsigned kmax, unsigned kmin,
                                                     unsigned long long pos, int lane)
{
    kmax = __reduce_max_sync(0xffffffffu, kmax);
    kmin = __reduce_min_sync(0xffffffffu, kmin);
    for (int o = 16; o > 0; o >>= 1) pos += __shfl_xor_sync(0xffffffffu, pos, o);
    if (lane == 0) {
        if (kmax) {
            atomicMax(a.ext, (unsigned long long)kmax);
            atomicMax(a.ext + 1, (unsigned long long)(~kmin));
        }
        if (pos) atomicAdd(a.gtp, pos);
    }
}

// Scan pass.  One warp per (stream, tile of kPrTile places), queries in ascending order.  48 registers (five CTAs
// per SM): capped at 40 like K4, the per-place and multi forms spill.
template <int kMode>
__global__ void __launch_bounds__(256, 5) seqpr_scan_kernel(SeqPrArgs a)
{
    const int lane = threadIdx.x & 31;
    const long long warp0 = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
    const long long n_warps = ((long long)gridDim.x * blockDim.x) >> 5;
    const long long n_tiles = ceil_div(a.Po, kPrTile), n_items = (long long)a.B * n_tiles;
    unsigned kmax = 0u, kmin = 0xffffffffu;
    unsigned long long pos = 0;
    for (long long w = warp0; w < n_items; w += n_warps) {
        const int b = (int)(w / n_tiles), p0 = (int)(w - (long long)b * n_tiles) * kPrTile;
        const float *Sb = a.S + (size_t)b * a.Q * a.P;
        float best[kUnrollR];
        bool hit[kUnrollR], any[kUnrollR];
#pragma unroll
        for (int u = 0; u < kUnrollR; ++u) { best[u] = 0.0f; hit[u] = any[u] = false; }
        for (int q = 0; q < a.Qo; ++q) {
            float d[kUnrollR];
            seqpr_tile_values(a, Sb, q, p0, lane, d);
            const int c = seqpr_center(a, b, q);
            unsigned long long kq = 0ull;
            bool anyq = false;
#pragma unroll
            for (int u = 0; u < kUnrollR; ++u) {
                const int p = p0 + 32 * u + lane;
                if (p >= a.Po) continue;
                const bool g = seqpr_positive(a, b, p, q, c);
                if (kMode == kPrPlace) {
                    if (q == 0 || d[u] > best[u]) { best[u] = d[u]; hit[u] = g; }   // strict: first maximum
                    any[u] |= g;
                } else if (kMode == kPrQuery) {
                    // ~p: among equal values the lowest place wins (np.argmax); -0 keyed as +0, which numpy ties
                    const unsigned long long k =
                        ((unsigned long long)f32_orderable(__fadd_rn(d[u], 0.0f)) << 32) | (uint32_t)~p;
                    kq = k > kq ? k : kq;
                    anyq |= g;
                } else {
                    const unsigned o = f32_orderable(d[u]);
                    kmax = max(kmax, o); kmin = min(kmin, o);
                    pos += g;
                }
            }
            if (kMode == kPrQuery) {
                for (int o = 16; o > 0; o >>= 1) {
                    const unsigned long long other = shfl_xor_u64(kq, o);
                    kq = other > kq ? other : kq;
                }
                anyq = __any_sync(0xffffffffu, anyq);
                if (lane == 0) {
                    const size_t r = (size_t)b * a.Qo + q;
                    atomicMax(a.rec_key + r, kq);
                    if (anyq) a.rec_flag[r] = 1;
                }
            }
        }
        if (kMode == kPrPlace) {
#pragma unroll
            for (int u = 0; u < kUnrollR; ++u) {
                const int p = p0 + 32 * u + lane;
                if (p >= a.Po) continue;
                const size_t r = (size_t)b * a.Po + p;
                a.rec_val[r] = best[u];
                a.rec_flag[r] = hit[u];
                const unsigned o = f32_orderable(best[u]);
                kmax = max(kmax, o); kmin = min(kmin, o);
                pos += any[u];
            }
        }
    }
    if (kMode != kPrQuery) seqpr_merge_extremes(a, kmax, kmin, pos, lane);
}

// Per-query records are final only once every tile has merged into them: their extremes and gtp come after.
__global__ void __launch_bounds__(256) seqpr_query_extremes_kernel(SeqPrArgs a)
{
    const long long n = (long long)a.B * a.Qo;
    unsigned kmax = 0u, kmin = 0xffffffffu;
    unsigned long long pos = 0;
    for (long long i0 = blockIdx.x * (long long)blockDim.x; i0 < n; i0 += (long long)gridDim.x * blockDim.x) {
        const long long i = i0 + threadIdx.x;
        if (i < n) {
            const unsigned o = (unsigned)(a.rec_key[i] >> 32);
            kmax = max(kmax, o); kmin = min(kmin, o);
            pos += a.rec_flag[i];
        }
    }
    seqpr_merge_extremes(a, kmax, kmin, pos, threadIdx.x & 31);
}

// Bin of value v: the first k <= n - 2 with y[k] <= v, else n - 1.  The float32 table is non-increasing over
// 0 .. n - 2 (each step a monotone operation, monotonically rounded); only y[n - 1] = stop can break the order, and
// every value is >= stop (the minimum of the very values binned), so threshold n - 1 counts everything.
__device__ __forceinline__ int seqpr_bin(const float *y, int n, float v)
{
    int lo = 0, hi = n - 1;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (y[mid] <= v) hi = mid; else lo = mid + 1;
    }
    return lo;
}

// Every lane of the warp calls this; lanes with the same (bin, hit) add once (spike-count D takes few values).
__device__ __forceinline__ void seqpr_add(unsigned *h, int n, bool valid, int bin, bool hit, int lane)
{
    const unsigned key = valid ? ((unsigned)bin << 1 | (unsigned)hit) : 0xffffffffu;
    const unsigned peers = __match_any_sync(0xffffffffu, key);
    if (valid && __ffs(peers) - 1 == lane) atomicAdd(h + (hit ? 0 : n) + bin, (unsigned)__popc(peers));
}

// Count pass: histograms per CTA in shared memory ([n] thresholds, [2][n] counts), merged into a.hist.
template <int kMode>
__global__ void __launch_bounds__(256, 5) seqpr_count_kernel(SeqPrArgs a)
{
    extern __shared__ float s_y[];
    unsigned *s_h = reinterpret_cast<unsigned *>(s_y + a.n_thresh);
    const int n = a.n_thresh, lane = threadIdx.x & 31;
    const float start = f32_from_orderable((uint32_t)a.ext[0]), stop = f32_from_orderable(~(uint32_t)a.ext[1]);
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        s_y[i] = (float)pr_threshold(i, n, start, stop, false);
        s_h[i] = s_h[n + i] = 0u;
    }
    __syncthreads();
    if (kMode == kPrMulti) {
        const long long warp0 = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
        const long long n_warps = ((long long)gridDim.x * blockDim.x) >> 5;
        const long long n_tiles = ceil_div(a.Po, kPrTile), n_items = (long long)a.B * n_tiles;
        for (long long w = warp0; w < n_items; w += n_warps) {
            const int b = (int)(w / n_tiles), p0 = (int)(w - (long long)b * n_tiles) * kPrTile;
            const float *Sb = a.S + (size_t)b * a.Q * a.P;
            for (int q = 0; q < a.Qo; ++q) {
                float d[kUnrollR];
                seqpr_tile_values(a, Sb, q, p0, lane, d);
                const int c = seqpr_center(a, b, q);
#pragma unroll
                for (int u = 0; u < kUnrollR; ++u) {
                    const int p = p0 + 32 * u + lane;
                    const bool valid = p < a.Po;
                    const bool g = valid && seqpr_positive(a, b, p, q, c);
                    seqpr_add(s_h, n, valid, valid ? seqpr_bin(s_y, n, d[u]) : 0, g, lane);
                }
            }
        }
    } else {
        // records: four per thread and iteration, loads first; every lane runs the same number of iterations
        constexpr int kPer = 4;
        const long long n_rec = (long long)a.B * (kMode == kPrPlace ? a.Po : a.Qo);
        const long long stride = (long long)gridDim.x * blockDim.x;
        for (long long i0 = blockIdx.x * (long long)blockDim.x; i0 < n_rec; i0 += stride * kPer) {
            float v[kPer];
            bool g[kPer], valid[kPer];
#pragma unroll
            for (int k = 0; k < kPer; ++k) {
                const long long i = i0 + k * stride + threadIdx.x;
                valid[k] = i < n_rec;
                v[k] = 0.0f; g[k] = false;
                if (!valid[k]) continue;
                if (kMode == kPrPlace) {
                    v[k] = a.rec_val[i];
                    g[k] = a.rec_flag[i] != 0;
                } else {
                    const unsigned long long key = a.rec_key[i];
                    const int b = (int)(i / a.Qo), q = (int)(i - (long long)b * a.Qo);
                    v[k] = f32_from_orderable((uint32_t)(key >> 32));
                    g[k] = seqpr_positive(a, b, (int)~(uint32_t)key, q, seqpr_center(a, b, q));
                }
            }
#pragma unroll
            for (int k = 0; k < kPer; ++k) seqpr_add(s_h, n, valid[k], valid[k] ? seqpr_bin(s_y, n, v[k]) : 0, g[k], lane);
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 2 * n; i += blockDim.x)
        if (s_h[i]) atomicAdd(a.hist + i, (unsigned long long)s_h[i]);
}

// tp[i] += positives with bin <= i, fp[i] likewise (the values >= threshold i).  Warp 0: tp, warp 1: fp.
__global__ void __launch_bounds__(64) seqpr_prefix_kernel(const unsigned long long *__restrict__ hist, int n,
                                                          unsigned long long *__restrict__ tp,
                                                          unsigned long long *__restrict__ fp)
{
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const unsigned long long *h = hist + (size_t)w * n;
    unsigned long long *out = w ? fp : tp, carry = 0;
    for (int base = 0; base < n; base += 32) {
        const int i = base + lane;
        unsigned long long v = i < n ? h[i] : 0ull;
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long up = shfl_u64(v, max(lane - o, 0));
            if (lane >= o) v += up;
        }
        v += carry;
        if (i < n) out[i] += v;
        carry = shfl_u64(v, 31);
    }
}

// ---- session precision-recall of a live fleet (lens_seqpr_stream_*) -------------------------------------------
// Every D entry is __fdiv_rn(acc, L) with acc an integer-valued sum of spike counts; for an integer 0 <= k < 2^16,
// fl(k / L) is strictly increasing in k, so a session's createPR curve depends only on the k of its entries:
// place mode keeps one record per (stream, place) (the first maximum over the session's rows), query and multi mode
// a histogram over k.  Accumulators start with a header {n_bad, gtp} (u64); zeroed memory is an empty session.
constexpr int kStreamBins = LENS_SEQPR_STREAM_BINS;
constexpr int kStreamShBins = 2048;       // k below this is counted in shared memory first (spike sums are small)

struct SeqPrStreamArgs {
    const float *S, *ring;
    const int32_t *seen;
    long long t;
    int B, Q, P, L, Po;
    const int32_t *gt_center;            // [B][Q]
    int gt_tol;
    unsigned *rec;                       // place: [B][Po] records (k + 1) << 2 | hit at first max << 1 | any positive
    unsigned long long *key;             // query: [B][Q] per-push scratch, k << 32 | ~p of the row's first maximum
    unsigned long long *hist;            // multi: [2][kStreamBins], positives first
    unsigned long long *multi_gtp;
    unsigned long long *bad[3];          // n_bad of each tracked accumulator, NULL when the mode is not tracked
};

// One count of (k, hit) per valid lane; lanes with the same (k, hit) add once.  Small k goes to the block's shared
// histogram s_h [2][kStreamShBins], the rare large k straight to the global one g_h [2][kStreamBins].
__device__ __forceinline__ void stream_hist_add(unsigned *s_h, unsigned long long *g_h, bool valid, int k, bool hit,
                                                int lane)
{
    const unsigned key = valid ? ((unsigned)k << 1 | (unsigned)hit) : 0xffffffffu;
    const unsigned peers = __match_any_sync(0xffffffffu, key);
    if (valid && __ffs(peers) - 1 == lane) {
        if (k < kStreamShBins) atomicAdd(s_h + (hit ? 0 : kStreamShBins) + k, (unsigned)__popc(peers));
        else atomicAdd(g_h + (hit ? 0 : kStreamBins) + k, (unsigned long long)__popc(peers));
    }
}

__device__ __forceinline__ void stream_hist_flush(const unsigned *s_h, unsigned long long *g_h)
{
    __syncthreads();
    for (int i = threadIdx.x; i < 2 * kStreamShBins; i += blockDim.x)
        if (s_h[i]) atomicAdd(g_h + (i < kStreamShBins ? i : kStreamBins + i - kStreamShBins), (unsigned long long)s_h[i]);
}

// One warp per (stream, kPrTile places), the push's new rows in order; warm-up rows are skipped.  The diagonal terms
// come through StreamRows as in seqmatch_topk_stream_warp_kernel, so this runs before that call (same t, same seen).
// kIdx as in the streaming match: place records by fleet stream, gt_center and the query scratch by position.
template <bool kIdx>
__device__ __forceinline__ void stream_accumulate(SeqPrStreamArgs a, const int32_t *__restrict__ ids,
                                                  const int64_t *__restrict__ rows_of, int n_fleet)
{
    extern __shared__ unsigned s_h[];    // multi mode: [2][kStreamShBins]
    const int lane = threadIdx.x & 31;
    if (a.hist) {
        for (int i = threadIdx.x; i < 2 * kStreamShBins; i += blockDim.x) s_h[i] = 0u;
        __syncthreads();
    }
    const long long warp0 = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
    const long long n_warps = ((long long)gridDim.x * blockDim.x) >> 5;
    const long long n_tiles = ceil_div(a.Po, kPrTile), n_items = (long long)a.B * n_tiles;
    unsigned bad = 0, pos = 0;                       // per lane: at most kUnrollR * Q entries per item
    for (long long w = warp0; w < n_items; w += n_warps) {
        const int b = (int)(w / n_tiles), p0 = (int)(w - (long long)b * n_tiles) * kPrTile;
        int fb;
        long long tb;
        if (!fleet_stream<kIdx>(ids, rows_of, n_fleet, b, a.t, fb, tb)) continue;     // warp-uniform
        unsigned rec[kUnrollR];
#pragma unroll
        for (int u = 0; u < kUnrollR; ++u) {
            const int p = p0 + 32 * u + lane;
            rec[u] = (a.rec && p < a.Po) ? a.rec[(size_t)fb * a.Po + p] : 0u;
        }
        for (int q = 0; q < a.Q; ++q) {
            if (!stream_row_valid(a.seen, fb, q, a.L)) continue;          // warp-uniform
            const StreamRows rows(a.S, a.ring, b, fb, a.Q, q, a.P, a.L, kIdx ? tb : a.t);
            float acc[kUnrollR];
#pragma unroll
            for (int u = 0; u < kUnrollR; ++u) acc[u] = 0.0f;
            if (p0 + kPrTile <= a.Po) {
                for (int j = 0; j < a.L; ++j) {
                    const float *row = rows.row(j) + (p0 + lane + j);
#pragma unroll
                    for (int u = 0; u < kUnrollR; ++u) acc[u] += __ldg(row + 32 * u);
                }
            } else {
                for (int j = 0; j < a.L; ++j) {
                    const float *row = rows.row(j) + (p0 + lane + j);
#pragma unroll
                    for (int u = 0; u < kUnrollR; ++u)
                        if (p0 + 32 * u + lane < a.Po) acc[u] += __ldg(row + 32 * u);
                }
            }
            const int c = __ldg(a.gt_center + (size_t)b * a.Q + q);
            unsigned long long kq = 0ull;
#pragma unroll
            for (int u = 0; u < kUnrollR; ++u) {
                const int p = p0 + 32 * u + lane;
                const bool in = p < a.Po;
                // k is exact only for an integer-valued sum in [0, 2^16); anything else makes the session invalid
                const bool ok = in && acc[u] >= 0.0f && acc[u] < (float)kStreamBins && acc[u] == truncf(acc[u]);
                bad += in && !ok;
                const int k = ok ? (int)acc[u] : 0;
                const bool g = ok && c >= 0 && abs(p - c) <= a.gt_tol;
                if (a.rec && ok) {
                    const unsigned any = (rec[u] & 1u) | (unsigned)g;
                    if ((unsigned)(k + 1) > rec[u] >> 2) rec[u] = (unsigned)(k + 1) << 2 | (unsigned)g << 1 | any;  // strict: first maximum
                    else rec[u] |= any;
                }
                if (a.key && ok) {
                    const unsigned long long kk = (unsigned long long)k << 32 | (uint32_t)~p;   // lowest place among ties
                    kq = kk > kq ? kk : kq;
                }
                if (a.hist) {
                    stream_hist_add(s_h, a.hist, ok, k, g, lane);
                    pos += g;
                }
            }
            if (a.key) {
                for (int o = 16; o > 0; o >>= 1) {
                    const unsigned long long other = shfl_xor_u64(kq, o);
                    kq = other > kq ? other : kq;
                }
                if (lane == 0 && kq) atomicMax(a.key + (size_t)b * a.Q + q, kq);
            }
        }
        if (a.rec) {
#pragma unroll
            for (int u = 0; u < kUnrollR; ++u) {
                const int p = p0 + 32 * u + lane;
                if (p < a.Po) a.rec[(size_t)fb * a.Po + p] = rec[u];
            }
        }
    }
    const unsigned long long bad_w = __reduce_add_sync(0xffffffffu, bad), pos_w = __reduce_add_sync(0xffffffffu, pos);
    if (lane == 0) {
        if (bad_w)
            for (int m = 0; m < 3; ++m)
                if (a.bad[m]) atomicAdd(a.bad[m], bad_w);
        if (pos_w) atomicAdd(a.multi_gtp, pos_w);
    }
    if (a.hist) stream_hist_flush(s_h, a.hist);
}

__global__ void __launch_bounds__(256, 4) seqpr_stream_accumulate_kernel(SeqPrStreamArgs a)
{
    stream_accumulate<false>(a, nullptr, nullptr, 0);
}

__global__ void __launch_bounds__(256, 4) seqpr_stream_accumulate_ids_kernel(SeqPrStreamArgs a,
                                                                             const int32_t *__restrict__ ids,
                                                                             const int64_t *__restrict__ rows,
                                                                             int n_fleet)
{
    stream_accumulate<true>(a, ids, rows, n_fleet);
}

// Query mode, after the accumulate kernel: one thread per new row folds its first maximum into the histogram and
// clears the scratch; gtp counts the valid rows with a positive among the places [0, Po).
template <bool kIdx>
__device__ __forceinline__ void stream_query_fold(const SeqPrStreamArgs &a, unsigned long long *acc_hist,
                                                  unsigned long long *gtp, const int32_t *__restrict__ ids,
                                                  const int64_t *__restrict__ rows, int n_fleet)
{
    const long long n = (long long)a.B * a.Q;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const int b = (int)(i / a.Q), q = (int)(i - (long long)b * a.Q);
        int fb;
        long long tb;
        if (!fleet_stream<kIdx>(ids, rows, n_fleet, b, a.t, fb, tb) || !stream_row_valid(a.seen, fb, q, a.L))
            continue;
        const unsigned long long key = a.key[i];
        a.key[i] = 0ull;
        const int c = __ldg(a.gt_center + i);
        if (c >= 0 && c - a.gt_tol < a.Po) atomicAdd(gtp, 1ull);
        if (!key) continue;                                              // every entry of the row was bad
        const int k = (int)(key >> 32), p = (int)~(uint32_t)key;
        const bool g = c >= 0 && abs(p - c) <= a.gt_tol;
        atomicAdd(acc_hist + (g ? 0 : kStreamBins) + k, 1ull);
    }
}

__global__ void __launch_bounds__(256) seqpr_stream_query_fold_kernel(SeqPrStreamArgs a, unsigned long long *acc_hist,
                                                                      unsigned long long *gtp)
{
    stream_query_fold<false>(a, acc_hist, gtp, nullptr, nullptr, 0);
}

__global__ void __launch_bounds__(256) seqpr_stream_query_fold_ids_kernel(SeqPrStreamArgs a,
                                                                          unsigned long long *acc_hist,
                                                                          unsigned long long *gtp,
                                                                          const int32_t *__restrict__ ids,
                                                                          const int64_t *__restrict__ rows,
                                                                          int n_fleet)
{
    stream_query_fold<true>(a, acc_hist, gtp, ids, rows, n_fleet);
}

// Place mode, finish: every record that saw a valid row is one column (k, hit at its first maximum); gtp counts the
// records with a positive, n_bad takes the accumulator's.
__global__ void __launch_bounds__(256) seqpr_stream_place_hist_kernel(const unsigned long long *__restrict__ acc,
                                                                      long long n,
                                                                      unsigned long long *__restrict__ hist,
                                                                      unsigned long long *__restrict__ gtp,
                                                                      unsigned long long *__restrict__ n_bad)
{
    __shared__ unsigned s_h[2 * kStreamShBins];
    const int lane = threadIdx.x & 31;
    const unsigned *rec = reinterpret_cast<const unsigned *>(acc + 2);
    if (blockIdx.x == 0 && threadIdx.x == 0 && acc[0]) atomicAdd(n_bad, acc[0]);
    for (int i = threadIdx.x; i < 2 * kStreamShBins; i += blockDim.x) s_h[i] = 0u;
    __syncthreads();
    unsigned long long pos = 0;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i0 = blockIdx.x * (long long)blockDim.x; i0 < n; i0 += stride) {   // the same trip count per warp
        const long long i = i0 + threadIdx.x;
        const unsigned r = i < n ? __ldg(rec + i) : 0u;
        stream_hist_add(s_h, hist, r != 0u, r ? (int)(r >> 2) - 1 : 0, (r >> 1) & 1u, lane);
        pos += r & 1u;
    }
    for (int o = 16; o > 0; o >>= 1) pos += __shfl_xor_sync(0xffffffffu, pos, o);
    if (lane == 0 && pos) atomicAdd(gtp, pos);
    stream_hist_flush(s_h, hist);
}

// Query / multi mode, finish: hist += the accumulator's histogram, {n_bad, gtp} += its header.
__global__ void __launch_bounds__(256) seqpr_stream_add_kernel(const unsigned long long *__restrict__ acc,
                                                               unsigned long long *__restrict__ hist,
                                                               unsigned long long *__restrict__ gtp,
                                                               unsigned long long *__restrict__ n_bad)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < 2 * kStreamBins) hist[i] += acc[2 + i];
    if (i == 0) { *n_bad += acc[0]; *gtp += acc[1]; }
}

// createPR's thresholds from the lowest and highest non-empty k (values fl(k / L)), then every non-empty k binned
// once into binned [2][n]; seqpr_prefix_kernel turns that into tp / fp.  One CTA.
__global__ void __launch_bounds__(1024) seqpr_stream_bin_kernel(const unsigned long long *__restrict__ hist, int L,
                                                                int n, unsigned long long *__restrict__ binned)
{
    __shared__ float s_y[kPrMaxThresh];
    __shared__ int s_lo, s_hi;
    if (threadIdx.x == 0) { s_lo = kStreamBins; s_hi = -1; }
    __syncthreads();
    int lo = kStreamBins, hi = -1;
    for (int k = threadIdx.x; k < kStreamBins; k += blockDim.x)
        if (hist[k] | hist[kStreamBins + k]) { lo = min(lo, k); hi = max(hi, k); }
    lo = __reduce_min_sync(0xffffffffu, lo);
    hi = __reduce_max_sync(0xffffffffu, hi);
    if ((threadIdx.x & 31) == 0) { atomicMin(&s_lo, lo); atomicMax(&s_hi, hi); }
    __syncthreads();
    if (s_hi < 0) return;                                                // empty session: nothing to count
    const float fl = (float)L;
    const float start = __fdiv_rn((float)s_hi, fl), stop = __fdiv_rn((float)s_lo, fl);
    for (int i = threadIdx.x; i < n; i += blockDim.x) s_y[i] = (float)pr_threshold(i, n, start, stop, false);
    __syncthreads();
    for (int k = s_lo + threadIdx.x; k <= s_hi; k += blockDim.x) {
        const unsigned long long tp = hist[k], fp = hist[kStreamBins + k];
        if (!(tp | fp)) continue;
        const int bin = seqpr_bin(s_y, n, __fdiv_rn((float)k, fl));
        if (tp) atomicAdd(binned + bin, tp);
        if (fp) atomicAdd(binned + n + bin, fp);
    }
}

// ---- tie-aware Recall@N bounds straight from S (lens_seq_recall_bounds*) -------------------------------------------
// The rule of recall_bounds_kernel without its level walk.  In one column (one sequence end of one stream) let vg be
// the largest D among its positives, A the places with D > vg (none of them positive) and E the non-positive places
// with D == vg.  Then for every K: a hit is possible iff A < K, and certain iff A + E < K.  So a column needs vg, then
// one pass over its places counting two predicates, with D recomputed exactly as K4 computes it (terms j = 0 .. L - 1,
// one __fdiv_rn); the bounds then bracket K4's own ranking for any finite S.  Once A >= max(ns) every K is a miss and
// the pass stops; a place segment that stops there still adds >= max(ns) to the row's A, so the sum stays exact.
// Three kernels per call, whatever the number of streams: peak (vg and validity per row), count (A, E, places split
// into segments when rows are few), finish (per-K lo / hi / n_valid).  kStream / kIdx as in the streaming match:
// batch (rows of S), lockstep streaming (StreamRows with t) and indexed streaming (fleet_stream<true>).
constexpr unsigned kRbSkip = 0u;        // row key: not a column (warm-up row, skipped id, no positive in dense GT)
constexpr unsigned kRbNoPositive = 1u;  // row key: a column whose band lies outside [0, Po): valid, never a hit
                                        // (any finite vg has an orderable key above both)

struct RecallBoundsArgs {
    const float *S, *ring;
    const int32_t *seen;
    long long t;
    const int32_t *ids;
    const int64_t *rows;
    int n_fleet;
    int B, Q, P, L, Qr, Po;             // Qr: rows per stream, Qo (batch) or Q (streaming)
    const uint8_t *gt_dense;            // [B or 1][Po][Qo] (batch only)
    int64_t gt_stride;
    const int32_t *gt_center;           // [B][Qr] by position
    int gt_tol;
    int ns[8];
    int n_ns;
    unsigned *key;                      // [B * Qr] orderable(vg), kRbSkip or kRbNoPositive
    unsigned long long *ae;             // [B * Qr] A << 32 | E, summed over the row's place segments
    unsigned long long *lo, *hi, *n_valid;
};

// The diagonal terms of batch row q of stream b: term j is row q + j of S.
struct BatchRows {
    const float *Sq;
    size_t P;
    __device__ __forceinline__ const float *row(int j) const { return Sq + (size_t)j * P; }
};

template <bool kStream>
__device__ __forceinline__ auto rbounds_rows(const RecallBoundsArgs &a, int b, int fb, int q, long long tb)
{
    if constexpr (kStream) return StreamRows(a.S, a.ring, b, fb, a.Q, q, a.P, a.L, tb);
    else return BatchRows{a.S + ((size_t)b * a.Q + q) * a.P, (size_t)a.P};
}

// Row g = b * Qr + q of the call -> (b, q, fleet stream fb, its row counter tb); false when g is not a sequence end.
template <bool kStream, bool kIdx>
__device__ __forceinline__ bool rbounds_row(const RecallBoundsArgs &a, int g, int &b, int &q, int &fb, long long &tb)
{
    b = g / a.Qr;
    q = g - b * a.Qr;
    if (!fleet_stream<kIdx>(a.ids, a.rows, a.n_fleet, b, a.t, fb, tb)) return false;
    return !kStream || stream_row_valid(a.seen, fb, q, a.L);
}

__device__ __forceinline__ bool rbounds_positive(const RecallBoundsArgs &a, int b, int p, int q, int c)
{
    if (a.gt_dense) return __ldg(a.gt_dense + (size_t)b * a.gt_stride + (size_t)p * a.Qr + q) != 0;
    return c >= 0 && abs(p - c) <= a.gt_tol;
}

// One warp per row: vg over the positives only (a band: at most 2 * tol + 1 places of L loads; dense GT: the lanes
// walk the GT column and compute D at its positives), merged as order-preserving keys.
template <bool kStream, bool kIdx>
__global__ void __launch_bounds__(256, 1) rbounds_peak_kernel(RecallBoundsArgs a)
{
    const int lane = threadIdx.x & 31;
    const int n = a.B * a.Qr;                                       // < 2^31 (checked on the host)
    const float fl = (float)a.L;
    const int warp0 = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
    for (int g = warp0; g < n; g += n_warps) {
        int b, q, fb;
        long long tb;
        unsigned key = kRbSkip;
        if (rbounds_row<kStream, kIdx>(a, g, b, q, fb, tb)) {          // warp-uniform
            const auto rr = rbounds_rows<kStream>(a, b, fb, q, tb);
            int p0 = 0, p1 = a.Po, c = 0;
            if (!a.gt_dense) {
                c = __ldg(a.gt_center + g);
                p0 = (int)max(0ll, (long long)c - a.gt_tol);
                p1 = c >= 0 ? (int)min((long long)a.Po, (long long)c + a.gt_tol + 1) : 0;
            }
            unsigned best = 0u;
            for (int p = p0 + lane; p < p1; p += 32) {
                if (a.gt_dense && !rbounds_positive(a, b, p, q, c)) continue;
                float acc = 0.0f;
                for (int j = 0; j < a.L; ++j) acc += __ldg(rr.row(j) + (p + j));
                best = max(best, f32_orderable(__fdiv_rn(acc, fl)));
            }
            best = __reduce_max_sync(0xffffffffu, best);
            key = best ? best : (!a.gt_dense && c >= 0 ? kRbNoPositive : kRbSkip);
        }
        if (lane == 0) a.key[g] = key;
    }
}

// One warp per (row, place segment), rows with a positive only: A and E over the segment's places with K4's coalesced
// diagonal loads, kUnrollR batches of 32 places in flight; stops once the warp's A reaches max(ns).
template <bool kStream, bool kIdx>
__global__ void __launch_bounds__(256) rbounds_count_kernel(RecallBoundsArgs a, int kmax, int n_seg, int seg_len)
{
    const int lane = threadIdx.x & 31;
    const float fl = (float)a.L;
    const long long n_rows = (long long)a.B * a.Qr;
    const long long warp0 = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
    const long long n_warps = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long w = warp0; w < n_rows * n_seg; w += n_warps) {
        const int seg = (int)(w / n_rows);
        const int g = (int)(w - (long long)seg * n_rows);
        const unsigned key = a.key[g];
        if (key <= kRbNoPositive) continue;                                     // warp-uniform
        const float vg = f32_from_orderable(key);
        int b, q, fb;
        long long tb;
        rbounds_row<kStream, kIdx>(a, g, b, q, fb, tb);                         // true: the peak kernel found a positive
        const auto rr = rbounds_rows<kStream>(a, b, fb, q, tb);
        const int c = a.gt_dense ? 0 : __ldg(a.gt_center + g);
        const int pe = min(a.Po, (seg + 1) * seg_len);
        unsigned n_above = 0, n_tied = 0;                                        // per lane: A, E
        for (int r0 = seg * seg_len; r0 < pe; r0 += 32 * kUnrollR) {
            float acc[kUnrollR];
#pragma unroll
            for (int u = 0; u < kUnrollR; ++u) acc[u] = 0.0f;
            if (r0 + 32 * kUnrollR <= pe) {
                for (int j = 0; j < a.L; ++j) {
                    const float *row = rr.row(j) + (r0 + lane + j);
#pragma unroll
                    for (int u = 0; u < kUnrollR; ++u) acc[u] += __ldg(row + 32 * u);
                }
            } else {
                for (int j = 0; j < a.L; ++j) {
                    const float *row = rr.row(j) + (r0 + lane + j);
#pragma unroll
                    for (int u = 0; u < kUnrollR; ++u)
                        if (r0 + 32 * u + lane < pe) acc[u] += __ldg(row + 32 * u);
                }
            }
#pragma unroll
            for (int u = 0; u < kUnrollR; ++u) {
                const int p = r0 + 32 * u + lane;
                if (p >= pe) continue;
                const float d = __fdiv_rn(acc[u], fl);
                n_above += d > vg;
                if (d == vg && !rbounds_positive(a, b, p, q, c)) ++n_tied;
            }
            if (__reduce_add_sync(0xffffffffu, n_above) >= (unsigned)kmax) break;     // every K is a miss
        }
        n_above = __reduce_add_sync(0xffffffffu, n_above);
        n_tied = __reduce_add_sync(0xffffffffu, n_tied);
        if (lane == 0 && (n_above | n_tied))
            atomicAdd(a.ae + g, (unsigned long long)n_above << 32 | n_tied);
    }
}

// One thread per row: n_valid, and lo / hi per K, added to the caller's counters once per block.
__global__ void __launch_bounds__(256) rbounds_finish_kernel(RecallBoundsArgs a)
{
    __shared__ unsigned s_lo[8], s_hi[8], s_valid;
    if (threadIdx.x < 8) s_lo[threadIdx.x] = s_hi[threadIdx.x] = 0u;
    if (threadIdx.x == 0) s_valid = 0u;
    __syncthreads();
    const int n = a.B * a.Qr;
    unsigned lo[8], hi[8], valid = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) lo[i] = hi[i] = 0u;
    for (int g = blockIdx.x * blockDim.x + threadIdx.x; g < n; g += gridDim.x * blockDim.x) {
        const unsigned key = a.key[g];
        if (key == kRbSkip) continue;
        ++valid;
        if (key == kRbNoPositive) continue;
        const unsigned long long ae = a.ae[g];
        const unsigned long long above = ae >> 32, tied = ae & 0xffffffffull;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            if (i >= a.n_ns) break;
            hi[i] += above < (unsigned long long)a.ns[i];
            lo[i] += above + tied < (unsigned long long)a.ns[i];
        }
    }
    valid = __reduce_add_sync(0xffffffffu, valid);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        lo[i] = __reduce_add_sync(0xffffffffu, lo[i]);
        hi[i] = __reduce_add_sync(0xffffffffu, hi[i]);
    }
    if ((threadIdx.x & 31) == 0) {
        if (valid) atomicAdd(&s_valid, valid);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            if (lo[i]) atomicAdd(&s_lo[i], lo[i]);
            if (hi[i]) atomicAdd(&s_hi[i], hi[i]);
        }
    }
    __syncthreads();
    if (threadIdx.x < a.n_ns) {
        if (s_lo[threadIdx.x]) atomicAdd(a.lo + threadIdx.x, (unsigned long long)s_lo[threadIdx.x]);
        if (s_hi[threadIdx.x]) atomicAdd(a.hi + threadIdx.x, (unsigned long long)s_hi[threadIdx.x]);
    }
    if (threadIdx.x == 0 && s_valid) atomicAdd(a.n_valid, (unsigned long long)s_valid);
}

// SAD baseline (lens/src/sad.py:38): one warp per (query, reference) pair, 16 pixels per lane-iteration
// with byte-wise SIMD sum of absolute differences; integer accumulation (exact), stored as fp32.
__global__ void __launch_bounds__(256) sad_kernel(const uint8_t *__restrict__ a, const uint8_t *__restrict__ b,
                                                  int Q, int R, int npix, float *__restrict__ dist)
{
    const int lane = threadIdx.x & 31;
    const long long pair = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
    if (pair >= (long long)Q * R) return;
    const int q = (int)(pair / R), r = (int)(pair - (long long)q * R);
    const uint8_t *pa = a + (size_t)q * npix, *pb = b + (size_t)r * npix;
    unsigned int acc = 0;
    if ((npix & 15) == 0 && ((((uintptr_t)a | (uintptr_t)b)) & 15) == 0) {
        const uint4 *va = reinterpret_cast<const uint4 *>(pa), *vb = reinterpret_cast<const uint4 *>(pb);
        for (int i = lane; i < npix / 16; i += 32) {
            const uint4 x = __ldg(va + i), y = __ldg(vb + i);
            acc += __vsadu4(x.x, y.x) + __vsadu4(x.y, y.y) + __vsadu4(x.z, y.z) + __vsadu4(x.w, y.w);
        }
    } else {
        for (int i = lane; i < npix; i += 32) acc += (unsigned)abs((int)pa[i] - (int)pb[i]);
    }
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) dist[pair] = (float)acc;
}

__global__ void reciprocal_kernel(const float *__restrict__ in, int64_t n, float *__restrict__ out)
{
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) out[i] = __fdiv_rn(1.0f, in[i]);
}

// Online matcher (run_speck.py:155-226): a readout adds its spike counts to the running sums; every
// `div` readouts the sums, floor-divided, become one sequence row.
__global__ void online_accumulate_kernel(int32_t *__restrict__ sum, const float *__restrict__ counts, int P, int div,
                                         int32_t *__restrict__ row_out)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P) return;
    const int32_t s = sum[i] + (int32_t)counts[i];
    sum[i] = s;
    if (row_out) {
        int32_t q = s / div;
        if ((s % div != 0) && ((s < 0) != (div < 0))) --q;      // floor division like numpy's //
        row_out[i] = q;
    }
}

// result[p][r] = (1/L) sum_a seq[r+o-a][p+o-a] ('same' crop of the full convolution with eye(L)), then the
// first maximum of every column r.  One CTA per column: coalesced reads along p for each of the L taps.
__global__ void __launch_bounds__(256) online_match_kernel(const int32_t *__restrict__ seq, int R, int P, int L,
                                                           double *__restrict__ result, int32_t *__restrict__ argmax)
{
    const int r = blockIdx.x, o = (L - 1) / 2;
    double best = 0.0;
    int best_p = 0x7fffffff;
    bool have = false;
    for (int p = threadIdx.x; p < P; p += blockDim.x) {
        long long acc = 0;
        for (int a = 0; a < L; ++a) {
            const int rr = r + o - a, pp = p + o - a;
            if (rr >= 0 && rr < R && pp >= 0 && pp < P) acc += seq[(size_t)rr * P + pp];
        }
        const double v = __ddiv_rn((double)acc, (double)L);
        result[(size_t)p * R + r] = v;
        if (!have || v > best) { best = v; best_p = p; have = true; }   // p ascending per thread: first max kept
    }
    __shared__ double sv[256];
    __shared__ int sp[256];
    sv[threadIdx.x] = best; sp[threadIdx.x] = best_p;
    __syncthreads();
    for (int s = blockDim.x / 2; s > 0; s >>= 1) {
        if (threadIdx.x < s) {
            const double v2 = sv[threadIdx.x + s];
            const int p2 = sp[threadIdx.x + s];
            const int p1 = sp[threadIdx.x];
            if (p2 != 0x7fffffff && (p1 == 0x7fffffff || v2 > sv[threadIdx.x] || (v2 == sv[threadIdx.x] && p2 < p1))) {
                sv[threadIdx.x] = v2; sp[threadIdx.x] = p2;
            }
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) argmax[r] = sp[0];
}

}  // namespace lens

using namespace lens;

extern "C" int lens_online_accumulate(int32_t *sum, const float *counts, int P, int div, int32_t *row_out, void *stream)
{
    LENS_CHECK_ARG(sum && counts, "lens_online_accumulate: NULL buffer");
    LENS_CHECK_ARG(P > 0 && div != 0, "lens_online_accumulate: need P > 0 and div != 0");
    online_accumulate_kernel<<<(unsigned)((P + 255) / 256), 256, 0, as_stream(stream)>>>(sum, counts, P, div, row_out);
    LENS_LAUNCH_CHECK();
    return 0;
}

extern "C" int lens_online_match(const int32_t *seq, int R, int P, int L, double *result, int32_t *argmax, void *stream)
{
    LENS_CHECK_ARG(seq && result && argmax, "lens_online_match: NULL buffer");
    LENS_CHECK_ARG(P > 0 && R >= 1 && R <= 64 && L >= 1 && L <= 64, "lens_online_match: need P > 0, 1 <= R, L <= 64");
    online_match_kernel<<<(unsigned)R, 256, 0, as_stream(stream)>>>(seq, R, P, L, result, argmax);
    LENS_LAUNCH_CHECK();
    return 0;
}

extern "C" int lens_sad_matrix(const uint8_t *a, const uint8_t *b, int Q, int R, int npix, float *dist, void *stream)
{
    LENS_CHECK_ARG(a && b && dist, "lens_sad_matrix: NULL buffer");
    LENS_CHECK_ARG(Q > 0 && R > 0 && npix > 0 && npix <= 65793, "lens_sad_matrix: need Q, R > 0 and 0 < npix <= 65793 "
                   "(sums must stay below 2^24)");
    const long long pairs = (long long)Q * R;
    sad_kernel<<<(unsigned)((pairs * 32 + 255) / 256), 256, 0, as_stream(stream)>>>(a, b, Q, R, npix, dist);
    LENS_LAUNCH_CHECK();
    return 0;
}

extern "C" int lens_reciprocal(const float *in, int64_t n, float *out, void *stream)
{
    LENS_CHECK_ARG(in && out && n >= 0, "lens_reciprocal: bad arguments");
    if (n == 0) return 0;
    reciprocal_kernel<<<(unsigned)((n + 255) / 256), 256, 0, as_stream(stream)>>>(in, n, out);
    LENS_LAUNCH_CHECK();
    return 0;
}

extern "C" int lens_pr_counts(const float *S, const uint8_t *GT, int Po, int Qo, int n_thresh, int64_t *tp,
                              int64_t *fp, int64_t *gtp, void *stream, int thresh_f64)
{
    LENS_CHECK_ARG(S && GT && tp && fp && gtp, "lens_pr_counts: NULL buffer");
    LENS_CHECK_ARG(Po > 0 && Qo > 0 && Qo <= 8192, "lens_pr_counts: need 0 < Qo <= 8192, Po > 0");
    LENS_CHECK_ARG(n_thresh > 1, "lens_pr_counts: n_thresh must be > 1");
    pr_counts_kernel<<<1, 256, (size_t)Qo * 5, as_stream(stream)>>>(
        S, GT, Po, Qo, n_thresh, thresh_f64, reinterpret_cast<unsigned long long *>(tp),
        reinterpret_cast<unsigned long long *>(fp), reinterpret_cast<unsigned long long *>(gtp));
    LENS_LAUNCH_CHECK();
    return 0;
}

// Grid of the warp-per-query kernels.  Few queries against many places (config 5: 1 024 streams x 100 000 places)
// would leave most SMs without a warp: the places of a query are then split into n_seg segments ranked by different
// warps, and the per-segment lists are merged by the kernel that merges per-GPU lists (same order: value desc, place
// index desc).
static void plan_segments(long long n_queries, int Po, int N, int &n_seg, int &seg_len, long long &blocks)
{
    const long long sms = std::max(sm_count(), 1), want_warps = sms * 32;
    n_seg = 1;
    if (n_queries < want_warps && Po >= 8192)
        n_seg = (int)std::min<long long>(std::min<long long>(ceil_div64(want_warps, n_queries), (32 * kMergeSlots) / N),
                                         Po / 4096);
    n_seg = std::max(n_seg, 1);
    seg_len = ceil_div(ceil_div(Po, n_seg), 32 * kUnrollR) * (32 * kUnrollR);
    n_seg = ceil_div(Po, seg_len);
    blocks = std::min<long long>((n_queries * n_seg + 7) / 8, sms * 16);
}

extern "C" int lens_seqmatch_topk(const float *S, int B, int Q, int P, int L, int N, float *D_out,
                                  float *top_val, int32_t *top_idx, void *stream)
{
    LENS_CHECK_ARG(B >= 0 && Q > 0 && P > 0, "lens_seqmatch_topk: bad sizes");
    LENS_CHECK_ARG(L >= 1 && L <= Q && L <= P, "lens_seqmatch_topk: need 1 <= L <= min(Q, P), got L=%d", L);
    LENS_CHECK_ARG(N >= 1 && N <= kMaxTopN, "lens_seqmatch_topk: N=%d outside [1, %d]", N, kMaxTopN);
    LENS_CHECK_ARG(B == 0 || (S && top_val && top_idx), "lens_seqmatch_topk: NULL buffer");
    LENS_CHECK_ARG((int64_t)B * (Q - L + 1) <= 2147483647LL, "lens_seqmatch_topk: too many (stream, query) pairs");
    if (B == 0) return 0;
    const long long n_queries = (long long)B * (Q - L + 1);
    if (N <= 32) {
        int n_seg, seg_len;
        long long blocks;
        plan_segments(n_queries, P - L + 1, N, n_seg, seg_len, blocks);
        const long long n_work = n_queries * n_seg;
        cudaStream_t st = as_stream(stream);
        if (n_seg == 1) {
            seqmatch_topk_warp_kernel<false><<<(unsigned)blocks, 256, 0, st>>>(S, n_queries, Q, P, L, N, 1, seg_len, D_out,
                                                                              top_val, top_idx);
        } else {
            // stream-ordered scratch for the per-segment lists (no synchronisation)
            float *seg_val = nullptr;
            int32_t *seg_idx = nullptr;
            const size_t n_list = (size_t)n_work * N;
            LENS_CUDA(cudaMallocAsync(&seg_val, n_list * (sizeof(float) + sizeof(int32_t)), st));   // one block: values | indices
            seg_idx = reinterpret_cast<int32_t *>(seg_val + n_list);
            seqmatch_topk_warp_kernel<true><<<(unsigned)blocks, 256, 0, st>>>(S, n_queries, Q, P, L, N, n_seg, seg_len, D_out,
                                                                             seg_val, seg_idx);
            LENS_LAUNCH_CHECK();
            topn_merge_kernel<<<(unsigned)ceil_div64(n_queries, 8), 256, 0, st>>>(seg_val, seg_idx, n_seg, n_queries, N,
                                                                                   top_val, top_idx);
            LENS_CUDA(cudaFreeAsync(seg_val, st));
        }
    } else {
        dim3 grid((unsigned)n_queries);
        seqmatch_topk_kernel<<<grid, kMatchThreads, 0, as_stream(stream)>>>(S, Q, P, L, N, D_out, top_val, top_idx);
    }
    LENS_LAUNCH_CHECK();
    return 0;
}

// Host side of both streaming matches.  kIdx = false: lens_seqmatch_topk_stream (B streams in lockstep, t rows each);
// kIdx = true: lens_seqmatch_topk_stream_ids (B = the n pushing streams ids[0..n) of a fleet of n_fleet, rows[]).
template <bool kIdx>
static int stream_match(const char *fn, const float *S, int B, int Q, int P, int L, int N, const int32_t *ids,
                        int n_fleet, float *ring, int32_t *seen, int64_t t, int64_t *rows, float *top_val,
                        int32_t *top_idx, void *stream)
{
    LENS_CHECK_ARG(B >= 0 && Q > 0 && P > 0, "%s: bad sizes", fn);
    LENS_CHECK_ARG(L >= 1 && L <= P, "%s: need 1 <= L <= P, got L=%d", fn, L);
    LENS_CHECK_ARG(N >= 1 && N <= kMaxTopN, "%s: N=%d outside [1, %d]", fn, N, kMaxTopN);
    LENS_CHECK_ARG(t >= 0, "%s: t must be >= 0", fn);
    LENS_CHECK_ARG(seen != nullptr, "%s: NULL seen", fn);
    LENS_CHECK_ARG(L == 1 || ring != nullptr, "%s: NULL ring needs L == 1, got L=%d", fn, L);
    LENS_CHECK_ARG(B == 0 || (S && top_val && top_idx), "%s: NULL buffer", fn);
    LENS_CHECK_ARG((int64_t)B * Q <= 2147483647LL, "%s: too many (stream, row) pairs", fn);
    if constexpr (kIdx) {
        LENS_CHECK_ARG(n_fleet >= 0, "%s: bad fleet size %d", fn, n_fleet);
        LENS_CHECK_ARG(B == 0 || (ids && rows), "%s: NULL ids / rows", fn);
    }
    if (B == 0) return 0;
    cudaStream_t st = as_stream(stream);
    const long long n_queries = (long long)B * Q;
    if (N <= 32) {
        int n_seg, seg_len;
        long long blocks;
        plan_segments(n_queries, P - L + 1, N, n_seg, seg_len, blocks);
        if (n_seg == 1) {
            if constexpr (kIdx)
                seqmatch_topk_stream_ids_warp_kernel<false><<<(unsigned)blocks, 256, 0, st>>>(
                    S, ring, seen, ids, rows, n_fleet, n_queries, Q, P, L, N, 1, seg_len, top_val, top_idx);
            else
                seqmatch_topk_stream_warp_kernel<false><<<(unsigned)blocks, 256, 0, st>>>(
                    S, ring, seen, t, n_queries, Q, P, L, N, 1, seg_len, top_val, top_idx);
            LENS_LAUNCH_CHECK();
        } else {
            float *seg_val = nullptr;                      // stream-ordered scratch, as in lens_seqmatch_topk
            const size_t n_list = (size_t)n_queries * n_seg * N;
            LENS_CUDA(cudaMallocAsync(&seg_val, n_list * (sizeof(float) + sizeof(int32_t)), st));
            int32_t *seg_idx = reinterpret_cast<int32_t *>(seg_val + n_list);
            if constexpr (kIdx)
                seqmatch_topk_stream_ids_warp_kernel<true><<<(unsigned)blocks, 256, 0, st>>>(
                    S, ring, seen, ids, rows, n_fleet, n_queries, Q, P, L, N, n_seg, seg_len, seg_val, seg_idx);
            else
                seqmatch_topk_stream_warp_kernel<true><<<(unsigned)blocks, 256, 0, st>>>(
                    S, ring, seen, t, n_queries, Q, P, L, N, n_seg, seg_len, seg_val, seg_idx);
            LENS_LAUNCH_CHECK();
            topn_merge_kernel<<<(unsigned)ceil_div64(n_queries, 8), 256, 0, st>>>(seg_val, seg_idx, n_seg, n_queries, N,
                                                                                   top_val, top_idx);
            LENS_LAUNCH_CHECK();
            LENS_CUDA(cudaFreeAsync(seg_val, st));
        }
    } else {
        if constexpr (kIdx)
            seqmatch_topk_stream_kernel<true><<<(unsigned)n_queries, kMatchThreads, 0, st>>>(
                S, ring, seen, 0, Q, P, L, N, top_val, top_idx, ids, rows, n_fleet);
        else
            seqmatch_topk_stream_kernel<false><<<(unsigned)n_queries, kMatchThreads, 0, st>>>(
                S, ring, seen, t, Q, P, L, N, top_val, top_idx, nullptr, nullptr, 0);
        LENS_LAUNCH_CHECK();
    }
    const long long sms = std::max(sm_count(), 1);
    if (L > 1) {
        const long long n_rows = (long long)B * std::min(Q, L - 1);
        const long long blocks = std::min<long long>(n_rows, sms * 16);
        if constexpr (kIdx)
            ring_append_ids_kernel<<<(unsigned)blocks, 256, 0, st>>>(S, B, Q, P, L, ring, ids, rows, n_fleet);
        else
            ring_append_kernel<<<(unsigned)blocks, 256, 0, st>>>(S, B, Q, P, L, t, ring, seen);
        LENS_LAUNCH_CHECK();
    }
    if constexpr (kIdx) {
        stream_advance_kernel<<<(unsigned)std::min<long long>(ceil_div(B, 256), sms * 8), 256, 0, st>>>(
            ids, B, n_fleet, Q, L, seen, rows);
        LENS_LAUNCH_CHECK();
    }
    return 0;
}

extern "C" int lens_seqmatch_topk_stream(const float *S, int B, int Q, int P, int L, int N, float *ring, int32_t *seen,
                                         int64_t t, float *top_val, int32_t *top_idx, void *stream)
{
    return stream_match<false>("lens_seqmatch_topk_stream", S, B, Q, P, L, N, nullptr, B, ring, seen, t, nullptr,
                               top_val, top_idx, stream);
}

extern "C" int lens_seqmatch_topk_stream_ids(const float *S, int n, int Q, int P, int L, int N, const int32_t *ids,
                                             int B, float *ring, int32_t *seen, int64_t *rows, float *top_val,
                                             int32_t *top_idx, void *stream)
{
    return stream_match<true>("lens_seqmatch_topk_stream_ids", S, n, Q, P, L, N, ids, B, ring, seen, 0, rows, top_val,
                              top_idx, stream);
}

extern "C" int lens_recall(const int32_t *top_idx, int B, int Qo, int Po, int N,
                           const uint8_t *gt_dense, int64_t gt_stream_stride,
                           const int32_t *gt_center, int gt_tol, const int *ns, int n_ns,
                           int64_t *hits, int64_t *n_valid, void *stream)
{
    LENS_CHECK_ARG(B >= 0 && Qo > 0 && Po > 0 && N >= 1, "lens_recall: bad sizes");
    LENS_CHECK_ARG((gt_dense != nullptr) != (gt_center != nullptr),
                   "lens_recall: exactly one of gt_dense / gt_center must be given");
    LENS_CHECK_ARG(ns && n_ns >= 1 && n_ns <= 8, "lens_recall: n_ns must be in [1, 8]");
    LENS_CHECK_ARG(top_idx && hits && n_valid, "lens_recall: NULL buffer");
    RecallParams p;
    p.top_idx = top_idx; p.B = B; p.Qo = Qo; p.Po = Po; p.N = N;
    p.gt_dense = gt_dense; p.gt_stream_stride = gt_stream_stride;
    p.gt_center = gt_center; p.gt_tol = gt_tol; p.n_ns = n_ns;
    for (int i = 0; i < 8; ++i) p.ns[i] = 0;
    for (int i = 0; i < n_ns; ++i) {
        LENS_CHECK_ARG(ns[i] >= 1 && ns[i] <= N, "lens_recall: ns[%d]=%d outside [1, N=%d]", i, ns[i], N);
        p.ns[i] = ns[i];
    }
    p.hits = reinterpret_cast<unsigned long long *>(hits);
    p.n_valid = reinterpret_cast<unsigned long long *>(n_valid);
    if (B == 0) return 0;
    int64_t total = (int64_t)B * Qo;
    recall_kernel<<<(unsigned)ceil_div64(total, 256), 256, 0, as_stream(stream)>>>(p);
    LENS_LAUNCH_CHECK();
    return 0;
}

extern "C" int lens_recall_bounds(const float *D, const uint8_t *GT, int Po, int Qo, const int *ns, int n_ns,
                                  int64_t *lo, int64_t *hi, int64_t *n_valid, void *stream)
{
    LENS_CHECK_ARG(Po > 0 && Qo > 0, "lens_recall_bounds: bad sizes");
    LENS_CHECK_ARG(D && GT && lo && hi && n_valid, "lens_recall_bounds: NULL buffer");
    LENS_CHECK_ARG(ns && n_ns >= 1 && n_ns <= 8, "lens_recall_bounds: n_ns must be in [1, 8]");
    BoundsParams p;
    p.D = D; p.GT = GT; p.Po = Po; p.Qo = Qo; p.n_ns = n_ns;
    for (int i = 0; i < 8; ++i) p.ns[i] = 0;
    for (int i = 0; i < n_ns; ++i) {
        LENS_CHECK_ARG(ns[i] >= 1 && (i == 0 || ns[i] > ns[i - 1]), "lens_recall_bounds: ns must be ascending and >= 1");
        p.ns[i] = ns[i];
    }
    p.lo = reinterpret_cast<unsigned long long *>(lo);
    p.hi = reinterpret_cast<unsigned long long *>(hi);
    p.n_valid = reinterpret_cast<unsigned long long *>(n_valid);
    recall_bounds_kernel<<<(unsigned)ceil_div(Qo, 8), 256, 0, as_stream(stream)>>>(p);
    LENS_LAUNCH_CHECK();
    return 0;
}

extern "C" int lens_topn_merge(const float *val, const int32_t *idx, int W, int64_t M, int N, float *out_val,
                               int32_t *out_idx, void *stream)
{
    LENS_CHECK_ARG(W >= 1 && M >= 0 && N >= 1, "lens_topn_merge: bad sizes");
    LENS_CHECK_ARG((int64_t)W * N <= 32 * kMergeSlots, "lens_topn_merge: W * N = %lld exceeds %d", (long long)W * N,
                   32 * kMergeSlots);
    if (M == 0) return 0;
    LENS_CHECK_ARG(val && idx && out_val && out_idx, "lens_topn_merge: NULL buffer");
    topn_merge_kernel<<<(unsigned)ceil_div64(M, 8), 256, 0, as_stream(stream)>>>(val, idx, W, M, N, out_val, out_idx);
    LENS_LAUNCH_CHECK();
    return 0;
}

extern "C" int lens_pr_counts_multi(const float *S, const uint8_t *GT, int Po, int Qo, int n_thresh, int64_t *tp,
                                    int64_t *fp, int64_t *gtp, void *stream, int thresh_f64)
{
    LENS_CHECK_ARG(Po > 0 && Qo > 0, "lens_pr_counts_multi: bad sizes");
    LENS_CHECK_ARG(n_thresh > 1 && n_thresh <= 65535, "lens_pr_counts_multi: n_thresh must be in (1, 65535]");
    LENS_CHECK_ARG(S && GT && tp && fp && gtp, "lens_pr_counts_multi: NULL buffer");
    cudaStream_t st = as_stream(stream);
    const long long n = (long long)Po * Qo;
    unsigned int *mm = nullptr;                       // {max, min} of S as order-preserving integers
    LENS_CUDA(cudaMallocAsync(&mm, 2 * sizeof(unsigned int), st));
    LENS_CUDA(cudaMemsetAsync(mm, 0x00, sizeof(unsigned int), st));
    LENS_CUDA(cudaMemsetAsync(mm + 1, 0xff, sizeof(unsigned int), st));
    LENS_CUDA(cudaMemsetAsync(tp, 0, (size_t)n_thresh * sizeof(int64_t), st));
    LENS_CUDA(cudaMemsetAsync(fp, 0, (size_t)n_thresh * sizeof(int64_t), st));
    LENS_CUDA(cudaMemsetAsync(gtp, 0, sizeof(int64_t), st));
    const int blocks = (int)std::min<long long>(ceil_div64(n, 256), (long long)std::max(sm_count(), 1) * 8);
    pr_multi_minmax_kernel<<<blocks, 256, 0, st>>>(S, GT, n, mm, reinterpret_cast<unsigned long long *>(gtp));
    LENS_LAUNCH_CHECK();
    const int slices = (int)std::max<long long>(1, std::min<long long>(ceil_div64(n, 65536), 64));
    pr_multi_counts_kernel<<<dim3((unsigned)n_thresh, (unsigned)slices), 256, 0, st>>>(
        S, GT, n, n_thresh, thresh_f64, mm, reinterpret_cast<unsigned long long *>(tp),
        reinterpret_cast<unsigned long long *>(fp));
    LENS_LAUNCH_CHECK();
    LENS_CUDA(cudaFreeAsync(mm, st));
    return 0;
}

// Validates the arguments shared by lens_seqpr_scan / lens_seqpr_counts and fills the kernel arguments.
static int seqpr_args(SeqPrArgs &a, const char *fn, const float *S, int B, int Q, int P, int L, int mode,
                      const uint8_t *gt_dense, int64_t gt_stream_stride, const int32_t *gt_center, int gt_tol,
                      void *records)
{
    LENS_CHECK_ARG(B >= 0 && Q > 0 && P > 0, "%s: bad sizes", fn);
    LENS_CHECK_ARG(L >= 1 && L <= Q && L <= P, "%s: need 1 <= L <= min(Q, P), got L=%d", fn, L);
    LENS_CHECK_ARG(mode == LENS_SEQPR_PLACE || mode == LENS_SEQPR_QUERY || mode == LENS_SEQPR_MULTI,
                   "%s: unknown mode %d", fn, mode);
    LENS_CHECK_ARG((gt_dense != nullptr) != (gt_center != nullptr),
                   "%s: exactly one of gt_dense / gt_center must be given", fn);
    LENS_CHECK_ARG(gt_stream_stride >= 0 && gt_tol >= 0, "%s: gt_stream_stride and gt_tol must be >= 0", fn);
    LENS_CHECK_ARG(B == 0 || S != nullptr, "%s: NULL S", fn);
    LENS_CHECK_ARG(mode == LENS_SEQPR_MULTI || B == 0 || (records && (reinterpret_cast<uintptr_t>(records) & 7) == 0),
                   "%s: the single modes need 8-byte aligned records", fn);
    a = SeqPrArgs{};
    a.S = S; a.B = B; a.Q = Q; a.P = P; a.L = L; a.Qo = Q - L + 1; a.Po = P - L + 1;
    a.gt_dense = gt_dense; a.gt_stride = gt_stream_stride; a.gt_center = gt_center; a.gt_tol = gt_tol;
    const size_t n_rec = (size_t)B * (mode == LENS_SEQPR_PLACE ? a.Po : a.Qo);
    if (mode == LENS_SEQPR_PLACE) {
        a.rec_val = static_cast<float *>(records);
        a.rec_flag = reinterpret_cast<uint8_t *>(a.rec_val + n_rec);
    } else if (mode == LENS_SEQPR_QUERY) {
        a.rec_key = static_cast<unsigned long long *>(records);
        a.rec_flag = reinterpret_cast<uint8_t *>(a.rec_key + n_rec);
    }
    return 0;
}

extern "C" int lens_seqpr_records_bytes(int B, int Q, int P, int L, int mode, int64_t *bytes)
{
    LENS_CHECK_ARG(bytes != nullptr, "lens_seqpr_records_bytes: NULL bytes");
    LENS_CHECK_ARG(B >= 0 && L >= 1 && L <= Q && L <= P, "lens_seqpr_records_bytes: bad sizes");
    LENS_CHECK_ARG(mode == LENS_SEQPR_PLACE || mode == LENS_SEQPR_QUERY || mode == LENS_SEQPR_MULTI,
                   "lens_seqpr_records_bytes: unknown mode %d", mode);
    if (mode == LENS_SEQPR_PLACE) *bytes = (int64_t)B * (P - L + 1) * (sizeof(float) + 1);
    else if (mode == LENS_SEQPR_QUERY) *bytes = (int64_t)B * (Q - L + 1) * (sizeof(unsigned long long) + 1);
    else *bytes = 0;
    return 0;
}

extern "C" int lens_seqpr_scan(const float *S, int B, int Q, int P, int L, int mode, const uint8_t *gt_dense,
                               int64_t gt_stream_stride, const int32_t *gt_center, int gt_tol, void *records,
                               uint64_t *extremes, int64_t *gtp, void *stream)
{
    SeqPrArgs a;
    if (int rc = seqpr_args(a, "lens_seqpr_scan", S, B, Q, P, L, mode, gt_dense, gt_stream_stride, gt_center, gt_tol,
                            records))
        return rc;
    LENS_CHECK_ARG(extremes && gtp, "lens_seqpr_scan: NULL extremes / gtp");
    if (B == 0) return 0;
    a.ext = reinterpret_cast<unsigned long long *>(extremes);
    a.gtp = reinterpret_cast<unsigned long long *>(gtp);
    cudaStream_t st = as_stream(stream);
    const long long sms = std::max(sm_count(), 1);
    const long long items = (long long)B * ceil_div(a.Po, kPrTile);
    const unsigned blocks = (unsigned)std::min<long long>(ceil_div64(items, 8), sms * 16);
    if (mode == LENS_SEQPR_PLACE) {
        seqpr_scan_kernel<kPrPlace><<<blocks, 256, 0, st>>>(a);
        LENS_LAUNCH_CHECK();
    } else if (mode == LENS_SEQPR_QUERY) {
        const size_t n_rec = (size_t)B * a.Qo;
        LENS_CUDA(cudaMemsetAsync(records, 0, n_rec * (sizeof(unsigned long long) + 1), st));
        seqpr_scan_kernel<kPrQuery><<<blocks, 256, 0, st>>>(a);
        LENS_LAUNCH_CHECK();
        seqpr_query_extremes_kernel<<<(unsigned)std::min<long long>(ceil_div64((long long)n_rec, 256), sms * 8), 256, 0,
                                      st>>>(a);
        LENS_LAUNCH_CHECK();
    } else {
        seqpr_scan_kernel<kPrMulti><<<blocks, 256, 0, st>>>(a);
        LENS_LAUNCH_CHECK();
    }
    return 0;
}

extern "C" int lens_seqpr_counts(const float *S, int B, int Q, int P, int L, int mode, const uint8_t *gt_dense,
                                 int64_t gt_stream_stride, const int32_t *gt_center, int gt_tol, const void *records,
                                 const uint64_t *extremes, int n_thresh, int64_t *tp, int64_t *fp, void *stream)
{
    SeqPrArgs a;
    if (int rc = seqpr_args(a, "lens_seqpr_counts", S, B, Q, P, L, mode, gt_dense, gt_stream_stride, gt_center,
                            gt_tol, const_cast<void *>(records)))
        return rc;
    LENS_CHECK_ARG(n_thresh >= 2 && n_thresh <= kPrMaxThresh, "lens_seqpr_counts: n_thresh must be in [2, %d], got %d",
                   kPrMaxThresh, n_thresh);
    LENS_CHECK_ARG(extremes && tp && fp, "lens_seqpr_counts: NULL extremes / tp / fp");
    if (B == 0) return 0;
    a.ext = const_cast<unsigned long long *>(reinterpret_cast<const unsigned long long *>(extremes));
    a.n_thresh = n_thresh;
    cudaStream_t st = as_stream(stream);
    const long long sms = std::max(sm_count(), 1);
    const size_t hist_bytes = (size_t)2 * n_thresh * sizeof(unsigned long long);
    LENS_CUDA(cudaMallocAsync(&a.hist, hist_bytes, st));          // stream-ordered scratch, as in lens_seqmatch_topk
    LENS_CUDA(cudaMemsetAsync(a.hist, 0, hist_bytes, st));
    const size_t smem = (size_t)n_thresh * (sizeof(float) + 2 * sizeof(unsigned));   // <= 48 KB
    if (mode == LENS_SEQPR_MULTI) {
        const long long items = (long long)B * ceil_div(a.Po, kPrTile);
        seqpr_count_kernel<kPrMulti><<<(unsigned)std::min<long long>(ceil_div64(items, 8), sms * 8), 256, smem, st>>>(a);
    } else {
        const long long n_rec = (long long)B * (mode == LENS_SEQPR_PLACE ? a.Po : a.Qo);
        const unsigned blocks = (unsigned)std::min<long long>(ceil_div64(n_rec, 256 * 4), sms * 8);
        if (mode == LENS_SEQPR_PLACE) seqpr_count_kernel<kPrPlace><<<blocks, 256, smem, st>>>(a);
        else seqpr_count_kernel<kPrQuery><<<blocks, 256, smem, st>>>(a);
    }
    LENS_LAUNCH_CHECK();
    seqpr_prefix_kernel<<<1, 64, 0, st>>>(a.hist, n_thresh, reinterpret_cast<unsigned long long *>(tp),
                                          reinterpret_cast<unsigned long long *>(fp));
    LENS_LAUNCH_CHECK();
    LENS_CUDA(cudaFreeAsync(a.hist, st));
    return 0;
}

extern "C" int lens_seqpr_stream_bytes(int B, int P, int L, int mode, int64_t *bytes)
{
    LENS_CHECK_ARG(bytes != nullptr, "lens_seqpr_stream_bytes: NULL bytes");
    LENS_CHECK_ARG(B >= 0 && P > 0 && L >= 1 && L <= P, "lens_seqpr_stream_bytes: bad sizes");
    LENS_CHECK_ARG(mode == LENS_SEQPR_PLACE || mode == LENS_SEQPR_QUERY || mode == LENS_SEQPR_MULTI,
                   "lens_seqpr_stream_bytes: unknown mode %d", mode);
    const int64_t header = 2 * sizeof(unsigned long long);
    if (mode == LENS_SEQPR_PLACE) *bytes = header + (int64_t)B * (P - L + 1) * sizeof(unsigned);
    else *bytes = header + (int64_t)2 * kStreamBins * sizeof(unsigned long long);
    return 0;
}

// Host side of both accumulates, kIdx as in stream_match (B = the pushing streams, n_fleet = the fleet's size).
template <bool kIdx>
static int stream_accumulate_launch(const char *fn, const float *S, int B, int Q, int P, int L, const int32_t *ids,
                                    int n_fleet, const float *ring, const int32_t *seen, int64_t t,
                                    const int64_t *rows, const int32_t *gt_center, int gt_tol, void *acc_place,
                                    void *acc_query, void *acc_multi, void *stream)
{
    LENS_CHECK_ARG(B >= 0 && Q > 0 && P > 0, "%s: bad sizes", fn);
    LENS_CHECK_ARG(L >= 1 && L <= P, "%s: need 1 <= L <= P, got L=%d", fn, L);
    LENS_CHECK_ARG(t >= 0 && gt_tol >= 0, "%s: t and gt_tol must be >= 0", fn);
    LENS_CHECK_ARG((int64_t)B * Q <= 2147483647LL, "%s: too many (stream, row) pairs", fn);
    LENS_CHECK_ARG(B == 0 || (S && seen && gt_center), "%s: NULL S / seen / gt_center", fn);
    LENS_CHECK_ARG(B == 0 || L == 1 || ring, "%s: NULL ring needs L == 1, got L=%d", fn, L);
    if constexpr (kIdx) {
        LENS_CHECK_ARG(n_fleet >= 0, "%s: bad fleet size %d", fn, n_fleet);
        LENS_CHECK_ARG(B == 0 || (ids && rows), "%s: NULL ids / rows", fn);
    }
    void *accs[3] = {acc_place, acc_query, acc_multi};
    for (int m = 0; m < 3; ++m)
        LENS_CHECK_ARG((reinterpret_cast<uintptr_t>(accs[m]) & 7) == 0, "%s: accumulators must be 8-byte aligned", fn);
    if (B == 0 || !(acc_place || acc_query || acc_multi)) return 0;
    SeqPrStreamArgs a{};
    a.S = S; a.ring = ring; a.seen = seen; a.t = t;
    a.B = B; a.Q = Q; a.P = P; a.L = L; a.Po = P - L + 1;
    a.gt_center = gt_center; a.gt_tol = gt_tol;
    for (int m = 0; m < 3; ++m) a.bad[m] = static_cast<unsigned long long *>(accs[m]);     // header word 0
    if (acc_place) a.rec = reinterpret_cast<unsigned *>(static_cast<unsigned long long *>(acc_place) + 2);
    if (acc_multi) {
        a.multi_gtp = static_cast<unsigned long long *>(acc_multi) + 1;
        a.hist = static_cast<unsigned long long *>(acc_multi) + 2;
    }
    cudaStream_t st = as_stream(stream);
    if (acc_query) {
        LENS_CUDA(cudaMallocAsync(&a.key, (size_t)B * Q * sizeof(unsigned long long), st));   // stream-ordered scratch
        LENS_CUDA(cudaMemsetAsync(a.key, 0, (size_t)B * Q * sizeof(unsigned long long), st));
    }
    const long long sms = std::max(sm_count(), 1);
    const long long items = (long long)B * ceil_div(a.Po, kPrTile);
    const unsigned blocks = (unsigned)std::min<long long>(ceil_div64(items, 8), sms * 16);
    const size_t smem = acc_multi ? 2 * kStreamShBins * sizeof(unsigned) : 0;
    if constexpr (kIdx) seqpr_stream_accumulate_ids_kernel<<<blocks, 256, smem, st>>>(a, ids, rows, n_fleet);
    else seqpr_stream_accumulate_kernel<<<blocks, 256, smem, st>>>(a);
    LENS_LAUNCH_CHECK();
    if (acc_query) {
        unsigned long long *q = static_cast<unsigned long long *>(acc_query);
        const unsigned fold_blocks = (unsigned)std::min<long long>(ceil_div64((long long)B * Q, 256), sms * 8);
        if constexpr (kIdx)
            seqpr_stream_query_fold_ids_kernel<<<fold_blocks, 256, 0, st>>>(a, q + 2, q + 1, ids, rows, n_fleet);
        else seqpr_stream_query_fold_kernel<<<fold_blocks, 256, 0, st>>>(a, q + 2, q + 1);
        LENS_LAUNCH_CHECK();
        LENS_CUDA(cudaFreeAsync(a.key, st));
    }
    return 0;
}

extern "C" int lens_seqpr_stream_accumulate(const float *S, int B, int Q, int P, int L, const float *ring,
                                            const int32_t *seen, int64_t t, const int32_t *gt_center, int gt_tol,
                                            void *acc_place, void *acc_query, void *acc_multi, void *stream)
{
    return stream_accumulate_launch<false>("lens_seqpr_stream_accumulate", S, B, Q, P, L, nullptr, B, ring, seen, t,
                                           nullptr, gt_center, gt_tol, acc_place, acc_query, acc_multi, stream);
}

extern "C" int lens_seqpr_stream_accumulate_ids(const float *S, int n, int Q, int P, int L, const int32_t *ids, int B,
                                                const float *ring, const int32_t *seen, const int64_t *rows,
                                                const int32_t *gt_center, int gt_tol, void *acc_place,
                                                void *acc_query, void *acc_multi, void *stream)
{
    return stream_accumulate_launch<true>("lens_seqpr_stream_accumulate_ids", S, n, Q, P, L, ids, B, ring, seen, 0,
                                          rows, gt_center, gt_tol, acc_place, acc_query, acc_multi, stream);
}

extern "C" int lens_seqpr_stream_histogram(const void *acc, int B, int P, int L, int mode, uint64_t *hist,
                                           int64_t *gtp, int64_t *n_bad, void *stream)
{
    LENS_CHECK_ARG(B >= 0 && P > 0 && L >= 1 && L <= P, "lens_seqpr_stream_histogram: bad sizes");
    LENS_CHECK_ARG(mode == LENS_SEQPR_PLACE || mode == LENS_SEQPR_QUERY || mode == LENS_SEQPR_MULTI,
                   "lens_seqpr_stream_histogram: unknown mode %d", mode);
    LENS_CHECK_ARG(acc && hist && gtp && n_bad, "lens_seqpr_stream_histogram: NULL buffer");
    LENS_CHECK_ARG((reinterpret_cast<uintptr_t>(acc) & 7) == 0, "lens_seqpr_stream_histogram: acc must be 8-byte aligned");
    const unsigned long long *a = static_cast<const unsigned long long *>(acc);
    auto *h = reinterpret_cast<unsigned long long *>(hist);
    auto *g = reinterpret_cast<unsigned long long *>(gtp);
    auto *nb = reinterpret_cast<unsigned long long *>(n_bad);
    cudaStream_t st = as_stream(stream);
    if (mode == LENS_SEQPR_PLACE) {
        const long long n = (long long)B * (P - L + 1);
        const long long sms = std::max(sm_count(), 1);
        if (n > 0) {
            seqpr_stream_place_hist_kernel<<<(unsigned)std::min<long long>(ceil_div64(n, 256), sms * 8), 256, 0, st>>>(
                a, n, h, g, nb);
            LENS_LAUNCH_CHECK();
        }
    } else {
        seqpr_stream_add_kernel<<<(unsigned)ceil_div(2 * kStreamBins, 256), 256, 0, st>>>(a, h, g, nb);
        LENS_LAUNCH_CHECK();
    }
    return 0;
}

extern "C" int lens_seqpr_hist_counts(const uint64_t *hist, int L, int n_thresh, int64_t *tp, int64_t *fp,
                                      void *stream)
{
    LENS_CHECK_ARG(L >= 1, "lens_seqpr_hist_counts: need L >= 1, got L=%d", L);
    LENS_CHECK_ARG(n_thresh >= 2 && n_thresh <= kPrMaxThresh,
                   "lens_seqpr_hist_counts: n_thresh must be in [2, %d], got %d", kPrMaxThresh, n_thresh);
    LENS_CHECK_ARG(hist && tp && fp, "lens_seqpr_hist_counts: NULL buffer");
    cudaStream_t st = as_stream(stream);
    unsigned long long *binned = nullptr;
    const size_t bytes = (size_t)2 * n_thresh * sizeof(unsigned long long);
    LENS_CUDA(cudaMallocAsync(&binned, bytes, st));                     // stream-ordered scratch
    LENS_CUDA(cudaMemsetAsync(binned, 0, bytes, st));
    seqpr_stream_bin_kernel<<<1, 1024, 0, st>>>(reinterpret_cast<const unsigned long long *>(hist), L, n_thresh, binned);
    LENS_LAUNCH_CHECK();
    seqpr_prefix_kernel<<<1, 64, 0, st>>>(binned, n_thresh, reinterpret_cast<unsigned long long *>(tp),
                                          reinterpret_cast<unsigned long long *>(fp));
    LENS_LAUNCH_CHECK();
    LENS_CUDA(cudaFreeAsync(binned, st));
    return 0;
}

// Place segments of the bounds count: as in plan_segments, few rows against many places (one camera, 100 000 places)
// are split so that every SM gets warps.  Nothing is merged afterwards (the partial A, E of a row just add up), so a
// segment may be as short as 1 024 places.
static void plan_bounds_segments(long long n_rows, int Po, int &n_seg, int &seg_len, long long &blocks)
{
    const long long sms = std::max(sm_count(), 1), want_warps = sms * 32;
    n_seg = 1;
    if (n_rows < want_warps && Po >= 2048)
        n_seg = (int)std::min<long long>(ceil_div64(want_warps, n_rows), Po / 1024);
    n_seg = std::max(n_seg, 1);
    seg_len = ceil_div(ceil_div(Po, n_seg), 32 * kUnrollR) * (32 * kUnrollR);
    n_seg = ceil_div(Po, seg_len);
    blocks = std::min<long long>(ceil_div64(n_rows * n_seg, 8), sms * 16);
}

// Host side of the three bounds calls, after each has checked its own arguments and filled a's inputs: checks ns and
// the counters, then peak, count and finish on stream-ordered scratch of 12 bytes per row.
template <bool kStream, bool kIdx>
static int rbounds_launch(const char *fn, RecallBoundsArgs &a, const int *ns, int n_ns, int64_t *lo, int64_t *hi,
                          int64_t *n_valid, void *stream)
{
    LENS_CHECK_ARG(ns && n_ns >= 1 && n_ns <= 8, "%s: n_ns must be in [1, 8]", fn);
    for (int i = 0; i < 8; ++i) a.ns[i] = 0;
    for (int i = 0; i < n_ns; ++i) {
        LENS_CHECK_ARG(ns[i] >= 1 && (i == 0 || ns[i] > ns[i - 1]), "%s: ns must be ascending and >= 1", fn);
        a.ns[i] = ns[i];
    }
    LENS_CHECK_ARG(lo && hi && n_valid, "%s: NULL lo / hi / n_valid", fn);
    a.n_ns = n_ns;
    a.lo = reinterpret_cast<unsigned long long *>(lo);
    a.hi = reinterpret_cast<unsigned long long *>(hi);
    a.n_valid = reinterpret_cast<unsigned long long *>(n_valid);
    const long long n_rows = (long long)a.B * a.Qr;
    if (n_rows == 0) return 0;
    cudaStream_t st = as_stream(stream);
    LENS_CUDA(cudaMallocAsync(&a.ae, (size_t)n_rows * (sizeof(unsigned long long) + sizeof(unsigned)), st));
    a.key = reinterpret_cast<unsigned *>(a.ae + n_rows);
    LENS_CUDA(cudaMemsetAsync(a.ae, 0, (size_t)n_rows * sizeof(unsigned long long), st));
    const long long sms = std::max(sm_count(), 1);
    const unsigned row_blocks = (unsigned)std::min<long long>(ceil_div64(n_rows, 256), sms * 8);
    rbounds_peak_kernel<kStream, kIdx><<<(unsigned)std::min<long long>(ceil_div64(n_rows, 8), sms * 16), 256, 0, st>>>(a);
    LENS_LAUNCH_CHECK();
    int n_seg, seg_len;
    long long blocks;
    plan_bounds_segments(n_rows, a.Po, n_seg, seg_len, blocks);
    rbounds_count_kernel<kStream, kIdx><<<(unsigned)blocks, 256, 0, st>>>(a, a.ns[n_ns - 1], n_seg, seg_len);
    LENS_LAUNCH_CHECK();
    rbounds_finish_kernel<<<row_blocks, 256, 0, st>>>(a);
    LENS_LAUNCH_CHECK();
    LENS_CUDA(cudaFreeAsync(a.ae, st));
    return 0;
}

extern "C" int lens_seq_recall_bounds(const float *S, int B, int Q, int P, int L, const uint8_t *gt_dense,
                                      int64_t gt_stream_stride, const int32_t *gt_center, int gt_tol, const int *ns,
                                      int n_ns, int64_t *lo, int64_t *hi, int64_t *n_valid, void *stream)
{
    const char *fn = "lens_seq_recall_bounds";
    LENS_CHECK_ARG(B >= 0 && Q > 0 && P > 0, "%s: bad sizes", fn);
    LENS_CHECK_ARG(L >= 1 && L <= Q && L <= P, "%s: need 1 <= L <= min(Q, P), got L=%d", fn, L);
    LENS_CHECK_ARG((gt_dense != nullptr) != (gt_center != nullptr),
                   "%s: exactly one of gt_dense / gt_center must be given", fn);
    LENS_CHECK_ARG(gt_stream_stride >= 0 && gt_tol >= 0, "%s: gt_stream_stride and gt_tol must be >= 0", fn);
    LENS_CHECK_ARG(B == 0 || S != nullptr, "%s: NULL S", fn);
    LENS_CHECK_ARG((int64_t)B * (Q - L + 1) <= 2147483647LL, "%s: too many (stream, query) pairs", fn);
    RecallBoundsArgs a{};
    a.S = S; a.B = B; a.Q = Q; a.P = P; a.L = L; a.Qr = Q - L + 1; a.Po = P - L + 1;
    a.gt_dense = gt_dense; a.gt_stride = gt_stream_stride; a.gt_center = gt_center; a.gt_tol = gt_tol;
    return rbounds_launch<false, false>(fn, a, ns, n_ns, lo, hi, n_valid, stream);
}

// Checks shared by both streaming forms (B = the pushing streams, n_fleet = the fleet's size when kIdx).
template <bool kIdx>
static int rbounds_stream_args(RecallBoundsArgs &a, const char *fn, const float *S, int B, int Q, int P, int L,
                               const int32_t *ids, int n_fleet, const float *ring, const int32_t *seen, int64_t t,
                               const int64_t *rows, const int32_t *gt_center, int gt_tol)
{
    LENS_CHECK_ARG(B >= 0 && Q > 0 && P > 0, "%s: bad sizes", fn);
    LENS_CHECK_ARG(L >= 1 && L <= P, "%s: need 1 <= L <= P, got L=%d", fn, L);
    LENS_CHECK_ARG(t >= 0 && gt_tol >= 0, "%s: t and gt_tol must be >= 0", fn);
    LENS_CHECK_ARG((int64_t)B * Q <= 2147483647LL, "%s: too many (stream, row) pairs", fn);
    LENS_CHECK_ARG(B == 0 || (S && seen && gt_center), "%s: NULL S / seen / gt_center", fn);
    LENS_CHECK_ARG(B == 0 || L == 1 || ring, "%s: NULL ring needs L == 1, got L=%d", fn, L);
    if constexpr (kIdx) {
        LENS_CHECK_ARG(n_fleet >= 0, "%s: bad fleet size %d", fn, n_fleet);
        LENS_CHECK_ARG(B == 0 || (ids && rows), "%s: NULL ids / rows", fn);
    }
    a = RecallBoundsArgs{};
    a.S = S; a.ring = ring; a.seen = seen; a.t = t; a.ids = ids; a.rows = rows; a.n_fleet = n_fleet;
    a.B = B; a.Q = Q; a.P = P; a.L = L; a.Qr = Q; a.Po = P - L + 1;
    a.gt_center = gt_center; a.gt_tol = gt_tol;
    return 0;
}

extern "C" int lens_seq_recall_bounds_stream(const float *S, int B, int Q, int P, int L, const float *ring,
                                             const int32_t *seen, int64_t t, const int32_t *gt_center, int gt_tol,
                                             const int *ns, int n_ns, int64_t *lo, int64_t *hi, int64_t *n_valid,
                                             void *stream)
{
    const char *fn = "lens_seq_recall_bounds_stream";
    RecallBoundsArgs a;
    if (int rc = rbounds_stream_args<false>(a, fn, S, B, Q, P, L, nullptr, B, ring, seen, t, nullptr, gt_center, gt_tol))
        return rc;
    return rbounds_launch<true, false>(fn, a, ns, n_ns, lo, hi, n_valid, stream);
}

extern "C" int lens_seq_recall_bounds_stream_ids(const float *S, int n, int Q, int P, int L, const int32_t *ids, int B,
                                                 const float *ring, const int32_t *seen, const int64_t *rows,
                                                 const int32_t *gt_center, int gt_tol, const int *ns, int n_ns,
                                                 int64_t *lo, int64_t *hi, int64_t *n_valid, void *stream)
{
    const char *fn = "lens_seq_recall_bounds_stream_ids";
    RecallBoundsArgs a;
    if (int rc = rbounds_stream_args<true>(a, fn, S, n, Q, P, L, ids, B, ring, seen, 0, rows, gt_center, gt_tol))
        return rc;
    return rbounds_launch<true, true>(fn, a, ns, n_ns, lo, hi, n_valid, stream);
}
