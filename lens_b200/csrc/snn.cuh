// Internal definitions shared by the SNN translation units (snn.cu, snn_tc.cu).
#pragma once
#include "common.cuh"

#include <vector>

namespace lens {

// Fixed-point grid of a weight row: w = m * 2^q with |m| < 2^46 (see snn.cu).
constexpr int kFxBits = 46;
// Hidden-spike rows are stored as int8 padded to a multiple of 32 columns
// (16-byte loads, and the K granularity of tcgen05 kind::i8).
constexpr int kHiddenPad = 32;
// Hidden spikes are exchanged between the feature and output kernels as tiles covering up to
// kTileSteps consecutive timesteps of a PAIR of streams (2b, 2b+1), stored in the canonical
// no-swizzle K-major UMMA layout
//   S1[pair][chunk][kc = k / 16][row = 2 * (step in chunk) + (stream & 1)][k % 16]   (int8)
// i.e. a tile is 2 * kTileSteps * Fp contiguous bytes that one cp.async.bulk drops into shared
// memory ready to be the N = 64 B operand of tcgen05.mma.  The two streams are interleaved row by
// row, so accumulator column 2n + s holds step n of stream s and the IAF scan reads both streams'
// values of a step from adjacent registers (packed f32x2 arithmetic).
// Chunks never straddle a query: a query of T steps is ceil(T / kTileSteps) chunks, the last one
// ragged (its missing rows are zero), so every chunk belongs to exactly one similarity row.
constexpr int kTileSteps = 32;
constexpr int kTileRows = 2 * kTileSteps;
__host__ __device__ inline size_t s1_tile_bytes(int Fp) { return (size_t)kTileRows * Fp; }
__host__ __device__ inline int s1_row(int sp, int n) { return 2 * n + sp; }
// byte offset of (step n of stream-in-pair sp, hidden unit k) inside a pair tile
__host__ __device__ inline int s1_byte_in_tile(int sp, int n, int k)
{
    return (k >> 4) * (kTileRows * 16) + s1_row(sp, n) * 16 + (k & 15);
}
// byte offset inside a single-stream staging tile [kc][kTileSteps][16]
__host__ __device__ inline int s1_byte_in_half(int n, int k) { return (k >> 4) * (kTileSteps * 16) + n * 16 + (k & 15); }
// chunk schedule of a stream of `steps` timesteps made of queries of T steps (the last query may be partial)
__host__ __device__ inline int chunks_per_query(int T) { return (T + kTileSteps - 1) / kTileSteps; }
__host__ __device__ inline int n_chunks_of(int steps, int T)
{
    const int fq = steps / T;
    return fq * chunks_per_query(T) + (steps - fq * T + kTileSteps - 1) / kTileSteps;
}
// first step t0 and number of valid steps nc of chunk ch
__host__ __device__ inline void chunk_span(int ch, int steps, int T, int &t0, int &nc)
{
    const int cpq = chunks_per_query(T);
    const int q = ch / cpq, j = ch - q * cpq;
    t0 = q * T + j * kTileSteps;
    int n = T - j * kTileSteps;
    if (n > kTileSteps) n = kTileSteps;
    if (n > steps - t0) n = steps - t0;
    nc = n;
}
// Number of radix-256 balanced digits that cover the 47-bit signed fixed-point weights.
constexpr int kPlanes = 6;

struct SnnHandle {
    int I, F, P, T, Fp, maxB;
    float thr, vmin;
    // CUDA-core (event-driven) operands
    int64_t *Wf_fx = nullptr;   // [I][F]  feature weights, input-major, fixed point
    float *Wf_scale = nullptr;  // [F]     2^q per feature neuron
    int64_t *Wo_fx = nullptr;   // [F][P]  output weights, hidden-major, fixed point
    float *Wo_scale = nullptr;  // [P]     2^q per place
    float *U = nullptr;         // [T][I]  raster uniforms (nullable)
    uint8_t *Uq = nullptr;      // [T][I]  raster thresholds: input i spikes at step t iff pixel > Uq[t][i]
    bool v0_dirty = false;      // IAF#0 state may be non-zero (float path used): raster fast path is off
    float *v0 = nullptr, *v1 = nullptr, *v2 = nullptr;  // membrane potentials [maxB][I|F|P]
    int64_t *counters = nullptr;  // [0] spike overflow, [1] inexact weights
    bool feature_smem_optin = false, output_smem_optin = false;  // CUDA-core kernels opted in to > 48 KB
    int8_t *S1 = nullptr;         // scratch hidden spikes [streams][steps][Fp]
    size_t S1_cap = 0;
    float *ws = nullptr;          // lens_snn_forward_streams: v0 | v1 | v2 of the pushing streams, [ws_cap][I|F|P] each
    int ws_cap = 0;
    // tensor-core operands (built lazily by snn_tc.cu)
    int8_t *Wo_planes = nullptr;  // [P_tiles][kPlanes][Fp/16][128][16] canonical UMMA layout
    int *Wo_npl = nullptr;        // [P_tiles] digit planes in use per place tile (5 or 6)
    int P_tiles = 0;
    int8_t *Wf_planes = nullptr;  // [F_tiles][kPlanes][Ip/16][128][16]
    int *Wf_npl = nullptr;        // [F_tiles]
    int F_tiles = 0, Ip = 0;
    int8_t *S0 = nullptr;         // scratch input-spike pair tiles [pairs][chunks][Ip/16][64][16]
    size_t S0_cap = 0;
    int device = 0;
    // optional per-kernel timing (lens_snn_set_timing)
    struct TimedLaunch { cudaEvent_t start, stop; int kind; };   // kind 0 = feature, 1 = output
    bool timing = false;
    std::vector<TimedLaunch> timed;
};

// pending (uncollected) timed launches kept per handle; lens_snn_get_timing empties the list
constexpr size_t kMaxTimedLaunches = 4096;

// RAII bracket: records start/stop events around a launch when timing is enabled.
struct LaunchTimer {
    SnnHandle *h; cudaStream_t st; SnnHandle::TimedLaunch t; bool on;
    LaunchTimer(SnnHandle *h_, cudaStream_t st_, int kind) : h(h_), st(st_), on(h_->timing)
    {
        if (!on) return;
        t.kind = kind;
        cudaEventCreate(&t.start); cudaEventCreate(&t.stop);
        cudaEventRecord(t.start, st);
    }
    ~LaunchTimer()
    {
        if (!on) return;
        cudaEventRecord(t.stop, st);
        if (h->timed.size() >= kMaxTimedLaunches) {      // nobody collected them: forget the oldest
            cudaEventDestroy(h->timed.front().start);
            cudaEventDestroy(h->timed.front().stop);
            h->timed.erase(h->timed.begin());
        }
        h->timed.push_back(t);
    }
};

// snn_tc.cu
int snn_tc_prepare(SnnHandle *h, cudaStream_t st);
void snn_tc_release(SnnHandle *h);
int snn_tc_output(SnnHandle *h, const int8_t *S1, int nb, int b0, int steps, float *counts,
                  uint8_t *out_steps, cudaStream_t st);
bool snn_tc_supported(const SnnHandle *h);
bool snn_tc_hidden_supported(const SnnHandle *h);
int snn_tc_hidden(SnnHandle *h, const uint8_t *pooled, int nb, int b0, int steps, uint8_t *hidden_steps,
                  cudaStream_t st);

}  // namespace lens
