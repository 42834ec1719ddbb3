/*
 * lens_b200.h -- C ABI of liblens_b200.so, the B200 (sm_100a) implementation of
 * the LENS inference hot path (event binning -> IAF spiking network ->
 * similarity matrix -> sequence matching -> top-N / Recall@N).
 *
 * Conventions
 *   - every function returns int: 0 = ok, <0 = bad argument (see lens_last_error()),
 *     >0 = the cudaError_t that was raised;
 *   - every pointer is a DEVICE pointer unless it says "host"; the caller owns
 *     all buffers, the library owns only what lives inside an opaque handle
 *     (plus stream-ordered scratch, cudaMallocAsync / cudaFreeAsync on the given
 *     stream, inside lens_seqmatch_topk when it splits the places of a query);
 *   - every function is asynchronous and ordered on the cudaStream_t it is given
 *     (pass as void*: 0 = legacy default stream); none synchronises the device;
 *   - handles are not thread-safe (one per stream / rank);
 *   - no C++ types, no torch types, no exceptions cross this boundary;
 *   - there is no CPU fallback: without a CUDA device every compute call fails.
 *
 * Hard limits (a violation is reported as a negative return code, never silently):
 *   lens_snn_create        I <= 1024, F <= 992, every such shape runs on the CUDA-core path (LENS_SNN_SIMT);
 *                          the tensor-core output layer needs 6 * 128 * Fp + 3 * 64 * Fp bytes of shared memory
 *                          (Fp = F rounded up to 32: F <= 224), so LENS_SNN_TC rejects larger F and
 *                          LENS_SNN_AUTO runs it on the CUDA-core path
 *   hidden spikes          <= LENS_MAX_SPIKE (127) per neuron and timestep (int8 transport); larger counts are
 *                          clipped and counted (lens_snn_get_overflow)
 *   lens_seqmatch_topk     N <= 64, 1 <= L <= min(Q, P)
 *   lens_seqmatch_topk_stream
 *                          N <= 64, 1 <= L <= P, Q >= 1, B * Q <= 2^31 - 1; ring non-NULL unless L == 1, seen non-NULL
 *   lens_seqmatch_topk_stream_ids / lens_seqpr_stream_accumulate_ids
 *                          as their lockstep forms with n * Q <= 2^31 - 1; ids [n] i32 of the fleet of B: an id outside
 *                          [0, B) is skipped (never an out-of-bounds access), duplicate ids give unspecified values
 *   lens_snn_forward_streams
 *                          n * (I + F + P) * 4 bytes of handle-owned workspace (n rounded up to even), kept for the
 *                          largest n seen; ids outside [0, max_streams) are skipped, duplicates unspecified
 *   lens_recall / _bounds  at most 8 values of N per call
 *   lens_pr_counts         Qo <= 8192 (one CTA, shared-memory resident)
 *   lens_seqpr_scan / _counts
 *                          1 <= L <= min(Q, P), 2 <= n_thresh <= 4096 (table and histograms in 48 KB of shared memory)
 *   lens_seqpr_stream_*    1 <= L <= P, B * Q <= 2^31 - 1, every sequence sum k an integer in [0, 65 535]
 *                          (LENS_SEQPR_STREAM_BINS - 1; otherwise n_bad), 2 <= n_thresh <= 4096
 *   lens_sad_matrix        npix <= 65 793 (sums stay exact in fp32)
 *   lens_topn_merge        W * N <= 512
 *   lens_bin_events        t_us ascending (lens_check_sorted_u32), x / y 16-byte aligned
 *   lens_bin_event_streams B >= 0, Q >= 0, B * Q <= 2^31 - 1 windows; t_us ascending within every stream
 *                          (lens_check_sorted_segments_u32), x / y 16-byte aligned
 *   lens_snn_forward_float leaves IAF#0 possibly away from rest: the raster fast paths (and the tensor-core hidden
 *                          layer) stay disabled for the handle until lens_snn_reset; the raster feature path also needs
 *                          v_min <= 0 (v_min > 0 moves IAF#0 off rest by itself)
 *
 * Reference sites (relative to the reference repo root) each entry replaces are
 * cited per function.
 */
#ifndef LENS_B200_H
#define LENS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LENS_B200_VERSION_MAJOR 0
#define LENS_B200_VERSION_MINOR 1

/* Largest per-step spike count a neuron may emit and stay exact (int8 operand). */
#define LENS_MAX_SPIKE 127

/* ---- diagnostics -------------------------------------------------------- */
int lens_version(int *major, int *minor);
/* thread-local, never NULL, valid until the next failing call on this thread */
const char *lens_last_error(void);
/* number of SMs of the current device (grid sizing helper for callers) */
int lens_device_sm_count(int *n_sm);
/* kernels launched by this library since it was loaded (host counter; bench evidence) */
int lens_launch_count(int64_t *n_launches);

/* ---- K1: event binning + pooling ----------------------------------------
 * Replaces lens/collect_data.py:186-202 (event_collector + create_images; same
 * loop in lens/tools/manual_eventframe_generator.py:6-14) and the one-hot
 * strided pooling conv of lens/run_model.py:130-137.
 *
 * Events are SoA, sorted by time: t_us[n], x[n], y[n] (polarity already merged,
 * lens/run_speck.py:266).  Window w covers [t0 + w*window_us, t0 + (w+1)*window_us).
 * An event is kept when (x - roi_x0, y - roi_y0) lies inside the roi x roi crop;
 * it increments frame[(yr - index_shift) mod roi][(xr - index_shift) mod roi]
 * (index_shift = 1 is the reference's `frame[y-1, x-1]`).  Counts are stored as
 * uint8: wrap_u8 = 1 wraps modulo 256 (`astype(np.uint8)`), 0 saturates at 255.
 * pooled[w][i*dims + j] = frame[k*i + c][k*j + c], dims = roi / k, c = (k/2) - 1
 * (c = 0 when k == 1).
 *   frames      [n_win][roi][roi] u8   (nullable)
 *   pooled      [n_win][dims*dims] u8  (nullable)
 *   win_events  [n_win] i32 in-ROI events per window (nullable; the reference
 *               skips empty windows, collect_data.py:194,201-202)
 *   win_offsets [n_win + 1] i64 scratch/out: first event index of every window
 */
int lens_bin_events(const uint32_t *t_us, const uint16_t *x, const uint16_t *y, int64_t n_events,
                    uint32_t t0_us, uint32_t window_us, int roi_x0, int roi_y0, int roi, int k,
                    int index_shift, int wrap_u8, uint8_t *frames, uint8_t *pooled,
                    int32_t *win_events, int64_t *win_offsets, int64_t n_win, void *stream);

/* Precondition of lens_bin_events: t_us ascending (the window ranges are found by binary search, like the
 * reference's drain-every-timebin loop sees the events in arrival order, lens/collect_data.py:186-191).
 * Sets *unsorted (device int) to 1 if some t_us[i+1] < t_us[i], else 0.  One streaming pass over t_us
 * (4 B/event), therefore separate from the binning call; lens_b200.ops.bin_events(check_sorted=True)
 * runs it and raises.                                                                                  */
int lens_check_sorted_u32(const uint32_t *t_us, int64_t n, int *unsorted, void *stream);

/* K1 for B independent event streams in one call (launch count independent of B).
 * Stream b owns events [offsets[b], offsets[b+1]) of the SoA arrays; t_us is ascending WITHIN a stream
 * (streams may overlap in time and be stored in any order relative to each other).
 * Window q < Q of stream b covers [t0_us[b] + q*window_us, t0_us[b] + (q+1)*window_us); events of the
 * stream outside all Q windows are ignored.  Crop, index_shift, wrap_u8, pooling and win_events mean
 * exactly what they mean for lens_bin_events; for every b the outputs equal lens_bin_events run on a
 * copy of stream b's events with t0_us[b], byte for byte.  Every window range is clamped to
 * [offsets[b], offsets[b+1]] inside [0, n_events], so malformed offsets never cause a read outside the
 * event arrays (the outputs are then meaningless: check them with lens_check_sorted_segments_u32).
 * B = 0 or Q = 0 returns 0 without launching.
 *   offsets     [B + 1] i64 device, 0 <= offsets[0] <= ... <= offsets[B] <= n_events
 *   t0_us       [B] u32 device
 *   frames      [B][Q][roi][roi] u8 (nullable), pooled [B][Q][dims*dims] u8 (nullable)
 *   win_events  [B][Q] i32 (nullable)
 *   win_offsets [B][Q + 1] i64 scratch/out: absolute first event index of each window + end of the last */
int lens_bin_event_streams(const uint32_t *t_us, const uint16_t *x, const uint16_t *y, int64_t n_events,
                           const int64_t *offsets, const uint32_t *t0_us, int B, int Q, uint32_t window_us,
                           int roi_x0, int roi_y0, int roi, int k, int index_shift, int wrap_u8,
                           uint8_t *frames, uint8_t *pooled, int32_t *win_events, int64_t *win_offsets,
                           void *stream);
/* Precondition of lens_bin_event_streams.  *bad (device int) = 1 if some offsets[b] > offsets[b+1],
 * offsets[0] < 0, offsets[B] > n, or t_us descends inside a stream (a descent where a new stream starts is
 * allowed); else 0.  One streaming pass over t_us; memory-safe for any offsets content.  t_us 16-byte
 * aligned.  lens_b200.ops.bin_event_streams(check_sorted=True) runs it and raises.                      */
int lens_check_sorted_segments_u32(const uint32_t *t_us, int64_t n, const int64_t *offsets, int B, int *bad,
                                   void *stream);

/* Pooling alone (frames already exist, e.g. decoded PNGs):
 * frames [n][roi][roi] u8 -> pooled [n][dims*dims] u8.  lens/run_model.py:130-137. */
int lens_pool_frames(const uint8_t *frames, int64_t n, int roi, int k, uint8_t *pooled,
                     void *stream);

/* ---- K2 + K3: the spiking network --------------------------------------
 * Stands where `self.sinabs_model` stands (lens/run_model.py:139-156,238):
 *   IAF#0 -> Linear(I->F, no bias) -> IAF#1 -> Linear(F->P, no bias) -> IAF#2
 * with sinabs IAFSqueeze semantics (spike_threshold = thr, MultiSpike,
 * MembraneSubtract, min_v_mem = v_min), lens/src/blitnet.py:59-64 weights.
 * The handle owns fixed-point copies of the weights and the membrane potentials
 * v0[B][I], v1[B][F], v2[B][P], which persist across calls exactly like the
 * reference's (it never calls reset_states()).
 *   W_feat [F][I] f32, W_out [P][F] f32, U [T][I] f32 (the sub-sampled columns of
 *   dataset.py:120-121's seed-50 `torch.rand(T, roi*roi)`; nullable if only
 *   lens_snn_forward_float is used).
 * *n_inexact (host, nullable) receives the number of weights that needed rounding
 * to the 46-bit-per-row fixed-point grid (0 => every contraction is exact).      */
int lens_snn_create(int I, int F, int P, int T, float thr, float v_min, const float *W_feat,
                    const float *W_out, const float *U, int max_streams, void **handle,
                    int64_t *n_inexact, void *stream);
int lens_snn_destroy(void *handle);
/* sinabs Network.reset_states(): zero all membrane potentials. */
int lens_snn_reset(void *handle, void *stream);
/* Per-stream sinabs reset_states(): zero v0/v1/v2 of every stream b < max_streams with mask[b] != 0.
 *   mask [max_streams] u8 device.
 * Other streams' state, the overflow counter and the forward_float flag (IAF#0 off rest) are untouched.
 * One launch whatever the number of streams.                                                            */
int lens_snn_reset_streams(void *handle, const uint8_t *mask, void *stream);
/* copy membrane potentials out (any pointer nullable): v0 [B][I], v1 [B][F], v2 [B][P] */
int lens_snn_get_state(void *handle, float *v0, float *v1, float *v2, void *stream);
/* overflow[0] (device, i64) counts per-step spike counts that exceeded LENS_MAX_SPIKE */
int lens_snn_get_overflow(void *handle, int64_t *overflow, void *stream);

/* Optional per-kernel timing (bench.py's roofline): when enabled every feature- / output-layer
 * launch is bracketed by cudaEvents on its own stream.  lens_snn_get_timing waits for the recorded
 * events (host pointers), returns the accumulated milliseconds and launch counts, and clears them. */
int lens_snn_set_timing(void *handle, int enable);
int lens_snn_get_timing(void *handle, float *feature_ms, float *output_ms, int64_t *n_feature,
                        int64_t *n_output);

/* mode for lens_snn_forward: which output-layer kernel runs */
#define LENS_SNN_AUTO 0   /* pick by problem size                      */
#define LENS_SNN_SIMT 1   /* event-driven CUDA-core kernel             */
#define LENS_SNN_TC   2   /* tcgen05 digit-plane kernel (batched)      */

/* The per-query loop of lens/run_model.py:229-246 for B independent streams of Q
 * queries each, fed by the raster of lens/src/dataset.py:14-51,118-125:
 *   p = pooled / 255;  input spike at step t = (U[t][i] < p[i]);  T steps per query;
 *   counts[b][q][p] = number of output spikes of place p during query q.
 * Continues from the handle's current state (carry-over across queries and calls).
 *   pooled        [B][Q][I] u8
 *   counts        [B][Q][P] f32
 *   hidden_steps  [B][Q*T][F]  u8, nullable (debug / tests)
 *   out_steps     [B][Q*T][P]  u8, nullable (debug / tests)                      */
int lens_snn_forward(void *handle, const uint8_t *pooled, int B, int Q, float *counts,
                     uint8_t *hidden_steps, uint8_t *out_steps, int mode, void *stream);

/* Same for the sub-range [b0, b0 + nb) of the handle's streams (pooled / counts / debug buffers start
 * at stream b0): lets a caller pipeline host->device copies of one group of streams with the
 * computation of the previous group.  b0 must be even (streams are tiled in pairs). */
int lens_snn_forward_range(void *handle, const uint8_t *pooled, int b0, int nb, int Q, float *counts,
                           uint8_t *hidden_steps, uint8_t *out_steps, int mode, void *stream);

/* lens_snn_forward for the streams ids[0..n) of the handle, in any order, each advancing from its own state; every
 * other stream's state is untouched.  pooled [n][Q][I] u8 and counts [n][Q][P] f32 are by position (row i is stream
 * ids[i]); ids [n] i32 device.  The rows ids[i] of v0 / v1 / v2 are gathered into a handle-owned workspace, run through
 * the same kernels as lens_snn_forward (mode as there; the counts equal those of lens_snn_forward on the same state),
 * and scattered back: two launches more than lens_snn_forward, 2 * 2 * n * (I + F + P) * 4 bytes of extra traffic.
 * The workspace grows on the first call with a larger n (a cudaMalloc) and is freed with the handle.  n = 0 or Q = 0
 * returns 0 without launching.                                                                                   */
int lens_snn_forward_streams(void *handle, const uint8_t *pooled, const int32_t *ids, int n, int Q, float *counts,
                             int mode, void *stream);

/* Operator seam `sinabs_model(x)` (lens/run_model.py:238) for an arbitrary float
 * raster: x [B][steps][I] f32 (already pooled), spikes_out [B][steps][P] f32.     */
int lens_snn_forward_float(void *handle, const float *x, int B, int steps, float *spikes_out,
                           void *stream);

/* ---- K4: sequence matching + top-N --------------------------------------
 * Replaces lens/run_model.py:248-254 (conv2d with eye(L), / L, transpose) and the
 * selection half of lens/src/metrics.py:183-226 (argsort(0)[-K:]).
 *   S [B][Q][P] f32 similarity (spike counts).  Qo = Q - L + 1, Po = P - L + 1.
 *   D[b][r][q] = (sum_{j<L} S[b][q+j][r+j]) / L
 *   D_out   [B][Po][Qo] f32, nullable (rows = database, as the reference returns it)
 *   top_val [B][Qo][N] f32, top_idx [B][Qo][N] i32: the N largest D[b][.][q],
 *           ordered by (value desc, index desc) == np.argsort(kind='stable')[-N:][::-1];
 *           missing entries (N > Po) are -inf / -1.
 * L >= 1 (the reference's L == 0 branch returns S itself and is handled by the caller). */
int lens_seqmatch_topk(const float *S, int B, int Q, int P, int L, int N, float *D_out,
                       float *top_val, int32_t *top_idx, void *stream);

/* K4 across calls, for live streams that deliver a few rows at a time.  All B streams advance in lockstep; number
 * a stream's rows g = 0, 1, 2, ... since its last reset.  New row g closes the sequence column
 *   D_g[r] = (1/L) * sum_{j<L} S[g - L + 1 + j][r + j],   r in [0, P - L + 1)
 * (same arithmetic and order as lens_seqmatch_topk).  It is valid once the stream has seen L rows (g >= L - 1);
 * a warm-up row gets -inf / -1 in every slot.  Fed any chunking of the same rows, the valid rows equal the columns
 * of one lens_seqmatch_topk over all of them, bit for bit.
 *   S       [B][Q][P] f32: the Q new rows of every stream
 *   ring    [B][L-1][P] f32, caller-owned: the last L-1 rows of every stream, row g at slot g mod (L-1), where g
 *           counts rows pushed (t), not rows since the reset; NULL allowed iff L == 1.  Need not be initialised.
 *   seen    [B] i32: rows seen since the stream's reset, saturating at L-1 (0 = fresh / just reset)
 *   t       rows pushed so far (the same for every stream; the caller adds Q after each call)
 *   top_val [B][Q][N] f32, top_idx [B][Q][N] i32: row q = the sequence ending at new row q
 * Matches first, then stores the last min(Q, L-1) rows of S into the ring and advances seen (stream order).
 * Two launches per call (one when L == 1), three when the places of a row are split into segments (the
 * segmented kernel and lens_topn_merge's kernel); never more with B.  B = 0 returns 0 without launching.  */
int lens_seqmatch_topk_stream(const float *S, int B, int Q, int P, int L, int N, float *ring, int32_t *seen,
                              int64_t t, float *top_val, int32_t *top_idx, void *stream);
/* The same for any subset of a fleet of B streams, in any order: the n streams ids[0..n) each push Q new rows, and
 * every other stream keeps its ring rows, seen and row counter.  Stream ids[i]'s rows are numbered by its own counter:
 *   S       [n][Q][P] f32, row i = stream ids[i]; top_val / top_idx [n][Q][N] by position, as above
 *   ids     [n] i32 device, distinct fleet indices in [0, B)
 *   ring    [B][L-1][P], seen [B] as above (row g of stream b at slot g mod (L-1), g counted by rows[b])
 *   rows    [B] i64 device: rows pushed to each stream (replaces the scalar t; a lockstep session has rows[b] = t)
 * Matches, then appends to the ring, then advances seen[ids[i]] (saturating) and rows[ids[i]] += Q (stream order).
 * For each pushed stream the result is exactly that of lens_seqmatch_topk_stream on that one stream with t = rows[b].
 * Three launches per call (two when L == 1), four when the places of a row are split into segments; never more with
 * n.  n = 0 returns 0 without launching.                                                                        */
int lens_seqmatch_topk_stream_ids(const float *S, int n, int Q, int P, int L, int N, const int32_t *ids, int B,
                                  float *ring, int32_t *seen, int64_t *rows, float *top_val, int32_t *top_idx,
                                  void *stream);

/* Recall@N counters (lens/src/metrics.py:213-224 + lens/run_model.py:301-302).
 * Ground truth is either dense, gt_dense [B or 1][Po][Qo] u8 (gt_stream_stride = Po*Qo
 * or 0 to share one matrix), or a band: gt_center [B][Qo] i32 (-1 = query has no
 * match) with |idx - center| <= gt_tol counting as a hit.  Exactly one is non-NULL.
 *   ns      [n_ns] host ints, ascending, each <= N (e.g. 1,5,10,15,20,25)
 *   hits    [n_ns] i64 device, ACCUMULATED (zero it first): queries with a hit in top-n
 *   n_valid [1]    i64 device, ACCUMULATED: queries that have at least one positive  */
int lens_recall(const int32_t *top_idx, int B, int Qo, int Po, int N, const uint8_t *gt_dense,
                int64_t gt_stream_stride, const int32_t *gt_center, int gt_tol, const int *ns,
                int n_ns, int64_t *hits, int64_t *n_valid, void *stream);

/* Final top-N merge for a PLACE-sharded database (BASELINE config 5: "NCCL all-gather of database
 * representations + top-N merge"): every shard ranks its own range of places with lens_seqmatch_topk, the
 * W per-shard lists of a query are gathered, and the global list is the N best of their union under the
 * same order as lens/src/metrics.py:218 under the deterministic rule (value desc, place index desc).
 *   val, idx [W][M][N] device (idx = GLOBAL place index, -1 = empty slot), M = streams * queries,
 *   out_val, out_idx [M][N] device.  W * N <= 512.                                                       */
int lens_topn_merge(const float *val, const int32_t *idx, int W, int64_t M, int N, float *out_val,
                    int32_t *out_idx, void *stream);

/* Tie-aware bounds of Recall@N (lens/src/metrics.py:218 ranks with numpy's default, unstable argsort, so the
 * reference's number is defined only up to the order of equal similarities): over every such order,
 *   lo [n_ns] i64 device, ACCUMULATED: queries that hit in the top ns[i] whatever the order,
 *   hi [n_ns] i64 device, ACCUMULATED: queries that hit for some order,
 *   n_valid [1] i64 device, ACCUMULATED: queries with at least one positive (metrics.py:214-216).
 * D, GT [Po][Qo] (rows = database, the matrices recallAtK receives), ns host ints ascending.          */
int lens_recall_bounds(const float *D, const uint8_t *GT, int Po, int Qo, const int *ns, int n_ns,
                       int64_t *lo, int64_t *hi, int64_t *n_valid, void *stream);

/* Precision-recall counters of lens/src/metrics.py:21-139 (createPR, matching='single'), used by
 * lens/run_model.py:319-327 with n_thresh = 100.  S and GT are [Po][Qo] (rows = database), exactly the
 * matrices the reference passes (after its transposes).  Per query column the best match is the FIRST
 * row attaining the maximum (np.argmax); thresholds are np.linspace(max, min, n_thresh) over the best
 * similarities, evaluated like numpy (>= 2.0) in the dtype of the caller's matrix: thresh_f64 = 0 for a
 * float32 matrix (float32 arithmetic and comparison), 1 for float64, integer or bool matrices (float64;
 * exact when every value is representable in float32, the type S is read in).
 *   tp, fp [n_thresh] i64 device: true / false positives with best >= threshold
 *   gtp    [1] i64 device: number of queries that have a positive at all (GT.any(0))             */
int lens_pr_counts(const float *S, const uint8_t *GT, int Po, int Qo, int n_thresh, int64_t *tp,
                   int64_t *fp, int64_t *gtp, void *stream, int thresh_f64);
/* The same for matching='multi' (lens/src/metrics.py:63-91): every entry of S counts, thresholds are
 * np.linspace(S.max(), S.min(), n_thresh) (thresh_f64 as above), gtp = count_nonzero(GT).  tp, fp, gtp are
 * overwritten.                                                                                              */
int lens_pr_counts_multi(const float *S, const uint8_t *GT, int Po, int Qo, int n_thresh, int64_t *tp,
                         int64_t *fp, int64_t *gtp, void *stream, int thresh_f64);

/* Fleet precision-recall: createPR's counts for B streams, straight from the spike counts S [B][Q][P] f32.
 * D_b[p][q] = (sum_{j<L} S[b][q+j][p+j]) / L is recomputed exactly as lens_seqmatch_topk computes it and never
 * written.  The fleet's matrix is the streams' matrices concatenated along createPR's column axis:
 *   LENS_SEQPR_PLACE  createPR(D_b.T, GT_b.T, 'single') at B = 1 (lens/run_model.py:321): a column per (stream,
 *                     place), its best query is the FIRST maximum (lowest query index); gtp = places with a positive
 *   LENS_SEQPR_QUERY  createPR(D_b, GT_b, 'single') at B = 1 (the SAD path, lens/src/sad.py): a column per (stream,
 *                     query), its best place is the first maximum (lowest place index); gtp = queries with a positive
 *   LENS_SEQPR_MULTI  createPR(D_b, GT_b, 'multi'): every entry; gtp = positive entries
 * Thresholds: np.linspace(max, min, n_thresh) of the float32 values (numpy's float32 recipe, as lens_pr_counts
 * with thresh_f64 = 0) over the whole fleet.  Ground truth as lens_recall: gt_dense [B or 1][Po][Qo] u8
 * (gt_stream_stride = Po*Qo, or 0 to share one matrix) or gt_center [B][Qo] i32 (< 0: no positive; else the
 * places |p - center| <= gt_tol), exactly one non-NULL.  Finite S only.
 *   lens_seqpr_records_bytes  *bytes (host) = the records a call needs: 5*B*Po (place), 9*B*Qo (query), 0 (multi)
 *   lens_seqpr_scan    one read of S (and GT).  records [bytes] 8-byte aligned, written (NULL allowed in multi
 *                      mode); extremes [2] u64 = {max key, ~min key} of the order-preserving float keys, MERGED by
 *                      max (zero them before the first call); gtp [1] i64 ACCUMULATED.  Groups of streams (or ranks,
 *                      by an all-reduce MAX of extremes) scanned into one extremes / gtp form one fleet.
 *   lens_seqpr_counts  thresholds from the merged extremes; every record (multi: every entry, a second read of
 *                      S) binned once.  tp, fp [n_thresh] i64 ACCUMULATED: true / false positives with value >=
 *                      threshold i.  The same S, sizes, mode, GT and records as the scan.
 * One launch per scan (two in query mode) and two per count, whatever B; stream-ordered scratch of 16 B per
 * threshold in lens_seqpr_counts.  B = 0 returns 0 without launching.                                        */
#define LENS_SEQPR_PLACE 0
#define LENS_SEQPR_QUERY 1
#define LENS_SEQPR_MULTI 2
int lens_seqpr_records_bytes(int B, int Q, int P, int L, int mode, int64_t *bytes);
int lens_seqpr_scan(const float *S, int B, int Q, int P, int L, int mode, const uint8_t *gt_dense,
                    int64_t gt_stream_stride, const int32_t *gt_center, int gt_tol, void *records,
                    uint64_t *extremes, int64_t *gtp, void *stream);
int lens_seqpr_counts(const float *S, int B, int Q, int P, int L, int mode, const uint8_t *gt_dense,
                      int64_t gt_stream_stride, const int32_t *gt_center, int gt_tol, const void *records,
                      const uint64_t *extremes, int n_thresh, int64_t *tp, int64_t *fp, void *stream);

/* Session precision-recall of a live fleet (lens_seqmatch_topk_stream), accumulated push by push in bounded memory.
 * A stream's session matrix has its valid rows as query columns, in push order (warm-up rows are never columns);
 * fleets and ranks concatenate along createPR's column axis, in the same three modes as the fleet calls above.
 * Every D entry is acc / L with acc an integer-valued spike sum; for 0 <= acc < LENS_SEQPR_STREAM_BINS the value is a
 * strictly increasing function of k = acc, so the curve depends on k only.  An entry outside that range, or not
 * integer-valued, is counted in n_bad and makes the session's numbers invalid.
 *   lens_seqpr_stream_bytes      *bytes (host) = the size of one mode's accumulator: 16 + 4*B*(P-L+1) (place) or
 *                                16 + 16*LENS_SEQPR_STREAM_BINS (query, multi).  Zeroed memory is an empty session.
 *   lens_seqpr_stream_accumulate folds the valid new rows of one push into the accumulators of the tracked modes
 *                                (NULL = not tracked; 8-byte aligned).  S, sizes, ring, seen and t as for the
 *                                lens_seqmatch_topk_stream call of the same push, which must come AFTER this one (it
 *                                advances seen and overwrites ring slots).  gt_center [B][Q] i32: the expected place
 *                                of each new row (< 0: no positive), positives |p - center| <= gt_tol.  One launch,
 *                                two when the query mode is tracked; never more with B.
 *   lens_seqpr_stream_accumulate_ids
 *                                the same for the push of lens_seqmatch_topk_stream_ids (S, n, ids, B, ring, seen, rows
 *                                as for that call, which must come AFTER this one); gt_center [n][Q] by position, the
 *                                accumulators sized for the fleet of B.  Launches as above; n = 0 launches nothing.
 *   lens_seqpr_stream_histogram  one accumulator -> hist [2][LENS_SEQPR_STREAM_BINS] u64 (positives | negatives per
 *                                k), gtp [1], n_bad [1], all ACCUMULATED.  Sums of these over ranks form one fleet.
 *   lens_seqpr_hist_counts       tp, fp [n_thresh] i64 ACCUMULATED: thresholds np.linspace(max, min, n_thresh) of the
 *                                float32 values fl(k / L) of the lowest and highest non-empty k (numpy's float32
 *                                recipe); nothing is added for an empty histogram.  2 <= n_thresh <= 4096.      */
#define LENS_SEQPR_STREAM_BINS 65536
int lens_seqpr_stream_bytes(int B, int P, int L, int mode, int64_t *bytes);
int lens_seqpr_stream_accumulate(const float *S, int B, int Q, int P, int L, const float *ring, const int32_t *seen,
                                 int64_t t, const int32_t *gt_center, int gt_tol, void *acc_place, void *acc_query,
                                 void *acc_multi, void *stream);
int lens_seqpr_stream_accumulate_ids(const float *S, int n, int Q, int P, int L, const int32_t *ids, int B,
                                     const float *ring, const int32_t *seen, const int64_t *rows,
                                     const int32_t *gt_center, int gt_tol, void *acc_place, void *acc_query,
                                     void *acc_multi, void *stream);
int lens_seqpr_stream_histogram(const void *acc, int B, int P, int L, int mode, uint64_t *hist, int64_t *gtp,
                                int64_t *n_bad, void *stream);
int lens_seqpr_hist_counts(const uint64_t *hist, int L, int n_thresh, int64_t *tp, int64_t *fp, void *stream);

/* Sum-of-absolute-differences baseline, lens/src/sad.py:25-42: dist[q][r] = sum_p |a[q][p] - b[r][p]|
 * (torch.cdist(a, b, p=1) on float32 copies of uint8 frames; the sums are integers < 2^24, hence exact
 * in fp32 in any order).  a [Q][npix] u8 (query frames), b [R][npix] u8 (reference frames),
 * dist [Q][R] f32.  lens_reciprocal: out[i] = 1.0f / in[i] (IEEE, numpy's `1 / dist`).             */
int lens_sad_matrix(const uint8_t *a, const uint8_t *b, int Q, int R, int npix, float *dist, void *stream);
int lens_reciprocal(const float *in, int64_t n, float *out, void *stream);

/* Online matcher of the event-driven deployment, lens/run_speck.py:155-226.
 *
 * lens_online_accumulate: one readout (run_speck.py:159-164, 188-198): sum[i] += (int32)counts[i]; when
 * row_out != NULL also row_out[i] = floor(sum[i] / div) (`vector // 4`, the averaged sequence row).
 *   sum [P] i32 device (running spike counts, NOT cleared between rows - the reference clears it only
 *   after a match), counts [P] f32 device (integer-valued spike counts of one readout interval).
 * lens_online_match: run_speck.py:200-204: result = scipy.signal.convolve2d(seq.T, eye(L), mode='same') / L
 * and its per-column first-maximum argmax:
 *   result[p][r] = (1/L) * sum_{a<L} seq[r + o - a][p + o - a],  o = (L-1)/2, zero outside the matrix.
 *   seq [R][P] i32 device (sequence rows, oldest first), result [P][R] f64 device (integer sums, one
 *   IEEE float64 division), argmax [R] i32 device.  1 <= L, R <= 64.                                */
int lens_online_accumulate(int32_t *sum, const float *counts, int P, int div, int32_t *row_out, void *stream);
int lens_online_match(const int32_t *seq, int R, int P, int L, double *result, int32_t *argmax, void *stream);

/* Event-driven frame representation, lens/tools/dvstools.py:279-349 (tool='simple_rep').
 *
 * lens_event_windows: index ranges of the frames.  A frame that starts at time c holds the events with
 * |t - c| <= interval (float64, the reference's own expression); the first later event that is not a hot
 * pixel closes it, is dropped, and its timestamp is the next frame's c.  Frame 0 starts at `start`
 * (events with t < start are skipped), or at t[0] when use_first_event != 0 (the reference's offset == 0
 * case).  The frame still open at the end of the stream is not reported (the reference never saves it).
 *   t [n] f64 device, seconds, ascending; x, y [n] u16 device
 *   lut [sensor_h][sensor_w] i16 device: -2 hot pixel (event ignored entirely), -1 no slot, >= 0 slot
 *   win_begin, win_end [max_windows] i64 device, win_t0 [max_windows] f64 device, n_windows [1] i64 device
 *   unsorted: nullable [1] i32 device, set to 1 when t is not ascending (the ranges are then meaningless)
 * lens_bin_events_lut: frames[w][slot] = (weight * #{events of range w whose pixel maps to slot}) mod 256
 * (`frame_data[index] += accum_factor` on a uint8 vector, dvstools.py:310-322).
 *   counts [n_windows][n_slots] u32 device scratch, frames [n_windows][n_slots] u8 device;
 *   events_per_window_hint only sizes the grid.  x / y 16-byte aligned, n_slots <= 8192.              */
int lens_event_windows(const double *t, const uint16_t *x, const uint16_t *y, int64_t n_events, const int16_t *lut,
                       int sensor_w, int sensor_h, int use_first_event, double start, double interval,
                       int64_t max_windows, int64_t *win_begin, int64_t *win_end, double *win_t0,
                       int64_t *n_windows, int *unsorted, void *stream);
int lens_bin_events_lut(const uint16_t *x, const uint16_t *y, const int16_t *lut, int sensor_w, int sensor_h,
                        const int64_t *win_begin, const int64_t *win_end, int64_t n_windows, int n_slots, int weight,
                        int64_t events_per_window_hint, uint32_t *counts, uint8_t *frames, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* LENS_B200_H */
