/* qa_b200.h — C ABI of the B200-native quantize-and-score library (libqa_b200.so).
 *
 * The reference (johanna-rock/quantization_analysis) is pure Python/NumPy and has no FFI of
 * its own; each entry point below names the reference function(s) whose inner loop it
 * replaces (paths relative to the reference root).  The Python host side in
 * quantization_analysis_b200/ binds these with ctypes and keeps the reference's API.
 *
 * Conventions
 *  - every pointer is a DEVICE pointer owned by the caller (PyTorch allocates); no hidden
 *    allocations, no implicit synchronisation; work is enqueued on `stream` (a cudaStream_t).
 *  - return value 0 = ok, non-zero = error; qa_last_error() returns a thread-local message.
 *  - the small index arrays fmt_order / order / fmt_indices are HOST pointers (copied by value).
 *  - matrices are row-major [rows, cols] with leading dimension `ld` (elements).
 *  - x_dtype: QA_DT_BF16 = raw bf16 bit patterns (uint16), QA_DT_F32 = float32.
 *  - formats are numbered in the reference's MIXED_TILE_FORMATS order
 *    (compression_algorithms/tile_utils.py:8): 0 bf16, 1 bfp8, 2 bfp4, 3 bfp2; fmt_mask bit i
 *    selects format i.  fp0 (all zeros) needs no kernel.
 *  - tiles are 32x32, numbered row-major: tile = tr * tiles_w + tc, tiles_w = ceil(cols/32).
 */
#ifndef QA_B200_H
#define QA_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define QA_DT_BF16 0
#define QA_DT_F32 1

#define QA_METRIC_PCC 0
#define QA_METRIC_MAE 1
#define QA_METRIC_ATOL 2

#define QA_NFMT 4
/* tile-stat table: QA_NSTAT float64 columns, column-major: table[stat * ntiles + tile] */
#define QA_NSTAT 22
#define QA_STAT_SX 0  /* sum x            */
#define QA_STAT_SX2 1 /* sum x*x          */
/* for format f: base = 2 + 5*f; +0 sum y, +1 sum y*y, +2 sum x*y, +3 sum |x-y|, +4 max |x-y| */
#define QA_STAT_FMT(f, k) (2 + 5 * (f) + (k))

#define QA_STATS_FAST 0   /* bf16 input only; exact group-scaled partial sums               */
#define QA_STATS_STRICT 1 /* NumPy-order float64 pairwise sums (bit-faithful to the reference) */
#define QA_STATS_FAST_APPROX_ABS 2 /* as FAST, but sum|x-y| from fp32 group partials (~1e-9 rel.):
                                      enough for pcc/atol-driven assignment and reported mae */

/* State of a numpy.random.Generator(PCG64) (bit_generator.state), resident in device memory.
 * Kernels advance it in place so successive calls continue the same stream. */
typedef struct qa_pcg64 {
    uint64_t state_hi, state_lo; /* 128-bit LCG state   */
    uint64_t inc_hi, inc_lo;     /* 128-bit increment   */
    uint32_t has_uint32;         /* buffered upper half */
    uint32_t uinteger;
} qa_pcg64;

typedef void* qa_stream_t; /* cudaStream_t */

int qa_version(void);
const char* qa_last_error(void);

/* Quantize->dequantize emulation for the selected formats, bit-exact, in one pass over x.
 * Replaces quantization_formats.py:84-164 (quantize_dequantize_bfp_ttnn) and :29-45 (bf16 RNE)
 * as called through quantize_weight_values (:171-194) / Quantizer.quantize (quantizer.py:13-34).
 * out[f] (f in fmt_mask) receives rows*cols bf16 bit patterns, contiguous (ld = cols): every
 * reconstruction has <= 7 explicit mantissa bits, so bf16 holds it exactly. */
int qa_quant_recon(const void* x, int x_dtype, int64_t rows, int64_t cols, int64_t ld,
                   uint32_t fmt_mask, void* const out[QA_NFMT], qa_stream_t stream);

/* qa_quant_recon with the shared exponent along COLUMNS: groups are 16 consecutive rows of one column (rows beyond the
 * end read as zero).  Replaces compression_algorithms/transpose.py:13-33 (quantize x.T, transpose back) without moving
 * the data: for an n-d array pass rows = shape[0], cols = prod(shape[1:]).  The bf16 format (bit 0) is elementwise. */
int qa_quant_recon_cols(const void* x, int x_dtype, int64_t rows, int64_t cols, int64_t ld,
                        uint32_t fmt_mask, void* const out[QA_NFMT], qa_stream_t stream);

/* mxfp4 (which = 0) / nvfp4 (which = 1) scalar proxies: the elementwise maps quantize_weight_values applies for these two
 * formats (quantization_formats.py:171-183; simulate_mxfp4_amax / simulate_nvfp4_amax :254-278 on a block of identical
 * values).  x: bf16 or float32 [n]; out: float32 [n]. */
int qa_scalar_proxy(const void* x, int x_dtype, int64_t n, int which, float* out, qa_stream_t stream);

/* fp8 e4m3fn weights + per-block inverse scales -> float32 (and / or bf16 patterns), the step in front of the path for
 * real checkpoints: hf_model_utils.py:199-215 (_dequantize_tensor_with_scale_inv), block = ceil(shape / scale shape).
 * w_fp8: uint8 [rows, cols]; scale_inv: float32 [scale_rows, scale_cols]; out_f32 / out_bf16: either may be NULL;
 * *inexact_count (device, may be NULL) = products that are not bf16-exact (then the float32 kernels must be used). */
int qa_fp8_block_dequant(const void* w_fp8, const float* scale_inv, int64_t rows, int64_t cols,
                         int64_t scale_rows, int64_t scale_cols, float* out_f32, void* out_bf16,
                         unsigned long long* inexact_count, qa_stream_t stream);

/* Fused quantize + per-tile reconstruction-error statistics (one read of x).
 * Replaces the per-tile sums of mixed_tile_greedy.py:135-220,245-254 and feeds the tensor-level
 * metrics of wq:684-687 / mixed_tile_random.py:135-141.  vec_tail: 0, or for a 1-D input laid
 * out as rows of 32 (tile_utils.py:96-102) the number of valid elements in the last row (strict
 * mode sums that ragged row as its own view, mixed_tile_greedy.py:111-131).
 * QA_STATS_STRICT is bit-equal to the reference's NumPy-order sums.  The fast modes (bf16 input) match them bit for bit in
 * every column whose sum is exactly representable, except sum x^2 (and the bf16 slot's sum y^2 and sum x*y, which are it):
 * <= 1e-13 relative per tile for any finite input.  Groups whose largest |x| is below 2^-51 or at least 2^64 are summed from
 * float32 products like the reference's, so denormal-only groups count and overflowing products give the reference's inf.
 * Only the columns of formats in fmt_mask (and SX/SX2) are written. */
int qa_tile_stats(const void* x, int x_dtype, int64_t rows, int64_t cols, int64_t ld,
                  int64_t vec_tail, uint32_t fmt_mask, int mode, double* table,
                  qa_stream_t stream);

/* qa_tile_stats (fast modes, bf16) restricted to tile rows [tile_row_begin, tile_row_end) of the same table: a large
 * tensor's table can be produced in pieces so that consumers of its first tiles (qa_greedy_init_sums_range) start early. */
int qa_tile_stats_rows(const void* x, int x_dtype, int64_t rows, int64_t cols, int64_t ld,
                       uint32_t fmt_mask, int mode, double* table, int64_t tile_row_begin,
                       int64_t tile_row_end, qa_stream_t stream);

/* Descriptor-array batched variants (SURVEY section 8(b)(8)): one launch for a whole list of tensors - the 768 expert matrices of
 * a MoE layer (cfg5) are 96 tensors per GPU, each worth a 17 us tile-stat kernel.  The caller owns the descriptor array in
 * DEVICE memory (it describes resident buffers, so it is built once per tensor list) and fills the two prefix fields:
 *   item_begin  = sum of qa_tile_stats_items(rows, cols) of the tensors before this one   (tile-stat launch)
 *   block_begin = sum of ceil(ntiles / 256) of the tensors before this one                (delta-record launch)
 * x: bf16 [rows][ld]; table: float64 [QA_NSTAT][ntiles]; init: qa_greedy_init_bytes(ntiles) bytes (only read by the delta launch). */
typedef struct qa_batch_desc {
    const void* x;
    double* table;
    void* init;
    int64_t rows, cols, ld;
    int64_t item_begin;
    int64_t block_begin;
} qa_batch_desc;

/* host helper: CTAs (tile row x 512-column chunk items) the fast tile-stat pass uses for a [rows, cols] tensor */
int64_t qa_tile_stats_items(int64_t rows, int64_t cols);

/* qa_tile_stats (fast modes, bf16 input) for n tensors in one launch; total_items = item_begin + items of the last tensor.
 * Same kernel body per item as qa_tile_stats: the tables are bit-identical to n separate calls. */
int qa_tile_stats_batch(const qa_batch_desc* descs_dev, int n, int64_t total_items, uint32_t fmt_mask, int mode,
                        qa_stream_t stream);

/* qa_greedy_init_deltas for n tensors in one launch (the per-transition delta records of mixed_tile_greedy.py:245-254);
 * total_blocks = block_begin + blocks of the last tensor. */
int qa_greedy_init_deltas_batch(const qa_batch_desc* descs_dev, int n, int64_t total_blocks, const int32_t* fmt_order, int nfmt,
                                qa_stream_t stream);

/* The fast tile-stat pass for inputs that are NOT bf16-exact - what the reference's loader produces from real checkpoints
 * (hf_model_utils.py:199-215,271-281: fp8 e4m3fn weights x per-block inverse scales -> float32 with 24-bit significands).
 * Same table as qa_tile_stats, all four formats (bf16 is a real quantization for these inputs), same lane-owns-a-group
 * layout; the arithmetic follows quantization_formats.py:121-145 on 24-bit mantissas (alignment shift truncates, then RNE)
 * and mixed_tile_greedy.py:147-174 (float32 product arrays x*x, x*y, y*y summed in float64).  sum y, sum y^2, sum |x-y| and
 * max |x-y| equal the reference's NumPy-order float64 sums whenever those are exactly representable; sum x, sum x^2 and
 * sum x*y of 24-bit data are order-dependent in the last float64 bits (<= 1e-13 relative per tile) - the greedy's decision-margin
 * certificate (state[20]) covers that, as for the bf16 kernel's sum x^2.  So is the bf16 slot's sum y^2, whose squares are exact
 * where the reference rounds those below 2^-134 in float32's denormal range.  Groups whose largest |x| is below 2^-51 or at least
 * 2^63 are summed from float32 products throughout, so squares in the denormal range and overflow to inf follow the reference.  mode: QA_STATS_FAST or QA_STATS_FAST_APPROX_ABS.
 * Tile rows [tile_row_begin, tile_row_end) are produced (tile_row_end < 0: all), so a large table can be made in pieces. */
int qa_tile_stats_f32(const float* x, int64_t rows, int64_t cols, int64_t ld, uint32_t fmt_mask, int mode, double* table,
                      int64_t tile_row_begin, int64_t tile_row_end, qa_stream_t stream);

/* qa_fp8_block_dequant fused into the read of qa_tile_stats_f32: 1 byte per element + the scale grid in, table out; the
 * float32 image of the tensor is never written.  w_fp8: uint8 [rows, ld]; scale_inv: float32 [scale_rows, scale_cols];
 * block = ceil(shape / scale shape) (hf_model_utils.py:199-207).  *inexact_count (device, may be NULL; zeroed by the
 * call that starts at tile row 0) = products that are not bf16-exact. */
int qa_tile_stats_fp8(const void* w_fp8, const float* scale_inv, int64_t rows, int64_t cols, int64_t ld,
                      int64_t scale_rows, int64_t scale_cols, uint32_t fmt_mask, int mode, double* table,
                      int64_t tile_row_begin, int64_t tile_row_end, unsigned long long* inexact_count, qa_stream_t stream);

/* NumPy-float32-faithful per-tile scores on zero-padded 32x32 tiles.
 * Replaces tile_utils.py:46-57 (tile_metrics) incl. metrics.py:6-16 (pearson_corr) with the
 * float32 summation orders of NumPy 2.3.5 / OpenBLAS 0.3.30 SkylakeX (SURVEY.md App. B).
 * scores[(metric * QA_NFMT + f) * ntiles + tile], float32, for all three metrics. */
int qa_tile_scores_f32(const void* x, int x_dtype, int64_t rows, int64_t cols, int64_t ld,
                       uint32_t fmt_mask, float* scores, qa_stream_t stream);

/* tile_metrics(ref_tiles, q_tiles, metric) for arbitrary operands (tile_utils.py:46-57): float32 [ntiles][32][32] stacks
 * of reference and candidate tiles -> scores float32 [3][ntiles] (pcc, mae, atol), same float32 orders. */
int qa_tile_scores_pair_f32(const float* ref_tiles, const float* q_tiles, int64_t ntiles, float* scores,
                            qa_stream_t stream);

/* numpy.random.Generator.permutation(n) / .integers(0, k, n) continued from *rng on device
 * (mixed_tile_greedy.py:225,231; mixed_tile_random.py:116,133).  out_perm: int32[n];
 * out_vals: int8[n].  work: int32[2*n] scratch for the permutation. */
int qa_numpy_permutation(qa_pcg64* rng, int64_t n, int32_t* out_perm, int32_t* work,
                         qa_stream_t stream);
int qa_numpy_integers(qa_pcg64* rng, int k, int64_t n, int8_t* out_vals, qa_stream_t stream);

/* Greedy per-tile format assignment under a global metric constraint.
 * Replaces MixedTileGreedyCompression._compress, mixed_tile_greedy.py:135-346, driven by the
 * tile-stat table.  fmt_order[nfmt] = candidate formats (first = base).  numel = element count
 * of the original tensor.  Outputs: assignment int8[ntiles]; counts int64[QA_NFMT];
 * state double[24] = final {sx, sx2, sy, sy2, sxy, sabs, max_abs, value, diagnostics...}.
 * work: at least qa_greedy_work_bytes(ntiles) bytes. */
int64_t qa_greedy_work_bytes(int64_t ntiles);
int qa_greedy_assign(const double* table, int64_t ntiles, double numel, int metric,
                     double threshold, const int32_t* fmt_order, int nfmt, qa_pcg64* rng,
                     int8_t* assignment, int64_t* counts, double* state, void* work,
                     qa_stream_t stream);

/* Same contract as qa_greedy_assign / qa_numpy_permutation, computed by ONE thread-block cluster
 * per tensor (up to 16 CTAs of 256 threads exchanging scan totals through distributed shared
 * memory) instead of one thread: the sequentially-rounded float64 sums are carried by a prefix
 * scan that reproduces every rounding, the accept/reject chain is resolved by speculation to its
 * sequential fixed point, and the NumPy permutation is generated and applied in parallel
 * (csrc/qa_greedy_par.cu).  metric: pcc or mae (atol keeps the sequential kernel).
 * state[6] = flag bits (bit0 sum x, bit1 sum y of the INITIAL sums of a zero-mean tensor were taken
 * as fixed-order tree sums; bit2 sum y ran on a fixed coarser grid during a pass that could carry
 * it across a binade boundary) + 65536 * speculation rounds; state[7] = final metric value;
 * state[11] = max |x - y| of the final assignment; state[20] = a lower bound of min |value - thr| / thr over every decision
 * the chain evaluated (speculative ones included): a caller whose sums may be up to eps away (relative) from the
 * reference's knows the map is the reference's when state[20] > 2 eps; the rest are cycle counters (profiles/).
 * work: at least qa_greedy_par_work_bytes(n) bytes. */
int64_t qa_greedy_par_work_bytes(int64_t n);
int qa_greedy_assign_par(const double* table, int64_t ntiles, double numel, int metric,
                         double threshold, const int32_t* fmt_order, int nfmt, qa_pcg64* rng,
                         int8_t* assignment, int64_t* counts, double* state, void* work,
                         qa_stream_t stream);
int qa_numpy_permutation_par(qa_pcg64* rng, int64_t n, int32_t* out_perm, void* work,
                             qa_stream_t stream);
/* Staging of a greedy run, so that its three independent parts can overlap on different streams:
 *
 *  permutations - the ones that depend only on (seed, tile count) (mixed_tile_greedy.py:228-231): #1 for the base format
 *      (only its stream position matters), #2 for the first candidate format, and - speculatively - #3 for the second
 *      one, which is the permutation of all n tiles whenever pass 2 accepted every tile.  qa_perm_resolve_chain draws #1
 *      and #2, qa_perm_resolve #3, and qa_perm_apply turns the swap targets of #2 and #3 into visiting orders.  The chain
 *      takes them as pre_order int32[(nfmt >= 3 ? 2 : 1)][n] (orders of passes 2 and 3) and pre_rng[same count] (stream
 *      states after #2 and #3); it checks the candidate count before it uses #3 and draws its own otherwise.
 *  init - the data-dependent, permutation-independent part: the sequentially rounded initial sums
 *      (mixed_tile_greedy.py:165-170, qa_greedy_init_sums_range) and the per-tile deltas of every format transition
 *      (qa_greedy_init_deltas).  init: at least qa_greedy_init_bytes(ntiles) bytes; fmt_order / metric must match the
 *      greedy call that consumes it.
 *  chain - qa_greedy_assign_passes; pre_order / pre_rng and init may each be NULL.  pre_order == NULL: the chain draws
 *      every permutation itself.  init == NULL: the call that runs pass 0 computes it into `work` (the delta records and
 *      the initial sums, ahead of the chain on the same stream).  Same results as qa_greedy_assign_par in every
 *      combination.
 *
 * The two halves of one numpy permutation, for callers that pipeline them across streams (a resolve needs the
 * stream state of the previous one; an apply only needs its own swap targets):
 *  qa_perm_resolve - swap targets jarr int32[n] (entries 1..n-1; NULL = only advance the stream) and the stream state
 *      after the permutation (rng_out may alias rng_in).  One cluster.
 *  qa_perm_apply   - out[k] = cand ? cand[perm[k]] : perm[k] from the swap targets, as grid kernels on the whole GPU.
 *      work: at least qa_perm_apply_work_bytes(n) bytes. */
int qa_perm_resolve(const qa_pcg64* rng_in, int64_t n, int32_t* jarr, qa_pcg64* rng_out, qa_stream_t stream);
/* `count` consecutive permutations of n items from one stream in one launch: jarr int32[count][n] (row k written iff bit k
 * of write_mask), rng_out[count] = stream state after each.  rng_out must not alias rng_in. */
int qa_perm_resolve_chain(const qa_pcg64* rng_in, int64_t n, int count, uint32_t write_mask, int32_t* jarr,
                          qa_pcg64* rng_out, qa_stream_t stream);
int64_t qa_perm_apply_work_bytes(int64_t n);
int qa_perm_apply(const int32_t* jarr, int64_t n, const int32_t* cand, int32_t* out, void* work,
                  qa_stream_t stream);
int64_t qa_greedy_init_bytes(int64_t ntiles);
/* The two halves of `init`, for callers that run them on different streams: the sums (one cluster, latency bound) and
 * the delta records (a plain grid kernel) write disjoint parts of it; the greedy needs both.  The sums go over tiles
 * [tile_begin, tile_end) in order: calls must cover [0, ntiles) consecutively on the same `init`; only the call that
 * reaches ntiles needs the whole table (the earlier ones read tiles < tile_end). */
int qa_greedy_init_sums_range(const double* table, int64_t ntiles, int metric, const int32_t* fmt_order,
                              int nfmt, void* init, int64_t tile_begin, int64_t tile_end,
                              qa_stream_t stream);
int qa_greedy_init_deltas(const double* table, int64_t ntiles, int metric, const int32_t* fmt_order, int nfmt,
                          void* init, qa_stream_t stream);
/* The accept/reject chain over passes [pass_begin, pass_end) of the format order (pass 0 = base format); pre_order /
 * pre_rng and init as above.  Consecutive calls covering [0, nfmt) on the same buffers give the results of the single
 * call; the running state travels in `work`.  Lets a caller start the early passes before the speculative third
 * permutation is ready. */
int qa_greedy_assign_passes(const double* table, int64_t ntiles, double numel, int metric,
                            double threshold, const int32_t* fmt_order, int nfmt, qa_pcg64* rng,
                            int8_t* assignment, int64_t* counts, double* state, void* work,
                            const int32_t* pre_order, const qa_pcg64* pre_rng, const void* init,
                            int pass_begin, int pass_end, int flags, qa_stream_t stream);
/* flags bit 0: the caller does not read *rng afterwards.  The reference creates its generator inside _compress and
 * drops it on return (mixed_tile_greedy.py:222-225); when the last pass cannot accept any tile its visiting order is
 * irrelevant, and with this flag its permutation is not drawn at all (*rng is then unspecified).  Maps, counts and
 * sums are unaffected. */
#define QA_GREEDY_SKIP_FINAL_STREAM 1

/* Greedy sweep: the chains of nthr thresholds over ONE table in one launch - what a bytes-versus-metric curve of the greedy
 * needs.  Every chain is the whole run (passes [0, nfmt)) of qa_greedy_assign_passes with thresholds[k] and gives its
 * results bit for bit; the table, the init and the prefetched permutations are shared and only read.
 *  pcc / mae: a grid of nthr clusters (the cluster size qa_greedy_assign_passes would pick, under qa_greedy_cluster_cap);
 *      clusters beyond what fits on the GPU at once queue.  init == NULL: computed once, ahead of the chains, on `stream`;
 *      pre_order / pre_rng == NULL: every chain draws its own permutations.
 *  atol: the one-thread chain of qa_greedy_assign, one block per threshold; pre_order, pre_rng and init are not used.
 * thresholds: DEVICE double[nthr]; rng: DEVICE, the stream state every chain starts from (not modified).
 * Outputs: assignment int8[nthr][ntiles], counts int64[nthr][QA_NFMT], state double[nthr][24] (the atol chain writes
 * state[0..7] only).  work: nthr * qa_greedy_sweep_work_bytes(ntiles, metric) bytes (-1: bad arguments).  flags as above. */
int64_t qa_greedy_sweep_work_bytes(int64_t ntiles, int metric);
int qa_greedy_assign_sweep(const double* table, int64_t ntiles, double numel, int metric, const double* thresholds, int nthr,
                           const int32_t* fmt_order, int nfmt, const qa_pcg64* rng, int8_t* assignment, int64_t* counts,
                           double* state, void* work, const int32_t* pre_order, const qa_pcg64* pre_rng, const void* init,
                           int flags, qa_stream_t stream);

/* Upper bound on the thread-block cluster size of the greedy kernels (1, 2, 4, 8, 16; 0 = automatic: large tensors get
 * 16 CTAs for latency).  A caller with many tensors in flight trades per-tensor latency for SM time with a smaller
 * cluster; results do not depend on the cluster size.  The setting belongs to the CALLING THREAD (thread-local): it
 * applies to the cluster launches that thread enqueues afterwards, so two host threads driving different batches do not
 * see each other's value.  Returns the previous value. */
int qa_greedy_cluster_cap(int max_cluster);

/* Diagnostic timeline: device timestamps (ns) {first start, last end} of the cluster kernels since the last reset -
 * resolve chain, init sums, chain launch containing pass 0, later chain launch - one row of 8 per cluster-size class
 * (log2 of the cluster size, 0..4).  out8_host: HOST array of 40 (may be NULL); reset != 0 re-arms the slots.  A debugging aid,
 * the one synchronous entry point (cudaMemcpy{From,To}Symbol), and only live in a library built with -DQA_STAMP_TIMES: the
 * shipped build compiles the in-kernel timestamps out and this call returns 3. */
int qa_debug_times(unsigned long long* out8_host, int reset);

/* Diagnostic: cycles per call of the cluster collectives used by qa_greedy_assign_par
 * (out double[8] on device: scan+flag exchange, 3-way min, cluster.sync, __syncthreads, pair scan). */
int qa_collective_bench(double* out, int iters, int cluster, qa_stream_t stream);

/* Per-tile threshold assignment for nthr thresholds at once.
 * Replaces mixed_tile_threshold.py:111-123 and scripts/sweep_mixed_tile_threshold.py:145-155.
 * scores: float32[QA_NFMT][ntiles] of ONE metric; order[norder]: formats by ascending bytes;
 * a tile takes the first format whose float32 score passes (>= for pcc, <= otherwise) the
 * float32 threshold, else order[norder-1].  assignment int8[nthr][ntiles],
 * counts int64[nthr][QA_NFMT].  Any nthr >= 1 that fits in int: more than 65535 thresholds are
 * launched in ranges of 65535 on the same stream. */
int qa_threshold_assign(const float* scores, int64_t ntiles, const int32_t* order, int norder,
                        int is_pcc, const float* thresholds, int nthr, int8_t* assignment,
                        int64_t* counts, qa_stream_t stream);

/* Random-assignment search: `iters` uniform assignments drawn from the NumPy stream, each scored
 * from the table (float64 recombination).  Replaces mixed_tile_random.py:132-155.
 * fmt_indices[nfmt]: candidate formats.  sample_metrics double[iters][3] = pcc, mae, atol;
 * sample_counts int64[iters][QA_NFMT].  choices: int8[iters][ntiles] (format index per tile)
 * must be pre-filled when `choices_ready` != 0 (k not a power of two), else it is produced
 * here by jumping the PCG64 stream; *rng is advanced past iters*ntiles draws. */
int qa_random_samples(const double* table, int64_t ntiles, double numel,
                      const int32_t* fmt_indices, int nfmt, int iters, qa_pcg64* rng,
                      int8_t* choices, int choices_ready, double* sample_metrics,
                      int64_t* sample_counts, qa_stream_t stream);

/* Apply a tile assignment: out = per-tile reconstruction in the assigned format (bf16 bits).
 * Replaces the gather of mixed_tile_threshold.py:125-130 / mixed_tile_random.py:74-86 and
 * scripts/reconstruct_mixed_tile_assignment.py:82-137.  assignment < 0 copies x (bf16-rounded). */
int qa_apply_assignment(const void* x, int x_dtype, int64_t rows, int64_t cols, int64_t ld,
                        const int8_t* assignment, void* out_bf16, qa_stream_t stream);

/* Whole-tensor sums for a given assignment (or a single format when assignment == NULL and
 * fmt >= 0), reduced from the table in a fixed order: out double[8] =
 * {sx, sx2, sy, sy2, sxy, sabs, max_abs, 0}.  Feeds wq:684-687-style scoring. */
int qa_assignment_sums(const double* table, int64_t ntiles, const int8_t* assignment, int fmt,
                       double* out, qa_stream_t stream);
/* qa_assignment_sums for nmaps assignment maps at once (one block per map): maps int8 [nmaps][ntiles] -> out double
 * [nmaps][8].  The sweep (scripts/sweep_mixed_tile_threshold.py:700-760) scores every threshold's map with one launch. */
int qa_assignment_sums_batch(const double* table, int64_t ntiles, const int8_t* maps, int nmaps,
                             double* out, qa_stream_t stream);

/* Sums over two arbitrary float32 arrays for compression_algorithms/metrics.py:6-27 (pearson_corr, mae, atol) and
 * the whole-tensor scoring of wq:684-687: out double[8] = {sum a, sum a^2, sum b, sum b^2, sum a*b, sum |a-b|,
 * max |a-b|, 0} in float64 with a fixed reduction tree (b == NULL means b = 0: the fp0 format).
 * work: qa_pair_sums_work_bytes() bytes. */
int64_t qa_pair_sums_work_bytes(void);
int qa_pair_sums(const float* a, const float* b, int64_t n, double* out, void* work, qa_stream_t stream);

/* Whole-tensor NumPy-float32-faithful scores: compression_algorithms/metrics.py:6-27 (pearson_corr, mae, atol) as the
 * reference evaluates them on flattened tensors at wq:684-687, scripts/sweep_mixed_tile_threshold.py:746-749 and
 * mixed_tile_random.py:137-141 - np.mean = pairwise float32 sum, np.dot = OpenBLAS 0.3.30 SkylakeX sdot (64 FMA chains,
 * its folds, the 32-element block and the double-accumulated tail), float32 sqrt / multiply / divide.
 *
 *  qa_pairwise_plan_words / qa_pairwise_plan_build - HOST helpers: the shape of np.add.reduce's pairwise tree over n
 *      contiguous elements (it depends on n only).  plan_host receives qa_pairwise_plan_words(n) int32 words; word 2 is
 *      the node count used by qa_tensor_scores_work_bytes.  The caller copies the plan to the device once per n.
 *  qa_tensor_scores_f32 - x: n elements (bf16 patterns or float32); y: nbatch arrays of n elements, y_stride elements
 *      apart (NULL = all zeros, the fp0 format); plan_dev: the plan on the device, plan_head_host: its first 4 words on
 *      the host.  out float32 [nbatch][4] = {pcc, mae, atol, mean(y)}.  work: qa_tensor_scores_work_bytes(plan[2], nbatch).
 *      Any nbatch >= 1 that fits in int (and whose work buffer fits in memory): more than 65535 items are launched in
 *      ranges of 65535 on the same stream.  x, y and y_stride may have any alignment; 32-byte aligned x, y and
 *      y_stride * sizeof(y) select the vector loads, and from n >= 16384 on the shared-memory pipeline. */
int64_t qa_pairwise_plan_words(int64_t n);
int qa_pairwise_plan_build(int64_t n, int32_t* plan_host);
int64_t qa_tensor_scores_work_bytes(int64_t plan_nnodes, int nbatch);
int qa_tensor_scores_f32(const void* x, int x_dtype, const void* y, int y_dtype, int64_t y_stride, int nbatch, int64_t n,
                         const int32_t* plan_dev, const int32_t* plan_head_host, float* out, void* work,
                         qa_stream_t stream);

/* fp32 -> bf16 bit patterns plus a count of elements that are NOT bf16-exact (low 16 bits != 0).
 * Host helper for the numpy-in API (SURVEY.md H7).  inexact_count: uint64 on device (accumulated). */
int qa_f32_to_bf16_checked(const float* x, int64_t n, void* out_bf16, unsigned long long* inexact_count,
                           qa_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* QA_B200_H */
