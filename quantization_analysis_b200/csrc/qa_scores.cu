// NumPy-float32-faithful per-tile scores (pcc / mae / atol) on zero-padded 32x32 tiles.
//
// The reference scores tiles with float32 NumPy calls (tile_utils.py:46-57 -> metrics.py:6-16),
// so the per-tile values - and the threshold decisions taken on them in float32 - depend on the
// library's summation orders.  This kernel evaluates exactly those orders (SURVEY.md App. B):
//   np.mean / reduce : pairwise sum, 128-element leaves with 8 strided accumulators
//   np.dot (sdot)    : 64 FMA chains (4 vectors x 16 lanes) over the flattened tile, then the
//                      OpenBLAS SkylakeX fold  l+8 | ((A0+A1)+A2)+A3 | l+4 | (v0+v1)+(v2+v3)
// One warp owns one tile; lane c owns column c, so each lane carries the even-row and odd-row
// FMA chains of its column and the folds are warp shuffles.
#include "qa_common.cuh"

namespace qa {

constexpr int SCP = 33;
constexpr int SC_WARPS = 4;

// pairwise float32 sum of the 1024 tile elements; `get(row, col)` supplies them.
template <typename F>
__device__ __forceinline__ float pairwise1024(F get, int lane) {
    const int b = lane >> 2, p = lane & 3;
    float r0, r1;
    {
        // accumulators k0 = 2p, k1 = 2p+1 of leaf b (rows 4b..4b+3); element j = k + 8 s
        const int k0 = 2 * p;
        r0 = get(4 * b, k0);
        r1 = get(4 * b, k0 + 1);
#pragma unroll
        for (int s = 1; s < 16; ++s) {
            const int j = k0 + 8 * s;
            r0 = __fadd_rn(r0, get(4 * b + (j >> 5), j & 31));
            r1 = __fadd_rn(r1, get(4 * b + ((j + 1) >> 5), (j + 1) & 31));
        }
    }
    float v = __fadd_rn(r0, r1);
    v = __fadd_rn(v, __shfl_xor_sync(0xFFFFFFFFu, v, 1));
    v = __fadd_rn(v, __shfl_xor_sync(0xFFFFFFFFu, v, 2));   // leaf sum
    v = __fadd_rn(v, __shfl_xor_sync(0xFFFFFFFFu, v, 4));
    v = __fadd_rn(v, __shfl_xor_sync(0xFFFFFFFFu, v, 8));
    v = __fadd_rn(v, __shfl_xor_sync(0xFFFFFFFFu, v, 16));
    return v;
}

// OpenBLAS-SkylakeX sdot fold of the per-lane even-row / odd-row chains.
__device__ __forceinline__ float sdot_fold(float accE, float accO, int lane) {
    const float hE = __fadd_rn(accE, __shfl_down_sync(0xFFFFFFFFu, accE, 8));
    const float hO = __fadd_rn(accO, __shfl_down_sync(0xFFFFFFFFu, accO, 8));
    const float h1 = __shfl_sync(0xFFFFFFFFu, hE, (lane + 16) & 31);
    const float h3 = __shfl_sync(0xFFFFFFFFu, hO, (lane + 16) & 31);
    const float s = __fadd_rn(__fadd_rn(__fadd_rn(hE, h1), hO), h3);       // valid on lanes 0..7
    const float q = __fadd_rn(s, __shfl_down_sync(0xFFFFFFFFu, s, 4));     // valid on lanes 0..3
    const float a = __fadd_rn(q, __shfl_down_sync(0xFFFFFFFFu, q, 1));     // lanes 0 and 2
    const float res = __fadd_rn(a, __shfl_down_sync(0xFFFFFFFFu, a, 2));   // lane 0
    return __shfl_sync(0xFFFFFFFFu, res, 0);
}

template <int DT>
__global__ void __launch_bounds__(SC_WARPS * 32) tile_scores_kernel(
    const void* __restrict__ x, int64_t rows, int64_t cols, int64_t ld, int64_t tiles_w, int64_t ntiles,
    uint32_t fmt_mask, float* __restrict__ scores) {
    __shared__ float xs_all[SC_WARPS][TILE * SCP];
    __shared__ float ys_all[SC_WARPS][TILE * SCP];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t t = (int64_t)blockIdx.x * SC_WARPS + warp;
    if (t >= ntiles) return;
    float* xs = xs_all[warp];
    float* ys = ys_all[warp];
    const int64_t tr = t / tiles_w, tc = t - tr * tiles_w;
    const int64_t row0 = tr * TILE, colb = tc * TILE;
    const int r_end = (int)min((int64_t)TILE, rows - row0);
    const int c_end = (int)min((int64_t)TILE, cols - colb);
    uint32_t nonfinite = 0u;    // an element with exponent field 255 (inf / nan)
    for (int r = 0; r < TILE; ++r) {
        float v = 0.f;
        if (r < r_end && lane < c_end) {
            if (DT == QA_DT_BF16)
                v = __uint_as_float((uint32_t)reinterpret_cast<const uint16_t*>(x)[(row0 + r) * ld + colb + lane] << 16);
            else
                v = reinterpret_cast<const float*>(x)[(row0 + r) * ld + colb + lane];
        }
        if (DT == QA_DT_BF16) nonfinite |= (~__float_as_uint(v) & 0x7F800000u) == 0u;
        xs[r * SCP + lane] = v;
    }
    __syncwarp();
    // a - mean(a), and ||a - mean||^2 chain sums (shared by all formats)
    const float mean_a = __fdiv_rn(pairwise1024([&](int r, int c) { return xs[r * SCP + c]; }, lane), 1024.f);
    float am[TILE];
    float eaa = 0.f, oaa = 0.f;
#pragma unroll
    for (int r = 0; r < TILE; r += 2) {
        am[r] = __fsub_rn(xs[r * SCP + lane], mean_a);
        am[r + 1] = __fsub_rn(xs[(r + 1) * SCP + lane], mean_a);
        eaa = __fmaf_rn(am[r], am[r], eaa);
        oaa = __fmaf_rn(am[r + 1], am[r + 1], oaa);
    }
    const float daa = sdot_fold(eaa, oaa, lane);
    const float na = __fsqrt_rn(daa);

    for (int f = 0; f < QA_NFMT; ++f) {
        if (!((fmt_mask >> f) & 1u)) continue;
        if (DT == QA_DT_BF16 && f == 0) {
            // bf16 of a bf16-exact tile is the tile itself: b == a, so every intermediate of pearson_corr repeats a's
            // (dot(a-m, b-m) = ||a-m||^2, nb = na) and |a - b| is 0, except at an inf or nan element, where it is nan
            // (inf - inf): then mae and atol are nan (np.max propagates it), else 0.  A tile of finite values near FLT_MAX
            // overflows mean_a and daa but still has mae = atol = 0, so the elements decide.  metrics.py:14-15 for a zero
            // denominator
            const float denom = __fmul_rn(na, na);
            const float d = __any_sync(0xFFFFFFFFu, nonfinite) ? __uint_as_float(0x7FFFFFFFu) : 0.f;
            if (lane == 0) {
                scores[(QA_METRIC_PCC * QA_NFMT + f) * ntiles + t] = denom == 0.f ? 1.f : __fdiv_rn(daa, denom);
                scores[(QA_METRIC_MAE * QA_NFMT + f) * ntiles + t] = d;
                scores[(QA_METRIC_ATOL * QA_NFMT + f) * ntiles + t] = d;
            }
            continue;
        }
        __syncwarp();
        for (int g = lane; g < 64; g += 32) {
            const int r = g >> 1, c0 = (g & 1) * GROUP;
            uint32_t u[GROUP];
#pragma unroll
            for (int i = 0; i < GROUP; ++i) u[i] = __float_as_uint(xs[r * SCP + c0 + i]);
            const uint32_t E = group_max_exp(u);
            if (DT == QA_DT_BF16 && f >= 1 && E >= 24u && E != 255u) {
                // bf16-exact values: magic-number rounding in group units (same arithmetic as recon_fast_kernel)
                const float inv = __uint_as_float((261u - E) << 23), back = __uint_as_float((E - 7u) << 23);
                const float M = f == 1 ? 25165824.f : f == 2 ? 402653184.f : 1610612736.f;
                const float L = f == 1 ? 254.f : f == 2 ? 224.f : 128.f;
#pragma unroll
                for (int i = 0; i < GROUP; ++i) {
                    float y = __fadd_rn(__fadd_rn(__fmul_rn(__uint_as_float(u[i]), inv), M), -M);
                    asm("min.xorsign.abs.f32 %0, %1, %2;" : "=f"(y) : "f"(y), "f"(L));
                    ys[r * SCP + c0 + i] = __fmul_rn(y, back);
                }
            } else {
#pragma unroll
                for (int i = 0; i < GROUP; ++i) ys[r * SCP + c0 + i] = __uint_as_float(recon_bits(f, u[i], E));
            }
        }
        __syncwarp();
        const float mean_b = __fdiv_rn(pairwise1024([&](int r, int c) { return ys[r * SCP + c]; }, lane), 1024.f);
        float ebb = 0.f, obb = 0.f, eab = 0.f, oab = 0.f;
        uint32_t mxb = 0u;      // max |x - y| as a bit pattern: non-negative floats order like unsigned ints, and a NaN
                                // (np.max propagates it, tile_utils.py:55-56) orders above +inf
#pragma unroll
        for (int r = 0; r < TILE; r += 2) {
            const float b0 = __fsub_rn(ys[r * SCP + lane], mean_b);
            const float b1 = __fsub_rn(ys[(r + 1) * SCP + lane], mean_b);
            ebb = __fmaf_rn(b0, b0, ebb);
            obb = __fmaf_rn(b1, b1, obb);
            eab = __fmaf_rn(am[r], b0, eab);
            oab = __fmaf_rn(am[r + 1], b1, oab);
            mxb = max(mxb, __float_as_uint(fabsf(__fsub_rn(xs[r * SCP + lane], ys[r * SCP + lane]))));
            mxb = max(mxb, __float_as_uint(fabsf(__fsub_rn(xs[(r + 1) * SCP + lane], ys[(r + 1) * SCP + lane]))));
        }
        const float nb = __fsqrt_rn(sdot_fold(ebb, obb, lane));
        const float dab = sdot_fold(eab, oab, lane);
#pragma unroll
        for (int o = 16; o; o >>= 1) mxb = max(mxb, __shfl_xor_sync(0xFFFFFFFFu, mxb, o));
        const float mx = __uint_as_float(mxb);
        const float denom = __fmul_rn(na, nb);
        float pcc;
        if (denom == 0.f) pcc = (mx == 0.f) ? 1.f : 0.f;      // metrics.py:14-15
        else pcc = __fdiv_rn(dab, denom);
        const float mae = __fdiv_rn(
            pairwise1024([&](int r, int c) { return fabsf(__fsub_rn(xs[r * SCP + c], ys[r * SCP + c])); }, lane), 1024.f);
        if (lane == 0) {
            scores[(QA_METRIC_PCC * QA_NFMT + f) * ntiles + t] = pcc;
            scores[(QA_METRIC_MAE * QA_NFMT + f) * ntiles + t] = mae;
            scores[(QA_METRIC_ATOL * QA_NFMT + f) * ntiles + t] = mx;
        }
    }
}

// tile_metrics(ref_tiles, q_tiles, metric) for ARBITRARY tile stacks (tile_utils.py:46-57): both operands are given,
// float32 [ntiles][32][32]; same summation orders as above.  scores: float32 [3][ntiles] (pcc, mae, atol).
__global__ void __launch_bounds__(SC_WARPS * 32) tile_scores_pair_kernel(const float* __restrict__ ref, const float* __restrict__ q,
                                                                         int64_t ntiles, float* __restrict__ scores) {
    __shared__ float xs_all[SC_WARPS][TILE * SCP];
    __shared__ float ys_all[SC_WARPS][TILE * SCP];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t t = (int64_t)blockIdx.x * SC_WARPS + warp;
    if (t >= ntiles) return;
    float* xs = xs_all[warp];
    float* ys = ys_all[warp];
    for (int r = 0; r < TILE; ++r) {
        xs[r * SCP + lane] = ref[t * 1024 + r * TILE + lane];
        ys[r * SCP + lane] = q[t * 1024 + r * TILE + lane];
    }
    __syncwarp();
    const float mean_a = __fdiv_rn(pairwise1024([&](int r, int c) { return xs[r * SCP + c]; }, lane), 1024.f);
    const float mean_b = __fdiv_rn(pairwise1024([&](int r, int c) { return ys[r * SCP + c]; }, lane), 1024.f);
    float eaa = 0.f, oaa = 0.f, ebb = 0.f, obb = 0.f, eab = 0.f, oab = 0.f;
    uint32_t mxb = 0u;
#pragma unroll
    for (int r = 0; r < TILE; r += 2) {
        const float a0 = __fsub_rn(xs[r * SCP + lane], mean_a), a1 = __fsub_rn(xs[(r + 1) * SCP + lane], mean_a);
        const float b0 = __fsub_rn(ys[r * SCP + lane], mean_b), b1 = __fsub_rn(ys[(r + 1) * SCP + lane], mean_b);
        eaa = __fmaf_rn(a0, a0, eaa); oaa = __fmaf_rn(a1, a1, oaa);
        ebb = __fmaf_rn(b0, b0, ebb); obb = __fmaf_rn(b1, b1, obb);
        eab = __fmaf_rn(a0, b0, eab); oab = __fmaf_rn(a1, b1, oab);
        mxb = max(mxb, __float_as_uint(fabsf(__fsub_rn(xs[r * SCP + lane], ys[r * SCP + lane]))));
        mxb = max(mxb, __float_as_uint(fabsf(__fsub_rn(xs[(r + 1) * SCP + lane], ys[(r + 1) * SCP + lane]))));
    }
    const float na = __fsqrt_rn(sdot_fold(eaa, oaa, lane)), nb = __fsqrt_rn(sdot_fold(ebb, obb, lane));
    const float dab = sdot_fold(eab, oab, lane);
#pragma unroll
    for (int o = 16; o; o >>= 1) mxb = max(mxb, __shfl_xor_sync(0xFFFFFFFFu, mxb, o));
    const float mx = __uint_as_float(mxb);
    const float denom = __fmul_rn(na, nb);
    float pcc;
    if (denom == 0.f) pcc = (mx == 0.f) ? 1.f : 0.f;
    else pcc = __fdiv_rn(dab, denom);
    const float mae = __fdiv_rn(
        pairwise1024([&](int r, int c) { return fabsf(__fsub_rn(xs[r * SCP + c], ys[r * SCP + c])); }, lane), 1024.f);
    if (lane == 0) {
        scores[QA_METRIC_PCC * ntiles + t] = pcc;
        scores[QA_METRIC_MAE * ntiles + t] = mae;
        scores[QA_METRIC_ATOL * ntiles + t] = mx;
    }
}

}  // namespace qa

using namespace qa;

extern "C" int qa_tile_scores_f32(const void* x, int x_dtype, int64_t rows, int64_t cols, int64_t ld,
                                  uint32_t fmt_mask, float* scores, qa_stream_t stream) {
    if (rows < 0 || cols < 0 || ld < cols || !scores) { set_error("qa_tile_scores_f32: bad args"); return 1; }
    if (rows == 0 || cols == 0) return 0;
    const int64_t tiles_w = cdiv(cols, TILE), ntiles = cdiv(rows, TILE) * tiles_w;
    const int64_t grid = cdiv(ntiles, SC_WARPS);
    cudaStream_t s = (cudaStream_t)stream;
    if (x_dtype == QA_DT_BF16)
        tile_scores_kernel<QA_DT_BF16><<<(unsigned)grid, SC_WARPS * 32, 0, s>>>(x, rows, cols, ld, tiles_w, ntiles, fmt_mask & 0xFu, scores);
    else if (x_dtype == QA_DT_F32)
        tile_scores_kernel<QA_DT_F32><<<(unsigned)grid, SC_WARPS * 32, 0, s>>>(x, rows, cols, ld, tiles_w, ntiles, fmt_mask & 0xFu, scores);
    else { set_error("qa_tile_scores_f32: bad dtype"); return 1; }
    return check_launch("qa_tile_scores_f32");
}

extern "C" int qa_tile_scores_pair_f32(const float* ref_tiles, const float* q_tiles, int64_t ntiles, float* scores, qa_stream_t stream) {
    if (ntiles < 0 || !scores || (ntiles && (!ref_tiles || !q_tiles))) { set_error("qa_tile_scores_pair_f32: bad args"); return 1; }
    if (ntiles == 0) return 0;
    tile_scores_pair_kernel<<<(unsigned)cdiv(ntiles, SC_WARPS), SC_WARPS * 32, 0, (cudaStream_t)stream>>>(ref_tiles, q_tiles, ntiles, scores);
    return check_launch("qa_tile_scores_pair_f32");
}
