// Fused quantize + per-tile statistics.
//
// FAST kernel (bf16 input).  A lane owns one 16-element shared-exponent group per row (one
// 256-bit load) and walks the 32 rows of a tile stripe; lanes (2j, 2j+1) together cover tile j of
// the warp's 512-column chunk.  All per-element arithmetic runs in "group units": the group is
// scaled by the exact power of two 2^(134-E) so that every value is a small dyadic number,
//   X = x * 2^(134-E)               |X| <= 255
//   y_f = clamp(rne(X, step_f))     via the (X + 1.5*2^23*step) - 1.5*2^23*step trick, exact
//   r_f = X - y_f                   exact
// and the in-group float32 partial sums  sum y, sum y^2, sum r*y, sum |r|, sum r8, sum r8^2  are
// exact (bounded integers / short dyadics; see DESIGN.md for the bit budget).  Once per group the
// partials are widened to float64 and scaled by 2^(E-134) or its square, so the per-tile float64
// sums are exact whenever they are representable - which is also when NumPy's pairwise float64
// sums in the reference are exact, making the two bit-identical in that (normal) case.
//   sum x y = (sum y^2 + sum r y) * s^2      sum |x-y| = sum |x| - (sum (|X| - |r|)) * s
// sum x, sum x^2 and sum |x| involve elements arbitrarily far below the group maximum, so they
// are accumulated per element in float64 (B200 runs DFMA at 64/clk/SM on its own pipe).
//
// STRICT kernel (bf16 or fp32 input).  One warp per tile; float32 products and float64 sums in
// NumPy's pairwise order over the flattened valid view(s) of the tile, i.e. the same roundings
// as np.sum(..., dtype=np.float64) in mixed_tile_greedy.py:147-174.
#include "qa_common.cuh"

namespace qa {

// ------------------------------------------------------------------------------------------
// FAST
// ------------------------------------------------------------------------------------------
struct TileAcc {
    double sx, sx2;
    double sy[3], sy2[3], sxy[3], sab[3];
    float amax[3];
};

__device__ __forceinline__ void acc_zero(TileAcc& a) {
    a.sx = a.sx2 = 0.0;
#pragma unroll
    for (int f = 0; f < 3; ++f) { a.sy[f] = a.sy2[f] = a.sxy[f] = a.sab[f] = 0.0; a.amax[f] = 0.f; }
}

// Generic (any exponent, inf/nan, tiny E) fallback: integer quantizer + direct f64 accumulation.
__device__ __noinline__ void group_slow(const uint32_t (&w)[8], uint32_t E, TileAcc& a) {
#pragma unroll 1
    for (int i = 0; i < GROUP; ++i) {
        const uint32_t u = (i & 1) ? (w[i >> 1] & 0xFFFF0000u) : (w[i >> 1] << 16);
        const float x = __uint_as_float(u);
        a.sx += (double)x;
        a.sx2 += (double)__fmul_rn(x, x);
#pragma unroll
        for (int f = 0; f < 3; ++f) {
            const uint32_t yb = f == 0 ? bfp_recon_bits<7>(u, E) : f == 1 ? bfp_recon_bits<3>(u, E) : bfp_recon_bits<1>(u, E);
            const float y = __uint_as_float(yb);
            const float r = fabsf(__fsub_rn(x, y));
            a.sy[f] += (double)y;
            a.sy2[f] += (double)__fmul_rn(y, y);
            a.sxy[f] += (double)__fmul_rn(x, y) - (double)__fmul_rn(y, y);   // sxy holds sum (x-y)*y until the tile end
            a.sab[f] += (double)r;
            a.amax[f] = fmaxf(a.amax[f], r);
        }
    }
    // 191 <= E < 255: the group's largest |x| is at least 2^64 and its reconstruction in every format has the same sign and
    // at least the magnitude 2^(E-127), so that float32 x*y is +inf (as are x*x and y*y).  Every other x*y is >= 0, so the
    // reference's sum x*y is +inf; the difference above would be inf - inf.
    if (E - 191u < 64u) {
#pragma unroll
        for (int f = 0; f < 3; ++f) a.sxy[f] = __longlong_as_double(0x7FF0000000000000LL);
    }
}

template <int F>
struct Fmt;
template <> struct Fmt<0> { static constexpr float M = 25165824.f, L = 254.f; };     // bfp8: step 2
template <> struct Fmt<1> { static constexpr float M = 402653184.f, L = 224.f; };    // bfp4: step 32
template <> struct Fmt<2> { static constexpr float M = 1610612736.f, L = 128.f; };   // bfp2: step 128

// sm_100 packed-float2 arithmetic (FADD2 / FMUL2 / FFMA2: two fp32 lanes per issue slot)
#ifdef QA_STATS_SCALAR      // experiment (profiles/r2_stats_variants.txt): scalar FADD / FFMA instead of the packed forms
__device__ __forceinline__ float2 add2(float2 a, float2 b) { return make_float2(__fadd_rn(a.x, b.x), __fadd_rn(a.y, b.y)); }
__device__ __forceinline__ float2 sub2(float2 a, float2 b) { return make_float2(__fsub_rn(a.x, b.x), __fsub_rn(a.y, b.y)); }
__device__ __forceinline__ float2 mul2(float2 a, float2 b) { return make_float2(__fmul_rn(a.x, b.x), __fmul_rn(a.y, b.y)); }
__device__ __forceinline__ float2 fma2(float2 a, float2 b, float2 c) { return make_float2(__fmaf_rn(a.x, b.x, c.x), __fmaf_rn(a.y, b.y, c.y)); }
#else
__device__ __forceinline__ float2 add2(float2 a, float2 b) { return __fadd2_rn(a, b); }
__device__ __forceinline__ float2 sub2(float2 a, float2 b) { return __fadd2_rn(a, make_float2(-b.x, -b.y)); }
__device__ __forceinline__ float2 mul2(float2 a, float2 b) { return __fmul2_rn(a, b); }
__device__ __forceinline__ float2 fma2(float2 a, float2 b, float2 c) { return __ffma2_rn(a, b, c); }
#endif
// clamp(y, -L, L) in one instruction: min(|y|, L) with the sign of y (FMNMX.XORSIGN)
__device__ __forceinline__ float clamp_sym(float y, float L) {
    float r;
    asm("min.xorsign.abs.f32 %0, %1, %2;" : "=f"(r) : "f"(y), "f"(L));
    return r;
}
__device__ __forceinline__ float max3abs(float m, float a, float b) {
    float r;
    asm("max.NaN.abs.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(m), "f"(a), "f"(b));   // a NaN must surface: its exponent is 255
    return r;
}

struct GroupAcc {   // in-group float32 partials, two lanes (even / odd element) each
    float2 sy, sy2, sry, sab;
    float mx;
    double dab;         // QA_SAB_FP64: sum |r| accumulated on the FP64 pipe (exact)
};
#ifndef QA_SAB_FP64
#define QA_SAB_FP64 0
#endif

template <int F, bool EXACT_ABS>
__device__ __forceinline__ void fmt_step(const float2 X, const float2 aX, GroupAcc& g) {
    const float2 Mv = make_float2(Fmt<F>::M, Fmt<F>::M);
#ifdef QA_STATS_SCALAR_ROUND      // experiment: the rounding as scalar FADDs (they overlap the ALU clamps, the packed forms do not)
    float2 y = make_float2(__fadd_rn(__fadd_rn(X.x, Fmt<F>::M), -Fmt<F>::M), __fadd_rn(__fadd_rn(X.y, Fmt<F>::M), -Fmt<F>::M));
    (void)Mv;
#else
    float2 y = sub2(add2(X, Mv), Mv);                  // round to the format's step, ties to even
#endif
    y.x = clamp_sym(y.x, Fmt<F>::L);                   // mantissa clamp (no exponent bump)
    y.y = clamp_sym(y.y, Fmt<F>::L);
    const float2 r = sub2(X, y);
    g.sy = add2(g.sy, y);
    g.sy2 = fma2(y, y, g.sy2);
    g.sry = fma2(r, y, g.sry);
    if (EXACT_ABS) {
        // |X| - |r|: 0 for elements every format flushes, a short dyadic otherwise (exact in fp32)
        g.sab.x += aX.x - fabsf(r.x);
        g.sab.y += aX.y - fabsf(r.y);
    } else if (QA_SAB_FP64) {
        g.dab += fabs((double)r.x);
        g.dab += fabs((double)r.y);
    } else {
        g.sab.x += fabsf(r.x);
        g.sab.y += fabsf(r.y);
    }
    g.mx = max3abs(g.mx, r.x, r.y);
}

template <bool EXACT_ABS>
__device__ __forceinline__ void group_fast(const uint32_t (&w)[8], TileAcc& a) {
    // shared exponent = exponent of max |x| (one 3-input max with |.| modifiers per word)
    float2 xv[8];
    float mabs = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        xv[i] = make_float2(__uint_as_float(w[i] << 16), __uint_as_float(w[i] & 0xFFFF0000u));
        mabs = max3abs(mabs, xv[i].x, xv[i].y);
    }
    const uint32_t E = __float_as_uint(mabs) >> 23;
    // The generic path forms float32 products like the reference (x*x, y*y, x*y as float32 arrays); it takes
    //   E < 76: zeros and denormals only (E == 0: each counts in sum x and, unquantized, in sum |x-y| and max |x-y|), or
    //     squares that round or flush in float32's denormal range by more than the 1e-13 the table promises.  Below
    //     here an element's fast square is exact where the reference's is rounded to a multiple of 2^-149: off by at
    //     most 2^-150, 2^-146 per group, against a group sum x^2 of at least 2^(2E-254): <= 2^(108-2E) = 2^-44 at E = 76;
    //   E >= 191: |x| >= 2^64, where x*x, y*y and x*y overflow to inf in float32 (group_slow records sum x*y = +inf);
    //   E == 255: inf / nan.
    if (E < 76u || E >= 191u) {
        // rare: keep the caller's accumulators in registers by handing the slow path its own copy
        TileAcc t;
        acc_zero(t);
        uint32_t wc[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) wc[i] = w[i];
        group_slow(wc, E, t);
        a.sx += t.sx; a.sx2 += t.sx2;
#pragma unroll
        for (int f = 0; f < 3; ++f) {
            a.sy[f] += t.sy[f]; a.sy2[f] += t.sy2[f]; a.sxy[f] += t.sxy[f]; a.sab[f] += t.sab[f];
            a.amax[f] = fmaxf(a.amax[f], t.amax[f]);
        }
        return;
    }

    const float inv = __uint_as_float((261u - E) << 23);  // 2^(134-E)
    const float2 inv2 = make_float2(inv, inv);
    GroupAcc g[3];
#pragma unroll
    for (int f = 0; f < 3; ++f) {
        g[f].sy = g[f].sy2 = g[f].sry = g[f].sab = make_float2(0.f, 0.f);
        g[f].mx = 0.f;
        g[f].dab = 0.0;
    }
    double gx = 0.0, gx2 = 0.0, gax = 0.0;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const float2 x = xv[i];
        // sum x, sum x^2 (and sum |x|): float64 per element - exact whatever the exponent spread
        const double x0 = (double)x.x, x1 = (double)x.y;
        gx += x0;
        gx += x1;
        gx2 = fma(x0, x0, gx2);
        gx2 = fma(x1, x1, gx2);
        if (EXACT_ABS) { gax += fabs(x0); gax += fabs(x1); }
        const float2 X = mul2(x, inv2);
        const float2 aX = make_float2(fabsf(X.x), fabsf(X.y));
        fmt_step<0, EXACT_ABS>(X, aX, g[0]);
        fmt_step<1, EXACT_ABS>(X, aX, g[1]);
        fmt_step<2, EXACT_ABS>(X, aX, g[2]);
    }
    const double s1 = __hiloint2double((int)((E + 889u) << 20), 0);        // 2^(E-134)
    const double s2 = __hiloint2double((int)((2u * E + 755u) << 20), 0);   // 2^(2E-268)
    const float s1f = __uint_as_float((E - 7u) << 23);
    a.sx += gx;
    a.sx2 += gx2;
#pragma unroll
    for (int f = 0; f < 3; ++f) {
        a.sy[f] = fma((double)(g[f].sy.x + g[f].sy.y), s1, a.sy[f]);
        a.sy2[f] = fma((double)(g[f].sy2.x + g[f].sy2.y), s2, a.sy2[f]);
        a.sxy[f] = fma((double)(g[f].sry.x + g[f].sry.y), s2, a.sxy[f]);   // holds sum r*y; + sum y^2 at tile end
        if (EXACT_ABS) a.sab[f] += fma(-(double)(g[f].sab.x + g[f].sab.y), s1, gax);
        else if (QA_SAB_FP64) a.sab[f] = fma(g[f].dab, s1, a.sab[f]);
        else a.sab[f] = fma((double)(g[f].sab.x + g[f].sab.y), s1, a.sab[f]);
        a.amax[f] = fmaxf(a.amax[f], g[f].mx * s1f);
    }
}

__device__ __forceinline__ double shfl_xor_d(double v, int m) {
    return __hiloint2double(__shfl_xor_sync(0xFFFFFFFFu, __double2hiint(v), m),
                            __shfl_xor_sync(0xFFFFFFFFu, __double2loint(v), m));
}

template <bool VEC>
__device__ __forceinline__ void load_row_group(const uint16_t* __restrict__ x, int64_t row, int64_t col0,
                                               int64_t cols, int64_t ld, uint32_t (&w)[8]) {
    if (VEC) {
        ldg256(x + row * ld + col0, w);
    } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int64_t c = col0 + 2 * i;
            const uint32_t lo = c < cols ? x[row * ld + c] : 0u;
            const uint32_t hi = c + 1 < cols ? x[row * ld + c + 1] : 0u;
            w[i] = lo | (hi << 16);
        }
    }
}

constexpr int FAST_WARPS = 4;               // warps per CTA; one CTA = one 32-row x 512-column item
constexpr int FAST_RPW = TILE / FAST_WARPS; // rows per warp
#ifndef FAST_UNROLL_N
#define FAST_UNROLL_N 4
#endif
constexpr int FAST_UNROLL = FAST_UNROLL_N;
#ifndef FAST_MIN_BLOCKS
#define FAST_MIN_BLOCKS 4
#endif

// One CTA per (tile row, 512-column chunk); warp w walks rows 8w..8w+7 of the stripe, the four
// partial accumulator sets are summed in warp order through shared memory (fixed order => the
// result is deterministic, and exact whenever the float64 sums are representable).  Small items
// keep the last wave short: o_proj is 7168 CTAs = 12 waves of 592 instead of 3.03 waves of big ones.
template <bool VEC, bool EXACT_ABS>
__device__ __forceinline__ void stats_fast_item(double (&part)[FAST_WARPS - 1][14][32], float (&partmx)[FAST_WARPS - 1][3][32],
                                                const uint16_t* __restrict__ x, int64_t rows, int64_t cols, int64_t ld, int64_t tiles_w,
                                                int64_t chunks, int64_t item, int64_t ntiles, uint32_t fmt_mask,
                                                double* __restrict__ table) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int64_t tr = item / chunks;
    const int64_t ck = item - tr * chunks;
    const int64_t col0 = ck * 512 + (int64_t)lane * GROUP;
    const int64_t row0 = tr * TILE + w * FAST_RPW;
    const int nrows = (int)max((int64_t)0, min((int64_t)FAST_RPW, rows - row0));
    TileAcc a;
    acc_zero(a);
    if (col0 < cols) {
#ifdef QA_STATS_PREFETCH          // experiment: rows in batches of QA_STATS_PREFETCH, the next batch requested before this one is processed
        constexpr int PB = QA_STATS_PREFETCH, NB = FAST_RPW / PB;
        uint32_t buf[2][PB][8];
        auto load_batch = [&](int b, uint32_t (&dst)[PB][8]) {
#pragma unroll
            for (int k = 0; k < PB; ++k) {
                if (b * PB + k < nrows) load_row_group<VEC>(x, row0 + b * PB + k, col0, cols, ld, dst[k]);
                else {
#pragma unroll
                    for (int i = 0; i < 8; ++i) dst[k][i] = 0u;
                }
            }
        };
        load_batch(0, buf[0]);
#pragma unroll
        for (int b = 0; b < NB; ++b) {
            if (b + 1 < NB) load_batch(b + 1, buf[(b + 1) & 1]);
#pragma unroll
            for (int k = 0; k < PB; ++k) group_fast<EXACT_ABS>(buf[b & 1][k], a);
        }
        int r = nrows;
        uint32_t cur[1][8];
#else
        uint32_t cur[FAST_UNROLL][8];
        int r = 0;
#endif
        for (; r + FAST_UNROLL <= nrows; r += FAST_UNROLL) {
#pragma unroll
            for (int k = 0; k < FAST_UNROLL; ++k) load_row_group<VEC>(x, row0 + r + k, col0, cols, ld, cur[k]);
#pragma unroll
            for (int k = 0; k < FAST_UNROLL; ++k) group_fast<EXACT_ABS>(cur[k], a);
        }
        for (; r < nrows; ++r) {
            load_row_group<VEC>(x, row0 + r, col0, cols, ld, cur[0]);
            group_fast<EXACT_ABS>(cur[0], a);
        }
    }
#pragma unroll
    for (int f = 0; f < 3; ++f) a.sxy[f] += a.sy2[f];    // sum x*y = sum y^2 + sum (x-y)*y
    if (w > 0) {
        double (*p)[32] = part[w - 1];
        p[0][lane] = a.sx; p[1][lane] = a.sx2;
#pragma unroll
        for (int f = 0; f < 3; ++f) {
            p[2 + f][lane] = a.sy[f]; p[5 + f][lane] = a.sy2[f]; p[8 + f][lane] = a.sxy[f]; p[11 + f][lane] = a.sab[f];
            partmx[w - 1][f][lane] = a.amax[f];
        }
    }
    __syncthreads();
    if (w != 0) return;
#pragma unroll
    for (int q = 0; q < FAST_WARPS - 1; ++q) {
        a.sx += part[q][0][lane]; a.sx2 += part[q][1][lane];
#pragma unroll
        for (int f = 0; f < 3; ++f) {
            a.sy[f] += part[q][2 + f][lane]; a.sy2[f] += part[q][5 + f][lane];
            a.sxy[f] += part[q][8 + f][lane]; a.sab[f] += part[q][11 + f][lane];
            a.amax[f] = fmaxf(a.amax[f], partmx[q][f][lane]);
        }
    }
    // lanes 2j and 2j+1 hold the two halves of tile j
    a.sx += shfl_xor_d(a.sx, 1);
    a.sx2 += shfl_xor_d(a.sx2, 1);
#pragma unroll
    for (int f = 0; f < 3; ++f) {
        a.sy[f] += shfl_xor_d(a.sy[f], 1);
        a.sy2[f] += shfl_xor_d(a.sy2[f], 1);
        a.sxy[f] += shfl_xor_d(a.sxy[f], 1);
        a.sab[f] += shfl_xor_d(a.sab[f], 1);
        a.amax[f] = fmaxf(a.amax[f], __shfl_xor_sync(0xFFFFFFFFu, a.amax[f], 1));
    }
    const int64_t tc = ck * 16 + (lane >> 1);
    if ((lane & 1) == 0 && tc < tiles_w) {
        const int64_t t = tr * tiles_w + tc;
        table[QA_STAT_SX * ntiles + t] = a.sx;
        table[QA_STAT_SX2 * ntiles + t] = a.sx2;
        if (fmt_mask & 1u) {  // bf16-exact input: y == x
            table[QA_STAT_FMT(0, 0) * ntiles + t] = a.sx;
            table[QA_STAT_FMT(0, 1) * ntiles + t] = a.sx2;
            table[QA_STAT_FMT(0, 2) * ntiles + t] = a.sx2;
            table[QA_STAT_FMT(0, 3) * ntiles + t] = 0.0;
            table[QA_STAT_FMT(0, 4) * ntiles + t] = 0.0;
        }
#pragma unroll
        for (int f = 0; f < 3; ++f) {
            if (fmt_mask & (2u << f)) {
                table[QA_STAT_FMT(f + 1, 0) * ntiles + t] = a.sy[f];
                table[QA_STAT_FMT(f + 1, 1) * ntiles + t] = a.sy2[f];
                table[QA_STAT_FMT(f + 1, 2) * ntiles + t] = a.sxy[f];
                table[QA_STAT_FMT(f + 1, 3) * ntiles + t] = a.sab[f];
                table[QA_STAT_FMT(f + 1, 4) * ntiles + t] = (double)a.amax[f];
            }
        }
    }
}

template <bool VEC, bool EXACT_ABS>
__global__ void __launch_bounds__(FAST_WARPS * 32, FAST_MIN_BLOCKS) stats_fast_kernel(
    const uint16_t* __restrict__ x, int64_t rows, int64_t cols, int64_t ld, int64_t tiles_w,
    int64_t chunks, int64_t item0, int64_t ntiles, uint32_t fmt_mask, double* __restrict__ table) {
    __shared__ double part[FAST_WARPS - 1][14][32];
    __shared__ float partmx[FAST_WARPS - 1][3][32];
    // item0 > 0: a launch that covers a range of tile rows
    stats_fast_item<VEC, EXACT_ABS>(part, partmx, x, rows, cols, ld, tiles_w, chunks, blockIdx.x + item0, ntiles, fmt_mask, table);
}

// Descriptor-array batch: CTA b finds its tensor by bisection over the item prefix and runs the same item body.
template <bool EXACT_ABS>
__global__ void __launch_bounds__(FAST_WARPS * 32, FAST_MIN_BLOCKS) stats_fast_batch_kernel(const qa_batch_desc* __restrict__ descs, int n,
                                                                                            uint32_t fmt_mask) {
    __shared__ double part[FAST_WARPS - 1][14][32];
    __shared__ float partmx[FAST_WARPS - 1][3][32];
    const int64_t b = blockIdx.x;
    int lo = 0, hi = n - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (__ldg(&descs[mid].item_begin) <= b) lo = mid; else hi = mid - 1;
    }
    const qa_batch_desc d = descs[lo];
    const int64_t tiles_h = cdiv(d.rows, TILE), tiles_w = cdiv(d.cols, TILE), chunks = cdiv(d.cols, 512);
    const uint16_t* x = reinterpret_cast<const uint16_t*>(d.x);
    const bool vec = (d.cols % GROUP == 0) && (d.ld % GROUP == 0) && (reinterpret_cast<uintptr_t>(d.x) % 32 == 0);
    if (vec) stats_fast_item<true, EXACT_ABS>(part, partmx, x, d.rows, d.cols, d.ld, tiles_w, chunks, b - d.item_begin, tiles_h * tiles_w, fmt_mask, d.table);
    else stats_fast_item<false, EXACT_ABS>(part, partmx, x, d.rows, d.cols, d.ld, tiles_w, chunks, b - d.item_begin, tiles_h * tiles_w, fmt_mask, d.table);
}

// ------------------------------------------------------------------------------------------
// FAST, TMA-staged (experiment of round 2, selected with QA_STATS_TMA=1): a persistent CTA walks (tile row, 512-column chunk)
// items; thread 0 streams 16-row x 512-column half-items (16 bulk copies of 1 KB, one mbarrier per stage) into a two-stage
// shared-memory ring, each warp pulls its four rows into registers (LDS.128), frees the stage and runs the same group
// arithmetic.  The row loads leave the warps' scoreboards (12 % of the warp-time of stats_fast_kernel waits on them).
// ------------------------------------------------------------------------------------------
constexpr int TS_ROWS = 16, TS_NST = 2, TS_STAGE = TS_ROWS * 512 * 2;
__device__ __forceinline__ unsigned ts_s32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void ts_wait(unsigned bar, unsigned parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "TS_WAIT:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra TS_DONE;\n\t"
        "bra TS_WAIT;\n\t"
        "TS_DONE:\n\t}" ::"r"(bar), "r"(parity) : "memory");
}

template <bool EXACT_ABS>
__global__ void __launch_bounds__(FAST_WARPS * 32, FAST_MIN_BLOCKS) stats_tma_kernel(
    const uint16_t* __restrict__ x, int64_t ld, int64_t tiles_w, int64_t chunks, int64_t item0, int64_t nitems, int64_t ntiles,
    uint32_t fmt_mask, double* __restrict__ table) {
    __shared__ __align__(128) unsigned char ring[TS_NST][TS_STAGE];
    __shared__ __align__(8) unsigned long long full[TS_NST], empty[TS_NST];
    __shared__ double part[FAST_WARPS - 1][14][32];
    __shared__ float partmx[FAST_WARPS - 1][3][32];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    if (threadIdx.x == 0) {
        for (int s_ = 0; s_ < TS_NST; ++s_) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(ts_s32(&full[s_])) : "memory");
            asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(ts_s32(&empty[s_])), "r"(FAST_WARPS) : "memory");
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    __syncthreads();
    if ((int64_t)blockIdx.x >= nitems) return;
    const int64_t my_items = (nitems - blockIdx.x + gridDim.x - 1) / gridDim.x;
    const int64_t nh = 2 * my_items;                       // half-items of this CTA, in order
    auto issue = [&](int64_t h) {                          // thread 0: stage h % TS_NST <- half-item h
        const int64_t item = item0 + blockIdx.x + (h >> 1) * gridDim.x;
        const int64_t tr = item / chunks, ck = item - tr * chunks;
        const uint16_t* src = x + (tr * TILE + (h & 1) * TS_ROWS) * ld + ck * 512;
        const int s_ = (int)(h % TS_NST);
        const unsigned bar = ts_s32(&full[s_]);
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"((unsigned)TS_STAGE) : "memory");
#pragma unroll 4
        for (int r = 0; r < TS_ROWS; ++r)
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                             ts_s32(&ring[s_][r * 1024])),
                         "l"(src + (int64_t)r * ld), "r"(1024u), "r"(bar)
                         : "memory");
    };
    if (threadIdx.x == 0)
        for (int64_t h = 0; h < nh && h < TS_NST; ++h) issue(h);
    TileAcc a;
    acc_zero(a);
    for (int64_t h = 0; h < nh; ++h) {
        const int s_ = (int)(h % TS_NST);
        const unsigned parity = (unsigned)((h / TS_NST) & 1);
        ts_wait(ts_s32(&full[s_]), parity);
        uint32_t cur[TS_ROWS / FAST_WARPS][8];
        const unsigned char* base = &ring[s_][(w * (TS_ROWS / FAST_WARPS)) * 1024 + lane * 32];
#pragma unroll
        for (int k = 0; k < TS_ROWS / FAST_WARPS; ++k) {
            const uint4 lo = *reinterpret_cast<const uint4*>(base + k * 1024), hi = *reinterpret_cast<const uint4*>(base + k * 1024 + 16);
            cur[k][0] = lo.x; cur[k][1] = lo.y; cur[k][2] = lo.z; cur[k][3] = lo.w;
            cur[k][4] = hi.x; cur[k][5] = hi.y; cur[k][6] = hi.z; cur[k][7] = hi.w;
        }
        __syncwarp();
        if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(ts_s32(&empty[s_])) : "memory");
        if (threadIdx.x == 0 && h + TS_NST < nh) {         // every warp has its rows in registers: refill the stage
            ts_wait(ts_s32(&empty[s_]), parity);
            issue(h + TS_NST);
        }
#pragma unroll
        for (int k = 0; k < TS_ROWS / FAST_WARPS; ++k) group_fast<EXACT_ABS>(cur[k], a);
        if (!(h & 1)) continue;
        // end of an item: the four warps' partial sets are summed in warp order (as in stats_fast_kernel)
        const int64_t item = item0 + blockIdx.x + (h >> 1) * gridDim.x;
        const int64_t tr = item / chunks, ck = item - tr * chunks;
#pragma unroll
        for (int f = 0; f < 3; ++f) a.sxy[f] += a.sy2[f];
        if (w > 0) {
            double (*p)[32] = part[w - 1];
            p[0][lane] = a.sx; p[1][lane] = a.sx2;
#pragma unroll
            for (int f = 0; f < 3; ++f) {
                p[2 + f][lane] = a.sy[f]; p[5 + f][lane] = a.sy2[f]; p[8 + f][lane] = a.sxy[f]; p[11 + f][lane] = a.sab[f];
                partmx[w - 1][f][lane] = a.amax[f];
            }
        }
        __syncthreads();
        if (w == 0) {
#pragma unroll
            for (int q = 0; q < FAST_WARPS - 1; ++q) {
                a.sx += part[q][0][lane]; a.sx2 += part[q][1][lane];
#pragma unroll
                for (int f = 0; f < 3; ++f) {
                    a.sy[f] += part[q][2 + f][lane]; a.sy2[f] += part[q][5 + f][lane];
                    a.sxy[f] += part[q][8 + f][lane]; a.sab[f] += part[q][11 + f][lane];
                    a.amax[f] = fmaxf(a.amax[f], partmx[q][f][lane]);
                }
            }
            a.sx += shfl_xor_d(a.sx, 1);
            a.sx2 += shfl_xor_d(a.sx2, 1);
#pragma unroll
            for (int f = 0; f < 3; ++f) {
                a.sy[f] += shfl_xor_d(a.sy[f], 1); a.sy2[f] += shfl_xor_d(a.sy2[f], 1);
                a.sxy[f] += shfl_xor_d(a.sxy[f], 1); a.sab[f] += shfl_xor_d(a.sab[f], 1);
                a.amax[f] = fmaxf(a.amax[f], __shfl_xor_sync(0xFFFFFFFFu, a.amax[f], 1));
            }
            const int64_t tc = ck * 16 + (lane >> 1);
            if ((lane & 1) == 0 && tc < tiles_w) {
                const int64_t t = tr * tiles_w + tc;
                table[QA_STAT_SX * ntiles + t] = a.sx;
                table[QA_STAT_SX2 * ntiles + t] = a.sx2;
                if (fmt_mask & 1u) {
                    table[QA_STAT_FMT(0, 0) * ntiles + t] = a.sx;
                    table[QA_STAT_FMT(0, 1) * ntiles + t] = a.sx2;
                    table[QA_STAT_FMT(0, 2) * ntiles + t] = a.sx2;
                    table[QA_STAT_FMT(0, 3) * ntiles + t] = 0.0;
                    table[QA_STAT_FMT(0, 4) * ntiles + t] = 0.0;
                }
#pragma unroll
                for (int f = 0; f < 3; ++f) {
                    if (fmt_mask & (2u << f)) {
                        table[QA_STAT_FMT(f + 1, 0) * ntiles + t] = a.sy[f];
                        table[QA_STAT_FMT(f + 1, 1) * ntiles + t] = a.sy2[f];
                        table[QA_STAT_FMT(f + 1, 2) * ntiles + t] = a.sxy[f];
                        table[QA_STAT_FMT(f + 1, 3) * ntiles + t] = a.sab[f];
                        table[QA_STAT_FMT(f + 1, 4) * ntiles + t] = (double)a.amax[f];
                    }
                }
            }
        }
        __syncthreads();                                   // part[] is free again
        acc_zero(a);
    }
}

// ------------------------------------------------------------------------------------------
// STRICT
// ------------------------------------------------------------------------------------------
constexpr int SP = 33;  // padded smem row pitch

struct View {
    int r0, nr, nc;  // rows [r0, r0+nr), cols [0, nc)
};

// value of statistic `kind` at flattened index i of a view (float32 arithmetic as NumPy does it)
__device__ __forceinline__ double strict_term(const float* xs, const float* ys, const View& v, int i, int kind) {
    const int r = v.r0 + i / v.nc, c = i % v.nc;
    const float x = xs[r * SP + c];
    if (kind == 0) return (double)x;
    if (kind == 1) return (double)__fmul_rn(x, x);
    const float y = ys[r * SP + c];
    if (kind == 2) return (double)y;
    if (kind == 3) return (double)__fmul_rn(y, y);
    if (kind == 4) return (double)__fmul_rn(x, y);
    return (double)fabsf(__fsub_rn(x, y));
}

// NumPy pairwise leaf (n <= 128) starting at flattened index lo
__device__ double strict_leaf(const float* xs, const float* ys, const View& v, int lo, int n, int kind) {
    if (n < 8) {
        double res = 0.0;
        for (int i = 0; i < n; ++i) res = __dadd_rn(res, strict_term(xs, ys, v, lo + i, kind));
        return res;
    }
    double r[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) r[k] = strict_term(xs, ys, v, lo + k, kind);
    int i = 8;
    for (; i < n - (n % 8); i += 8) {
#pragma unroll
        for (int k = 0; k < 8; ++k) r[k] = __dadd_rn(r[k], strict_term(xs, ys, v, lo + i + k, kind));
    }
    double res = __dadd_rn(__dadd_rn(__dadd_rn(r[0], r[1]), __dadd_rn(r[2], r[3])),
                           __dadd_rn(__dadd_rn(r[4], r[5]), __dadd_rn(r[6], r[7])));
    for (; i < n; ++i) res = __dadd_rn(res, strict_term(xs, ys, v, lo + i, kind));
    return res;
}

// enumerate the leaves of NumPy's recursion over n elements (at most 16 for n <= 1024)
__device__ int strict_leaves(int n, int* lo, int* len) {
    int cnt = 0, sp = 0;
    int st_lo[16], st_n[16];
    st_lo[0] = 0; st_n[0] = n; sp = 1;
    while (sp) {
        --sp;
        const int l = st_lo[sp], m = st_n[sp];
        if (m <= 128) { lo[cnt] = l; len[cnt] = m; ++cnt; continue; }
        int n2 = m / 2; n2 -= n2 % 8;
        st_lo[sp] = l + n2; st_n[sp] = m - n2; ++sp;   // right pushed first, so left pops first
        st_lo[sp] = l; st_n[sp] = n2; ++sp;
    }
    return cnt;
}

// combine leaf sums with the recursion's tree: sum(n) = sum(left n2) + sum(right)
__device__ double strict_combine(const double* leaf, int& li, int n) {
    if (n <= 128) return leaf[li++];
    int n2 = n / 2; n2 -= n2 % 8;
    const double a = strict_combine(leaf, li, n2);
    const double b = strict_combine(leaf, li, n - n2);
    return __dadd_rn(a, b);
}

constexpr int STRICT_WARPS = 4;

template <int DT>
__global__ void __launch_bounds__(STRICT_WARPS * 32) stats_strict_kernel(
    const void* __restrict__ x, int64_t rows, int64_t cols, int64_t ld, int64_t tiles_w, int64_t ntiles,
    int64_t vec_tail, uint32_t fmt_mask, double* __restrict__ table) {
    __shared__ float xs_all[STRICT_WARPS][TILE * SP];
    __shared__ float ys_all[STRICT_WARPS][TILE * SP];
    __shared__ double leaf_all[STRICT_WARPS][6][16];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t t = (int64_t)blockIdx.x * STRICT_WARPS + warp;
    if (t >= ntiles) return;
    float* xs = xs_all[warp];
    float* ys = ys_all[warp];
    const int64_t tr = t / tiles_w, tc = t - tr * tiles_w;
    const int64_t row0 = tr * TILE, colb = tc * TILE;
    const int r_end = (int)min((int64_t)TILE, rows - row0);
    const int c_end = (int)min((int64_t)TILE, cols - colb);
    // stage the zero-padded tile
    for (int r = 0; r < TILE; ++r) {
        float v = 0.f;
        if (r < r_end && lane < c_end) {
            if (DT == QA_DT_BF16)
                v = __uint_as_float((uint32_t)reinterpret_cast<const uint16_t*>(x)[(row0 + r) * ld + colb + lane] << 16);
            else
                v = reinterpret_cast<const float*>(x)[(row0 + r) * ld + colb + lane];
        }
        xs[r * SP + lane] = v;
    }
    __syncwarp();
    // the views the reference sums over (mixed_tile_greedy.py:122-131)
    View views[2];
    int nviews = 1;
    const bool last_tr = (row0 + r_end == rows);
    if (vec_tail > 0 && vec_tail < TILE && last_tr) {
        nviews = 0;
        if (r_end - 1 > 0) views[nviews++] = View{0, r_end - 1, c_end};
        views[nviews++] = View{r_end - 1, 1, (int)vec_tail};
    } else {
        views[0] = View{0, r_end, c_end};
    }

    auto reduce_kinds = [&](int kind_lo, int nkinds, double* out) {
        // out[k] = 0.0 + sum(view0) (+ sum(view1)), each sum in NumPy pairwise order
        for (int k = 0; k < nkinds; ++k) out[k] = 0.0;
        for (int vi = 0; vi < nviews; ++vi) {
            const View v = views[vi];
            const int n = v.nr * v.nc;
            int lo[16], len[16];
            const int nl = strict_leaves(n, lo, len);
            // (kind, leaf) pairs spread over lanes
            for (int job = lane; job < nkinds * nl; job += 32) {
                const int k = job / nl, li = job - k * nl;
                leaf_all[warp][k][li] = strict_leaf(xs, ys, v, lo[li], len[li], kind_lo + k);
            }
            __syncwarp();
            for (int k = 0; k < nkinds; ++k) {
                int li = 0;
                const double s = n > 0 ? strict_combine(leaf_all[warp][k], li, n) : 0.0;
                out[k] = __dadd_rn(out[k], s);
            }
            __syncwarp();
        }
    };

    double res[4];
    reduce_kinds(0, 2, res);
    if (lane == 0) {
        table[QA_STAT_SX * ntiles + t] = res[0];
        table[QA_STAT_SX2 * ntiles + t] = res[1];
    }
    for (int f = 0; f < QA_NFMT; ++f) {
        if (!((fmt_mask >> f) & 1u)) continue;
        // quantize the tile: 64 groups, two per lane
        __syncwarp();
        for (int g = lane; g < 64; g += 32) {
            const int r = g >> 1, c0 = (g & 1) * GROUP;
            uint32_t u[GROUP];
#pragma unroll
            for (int i = 0; i < GROUP; ++i) u[i] = __float_as_uint(xs[r * SP + c0 + i]);
            const uint32_t E = group_max_exp(u);
#pragma unroll
            for (int i = 0; i < GROUP; ++i) ys[r * SP + c0 + i] = __uint_as_float(recon_bits(f, u[i], E));
        }
        __syncwarp();
        reduce_kinds(2, 4, res);
        // max |x - y| over the views (float32, order-free)
        float mx = 0.f;
        for (int vi = 0; vi < nviews; ++vi) {
            const View v = views[vi];
            for (int i = lane; i < v.nr * v.nc; i += 32) {
                const int r = v.r0 + i / v.nc, c = i % v.nc;
                mx = fmaxf(mx, fabsf(__fsub_rn(xs[r * SP + c], ys[r * SP + c])));
            }
        }
#pragma unroll
        for (int o = 16; o; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xFFFFFFFFu, mx, o));
        if (lane == 0) {
            table[QA_STAT_FMT(f, 0) * ntiles + t] = res[0];
            table[QA_STAT_FMT(f, 1) * ntiles + t] = res[1];
            table[QA_STAT_FMT(f, 2) * ntiles + t] = res[2];
            table[QA_STAT_FMT(f, 3) * ntiles + t] = res[3];
            table[QA_STAT_FMT(f, 4) * ntiles + t] = (double)mx;
        }
    }
}

}  // namespace qa

using namespace qa;

static int tile_stats_fast(const void* x, int64_t rows, int64_t cols, int64_t ld, uint32_t fmt_mask, int mode, double* table,
                           int64_t tile_row_begin, int64_t tile_row_end, cudaStream_t s) {
    const int64_t tiles_h = cdiv(rows, TILE), tiles_w = cdiv(cols, TILE), ntiles = tiles_h * tiles_w;
    const int64_t chunks = cdiv(cols, 512);
    const int64_t grid = (tile_row_end - tile_row_begin) * chunks, item0 = tile_row_begin * chunks;
    const bool vec = (cols % GROUP == 0) && (ld % GROUP == 0) && (reinterpret_cast<uintptr_t>(x) % 32 == 0);
    const uint16_t* xp = reinterpret_cast<const uint16_t*>(x);
    const bool exact_abs = (mode == QA_STATS_FAST);
    static const int use_tma = getenv("QA_STATS_TMA") ? atoi(getenv("QA_STATS_TMA")) : 0;
    if (use_tma && vec && cols % 512 == 0 && rows % TILE == 0) {
        const unsigned g = (unsigned)std::min<int64_t>(grid, 148 * use_tma);
        if (exact_abs) stats_tma_kernel<true><<<g, FAST_WARPS * 32, 0, s>>>(xp, ld, tiles_w, chunks, item0, grid, ntiles, fmt_mask, table);
        else stats_tma_kernel<false><<<g, FAST_WARPS * 32, 0, s>>>(xp, ld, tiles_w, chunks, item0, grid, ntiles, fmt_mask, table);
        return check_launch("qa_tile_stats(fast, tma)");
    }
    if (vec && exact_abs) stats_fast_kernel<true, true><<<(unsigned)grid, FAST_WARPS * 32, 0, s>>>(xp, rows, cols, ld, tiles_w, chunks, item0, ntiles, fmt_mask, table);
    else if (vec) stats_fast_kernel<true, false><<<(unsigned)grid, FAST_WARPS * 32, 0, s>>>(xp, rows, cols, ld, tiles_w, chunks, item0, ntiles, fmt_mask, table);
    else if (exact_abs) stats_fast_kernel<false, true><<<(unsigned)grid, FAST_WARPS * 32, 0, s>>>(xp, rows, cols, ld, tiles_w, chunks, item0, ntiles, fmt_mask, table);
    else stats_fast_kernel<false, false><<<(unsigned)grid, FAST_WARPS * 32, 0, s>>>(xp, rows, cols, ld, tiles_w, chunks, item0, ntiles, fmt_mask, table);
    return check_launch("qa_tile_stats(fast)");
}

extern "C" int64_t qa_tile_stats_items(int64_t rows, int64_t cols) {
    if (rows <= 0 || cols <= 0) return 0;
    return cdiv(rows, TILE) * cdiv(cols, 512);
}

extern "C" int qa_tile_stats_batch(const qa_batch_desc* descs_dev, int n, int64_t total_items, uint32_t fmt_mask, int mode,
                                   qa_stream_t stream) {
    if (!descs_dev || n <= 0 || total_items <= 0 || total_items > 0x7FFFFFFF) { set_error("qa_tile_stats_batch: bad args"); return 1; }
    if (mode != QA_STATS_FAST && mode != QA_STATS_FAST_APPROX_ABS) { set_error("qa_tile_stats_batch: fast modes only"); return 1; }
    cudaStream_t s = (cudaStream_t)stream;
    if (mode == QA_STATS_FAST) stats_fast_batch_kernel<true><<<(unsigned)total_items, FAST_WARPS * 32, 0, s>>>(descs_dev, n, fmt_mask & 0xFu);
    else stats_fast_batch_kernel<false><<<(unsigned)total_items, FAST_WARPS * 32, 0, s>>>(descs_dev, n, fmt_mask & 0xFu);
    return check_launch("qa_tile_stats_batch");
}

extern "C" int qa_tile_stats_rows(const void* x, int x_dtype, int64_t rows, int64_t cols, int64_t ld, uint32_t fmt_mask, int mode,
                                  double* table, int64_t tile_row_begin, int64_t tile_row_end, qa_stream_t stream) {
    if (rows <= 0 || cols <= 0 || ld < cols || !table) { set_error("qa_tile_stats_rows: bad args"); return 1; }
    if (x_dtype != QA_DT_BF16 || (mode != QA_STATS_FAST && mode != QA_STATS_FAST_APPROX_ABS)) {
        set_error("qa_tile_stats_rows: bf16 input and a fast mode only");
        return 1;
    }
    if (tile_row_begin < 0 || tile_row_end <= tile_row_begin || tile_row_end > cdiv(rows, TILE)) { set_error("qa_tile_stats_rows: bad tile-row range"); return 1; }
    return tile_stats_fast(x, rows, cols, ld, fmt_mask & 0xFu, mode, table, tile_row_begin, tile_row_end, (cudaStream_t)stream);
}

extern "C" int qa_tile_stats(const void* x, int x_dtype, int64_t rows, int64_t cols, int64_t ld,
                             int64_t vec_tail, uint32_t fmt_mask, int mode, double* table,
                             qa_stream_t stream) {
    if (rows < 0 || cols < 0 || ld < cols || !table) { set_error("qa_tile_stats: bad args"); return 1; }
    if (rows == 0 || cols == 0) return 0;
    fmt_mask &= 0xFu;
    const int64_t tiles_h = cdiv(rows, TILE), tiles_w = cdiv(cols, TILE), ntiles = tiles_h * tiles_w;
    cudaStream_t s = (cudaStream_t)stream;
    if (mode == QA_STATS_FAST || mode == QA_STATS_FAST_APPROX_ABS) {
        if (x_dtype != QA_DT_BF16) { set_error("qa_tile_stats: fast mode needs bf16 input (use QA_STATS_STRICT for fp32)"); return 1; }
        return tile_stats_fast(x, rows, cols, ld, fmt_mask, mode, table, 0, tiles_h, s);
    }
    if (mode != QA_STATS_STRICT) { set_error("qa_tile_stats: bad mode"); return 1; }
    const int64_t grid = cdiv(ntiles, STRICT_WARPS);
    if (x_dtype == QA_DT_BF16)
        stats_strict_kernel<QA_DT_BF16><<<(unsigned)grid, STRICT_WARPS * 32, 0, s>>>(x, rows, cols, ld, tiles_w, ntiles, vec_tail, fmt_mask, table);
    else if (x_dtype == QA_DT_F32)
        stats_strict_kernel<QA_DT_F32><<<(unsigned)grid, STRICT_WARPS * 32, 0, s>>>(x, rows, cols, ld, tiles_w, ntiles, vec_tail, fmt_mask, table);
    else { set_error("qa_tile_stats: bad dtype"); return 1; }
    return check_launch("qa_tile_stats(strict)");
}
