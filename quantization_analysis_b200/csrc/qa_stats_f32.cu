// Fused quantize + per-tile statistics for inputs that are NOT bf16-exact: float32 tensors, and fp8 e4m3fn weights with
// per-block inverse scales dequantized on the fly (hf_model_utils.py:199-215 fused into the read: 1 B/element + scales in,
// tile-stat table out).  Real checkpoints take this path - their float32 images carry 24-bit significands.
//
// Same ownership as stats_fast_kernel (a lane owns one 16-element group per row, a CTA one 32-row x 512-column item), but
// the arithmetic has to follow what the reference does to 24-bit values (quantization_formats.py:121-145, mixed_tile_greedy.py
// :147-174):
//   * the aligned mantissa is TRUNCATED by the exponent gap d before the round-to-nearest-even on the dropped bits: the low
//     d fraction bits of the element are cleared (x_tr; all of it for d >= 24), then y = clamp(rne(x_tr * 2^(134-E), step))
//     with the magic-number add is exact (one rounding of an exact sum);
//   * the products are float32 ARRAYS in the reference (x*x, x*y rounded to 24 bits) summed in float64: sum x^2 and sum x*y
//     accumulate __fmul_rn products per element in float64; y*y is exact in float32, so sum y and sum y^2 keep the exact
//     float32 group partials of the bf16 kernel; sum |x-y| accumulates the float32 difference per element (float64 in
//     exact-abs mode, float32 group partials otherwise).
// Every sum equals the reference's NumPy-order float64 sum whenever that sum is exactly representable (the normal case); a tile
// that spans more octaves than float64 holds can differ in the last bits of sum x, sum x^2, sum |x-y| (<= 1e-13 relative), like
// the bf16 kernel's sum x^2.  Groups with E < 76 or E >= 190 (|x| near or past 2^64, inf / nan) use the integer recipe and
// float32 products directly.
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_fp8.h>

#include "qa_common.cuh"

namespace qa {

constexpr int NF = 4;      // accumulator slots: 0 = bf16 (a real quantization for these inputs), 1..3 = bfp8 / bfp4 / bfp2
struct TileAccF {
    double sx, sx2;
    double sy[NF], sy2[NF], sxy[NF], sab[NF];
    float amax[NF];
};
__device__ __forceinline__ void accf_zero(TileAccF& a) {
    a.sx = a.sx2 = 0.0;
#pragma unroll
    for (int f = 0; f < NF; ++f) { a.sy[f] = a.sy2[f] = a.sxy[f] = a.sab[f] = 0.0; a.amax[f] = 0.f; }
}
__device__ __forceinline__ float nanmax(float m, float v) { return (v != v || m != m) ? __uint_as_float(0x7FC00000u) : fmaxf(m, v); }

// two e4m3fn bytes -> two float32 (cvt.rn.f16x2.e4m3x2 is exact: every e4m3 value incl. its subnormals is an f16 normal;
// the two nan codes become nan) - torch's float8_e4m3fn -> float32 conversion of hf_model_utils.py:215
__device__ __forceinline__ float2 e4m3x2_f32(uint32_t two) {
    const __half2_raw h = __nv_cvt_fp8x2_to_halfraw2((__nv_fp8x2_storage_t)(two & 0xFFFFu), __NV_E4M3);
    return __half22float2(*reinterpret_cast<const __half2*>(&h));
}

template <int F> struct FmtF;
template <> struct FmtF<0> { static constexpr float M = 25165824.f, L = 254.f; static constexpr int MB = 7; };
template <> struct FmtF<1> { static constexpr float M = 402653184.f, L = 224.f; static constexpr int MB = 3; };
template <> struct FmtF<2> { static constexpr float M = 1610612736.f, L = 128.f; static constexpr int MB = 1; };

__device__ __forceinline__ float clamp_symf(float y, float L) {
    float r;
    asm("min.xorsign.abs.f32 %0, %1, %2;" : "=f"(r) : "f"(y), "f"(L));
    return r;
}

// generic group: integer quantizer + float32 products + float64 sums, element by element
template <bool EXACT_ABS>
__device__ __noinline__ void groupf_slow(const uint32_t (&u)[GROUP], uint32_t E, TileAccF& a) {
#pragma unroll 1
    for (int i = 0; i < GROUP; ++i) {
        const float x = __uint_as_float(u[i]);
        a.sx += (double)x;
        a.sx2 += (double)__fmul_rn(x, x);
#pragma unroll
        for (int f = 0; f < NF; ++f) {
            const float y = __uint_as_float(recon_bits(f, u[i], E));
            const float r = fabsf(__fsub_rn(x, y));
            a.sy[f] += (double)y;
            a.sy2[f] += (double)__fmul_rn(y, y);
            a.sxy[f] += (double)__fmul_rn(x, y);
            a.sab[f] += (double)r;
            a.amax[f] = nanmax(a.amax[f], r);
        }
    }
}

// sm_100 packed-float2 arithmetic (two fp32 lanes per issue slot)
__device__ __forceinline__ float2 f2add(float2 a, float2 b) { return __fadd2_rn(a, b); }
__device__ __forceinline__ float2 f2sub(float2 a, float2 b) { return __fadd2_rn(a, make_float2(-b.x, -b.y)); }
__device__ __forceinline__ float2 f2mul(float2 a, float2 b) { return __fmul2_rn(a, b); }
__device__ __forceinline__ float2 f2fma(float2 a, float2 b, float2 c) { return __ffma2_rn(a, b, c); }
__device__ __forceinline__ float max3absf(float m, float a, float b) {
    float r;
    asm("max.NaN.abs.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(m), "f"(a), "f"(b));
    return r;
}

struct GroupAccF {      // in-group partials of one BFP format, two lanes (even / odd element)
    float2 sy, sy2, sab;
    float mx;
    double dsxy, dsab;
};

// One BFP format, two elements: x = the elements, Xtr = their truncated images in group units, back = 2^(E-134) twice
template <int F, bool EXACT_ABS>
__device__ __forceinline__ void fmtf_step(const float2 x, const float2 Xtr, const float2 back, GroupAccF& g) {
    const float2 Mv = make_float2(FmtF<F>::M, FmtF<F>::M);
    float2 y = f2sub(f2add(Xtr, Mv), Mv);                              // rne to the format's step (exact: one rounding of an exact sum)
    y.x = clamp_symf(y.x, FmtF<F>::L);
    y.y = clamp_symf(y.y, FmtF<F>::L);
    g.sy = f2add(g.sy, y);
    g.sy2 = f2fma(y, y, g.sy2);                                        // exact small integers in group units
    const float2 yo = f2mul(y, back);                                  // the reconstructions in the tensor's units (exact)
    const float2 p = f2mul(x, yo);                                     // float32 products like the reference's x*y array
    g.dsxy += (double)p.x;
    g.dsxy += (double)p.y;
    const float2 r = f2sub(x, yo);
    if (EXACT_ABS) {
        g.dsab += fabs((double)r.x);
        g.dsab += fabs((double)r.y);
    } else {
        g.sab.x += fabsf(r.x);
        g.sab.y += fabsf(r.y);
    }
    g.mx = max3absf(g.mx, r.x, r.y);
}

template <bool EXACT_ABS>
__device__ __forceinline__ void groupf_fast(const uint32_t (&u)[GROUP], TileAccF& a) {
    float mabs = 0.f;
#pragma unroll
    for (int i = 0; i < GROUP; i += 2) mabs = max3absf(mabs, __uint_as_float(u[i]), __uint_as_float(u[i + 1]));   // a nan surfaces: E = 255
    const uint32_t E = __float_as_uint(mabs) >> 23;
    // generic path (float32 products like the reference) for E < 76: the bf16 slot's sum y^2 is exact below here where the
    // reference rounds y*y in float32's denormal range (the bound of qa_stats.cu's group_fast); E >= 190: the bf16 image
    // of |x| >= 2^64 - 2^55 is 2^64, and y*y (and from E = 191 every product) overflows to inf; E == 255: inf / nan
    if (E < 76u || E >= 190u) {
        if (E == 0u) {                     // zeros / denormals only: every format flushes them; they still count in sum x
#pragma unroll
            for (int i = 0; i < GROUP; ++i) {
                const float x = __uint_as_float(u[i]);
                a.sx += (double)x;
                a.sx2 += (double)__fmul_rn(x, x);
                // bf16 rounds a denormal like any pattern (it may even reach the smallest normal); the BFP formats flush it
                const float yb = __uint_as_float(bf16_rne_bits(u[i]));
                const float rb = fabsf(__fsub_rn(x, yb));
                a.sy[0] += (double)yb; a.sy2[0] += (double)__fmul_rn(yb, yb); a.sxy[0] += (double)__fmul_rn(x, yb);
                a.sab[0] += (double)rb; a.amax[0] = fmaxf(a.amax[0], rb);
#pragma unroll
                for (int f = 1; f < NF; ++f) { a.sab[f] += (double)fabsf(x); a.amax[f] = fmaxf(a.amax[f], fabsf(x)); }
            }
            return;
        }
        TileAccF t;
        accf_zero(t);
        uint32_t uc[GROUP];
#pragma unroll
        for (int i = 0; i < GROUP; ++i) uc[i] = u[i];
        groupf_slow<EXACT_ABS>(uc, E, t);
        a.sx += t.sx; a.sx2 += t.sx2;
#pragma unroll
        for (int f = 0; f < NF; ++f) {
            a.sy[f] += t.sy[f]; a.sy2[f] += t.sy2[f]; a.sxy[f] += t.sxy[f]; a.sab[f] += t.sab[f];
            a.amax[f] = nanmax(a.amax[f], t.amax[f]);
        }
        return;
    }
    const float inv = __uint_as_float((261u - E) << 23);    // 2^(134-E)
    const float bk = __uint_as_float((E - 7u) << 23);       // 2^(E-134)
    const float2 inv2 = make_float2(inv, inv), back = make_float2(bk, bk);
    GroupAccF g[3];
#pragma unroll
    for (int f = 0; f < 3; ++f) {
        g[f].sy = g[f].sy2 = g[f].sab = make_float2(0.f, 0.f);
        g[f].mx = 0.f;
        g[f].dsxy = g[f].dsab = 0.0;
    }
    double gx = 0.0, gx2 = 0.0, dsy0 = 0.0, dsy20 = 0.0, dsxy0 = 0.0, dsab0 = 0.0;
    float2 gsab0 = make_float2(0.f, 0.f);
    float gmx0 = 0.f;
#pragma unroll
    for (int i = 0; i < GROUP; i += 2) {
        const uint32_t ua = u[i], ub = u[i + 1];
        const float2 x = make_float2(__uint_as_float(ua), __uint_as_float(ub));
        const float2 xx = f2mul(x, x);                               // float32 squares like the reference's x*x array
        gx += (double)x.x;
        gx += (double)x.y;
        gx2 += (double)xx.x;
        gx2 += (double)xx.y;
        // the reference shifts the 24-bit mantissa right by d = E - e BEFORE rounding (quantization_formats.py:125-131): clear the
        // d low bits that fall off.  shl.b32 gives 0 for d >= 32; for 24 <= d < 32 the mask also eats exponent bits, which only
        // makes an element that rounds to zero in every format smaller.
        uint32_t ma, mb;
        asm("shl.b32 %0, %1, %2;" : "=r"(ma) : "r"(0xFFFFFFFFu), "r"(E - ((ua >> 23) & 0xFFu)));
        asm("shl.b32 %0, %1, %2;" : "=r"(mb) : "r"(0xFFFFFFFFu), "r"(E - ((ub >> 23) & 0xFFu)));
        const float2 Xtr = f2mul(make_float2(__uint_as_float(ua & ma), __uint_as_float(ub & mb)), inv2);
        fmtf_step<0, EXACT_ABS>(x, Xtr, back, g[0]);
        fmtf_step<1, EXACT_ABS>(x, Xtr, back, g[1]);
        fmtf_step<2, EXACT_ABS>(x, Xtr, back, g[2]);
        {   // bf16: round to nearest even on the pattern (quantization_formats.py:29-35; one cvt.rn.bf16x2.f32 for the pair).
            // A per-element floating-point format: its reconstructions do not share the group's grid, so sum y and sum y^2 go
            // through float64 per element (y*y is exact in float32 and in float64: the DFMA rounds the sum only).
            const __nv_bfloat162 q = __float22bfloat162_rn(x);
            const uint32_t qb = *reinterpret_cast<const uint32_t*>(&q);
            const float2 yo = make_float2(__uint_as_float(qb << 16), __uint_as_float(qb & 0xFFFF0000u));
            const double ya = (double)yo.x, yb = (double)yo.y;
            dsy0 += ya;
            dsy0 += yb;
            dsy20 = fma(ya, ya, dsy20);
            dsy20 = fma(yb, yb, dsy20);
            const float2 p = f2mul(x, yo);
            dsxy0 += (double)p.x;
            dsxy0 += (double)p.y;
            const float2 r = f2sub(x, yo);
            if (EXACT_ABS) {
                dsab0 += fabs((double)r.x);
                dsab0 += fabs((double)r.y);
            } else {
                gsab0.x += fabsf(r.x);
                gsab0.y += fabsf(r.y);
            }
            gmx0 = max3absf(gmx0, r.x, r.y);
        }
    }
    const double s1 = __hiloint2double((int)((E + 889u) << 20), 0);        // 2^(E-134)
    const double s2 = __hiloint2double((int)((2u * E + 755u) << 20), 0);   // 2^(2E-268)
    a.sx += gx;
    a.sx2 += gx2;
    a.sy[0] += dsy0;
    a.sy2[0] += dsy20;
    a.sxy[0] += dsxy0;
    a.sab[0] += EXACT_ABS ? dsab0 : (double)(gsab0.x + gsab0.y);
    a.amax[0] = fmaxf(a.amax[0], gmx0);
#pragma unroll
    for (int f = 0; f < 3; ++f) {
        a.sy[f + 1] = fma((double)(g[f].sy.x + g[f].sy.y), s1, a.sy[f + 1]);
        a.sy2[f + 1] = fma((double)(g[f].sy2.x + g[f].sy2.y), s2, a.sy2[f + 1]);
        a.sxy[f + 1] += g[f].dsxy;
        a.sab[f + 1] += EXACT_ABS ? g[f].dsab : (double)(g[f].sab.x + g[f].sab.y);
        a.amax[f + 1] = fmaxf(a.amax[f + 1], g[f].mx);
    }
}

__device__ __forceinline__ double shfl_xor_df(double v, int m) {
    return __hiloint2double(__shfl_xor_sync(0xFFFFFFFFu, __double2hiint(v), m), __shfl_xor_sync(0xFFFFFFFFu, __double2loint(v), m));
}

constexpr int F32_WARPS = 4;
constexpr int F32_RPW = TILE / F32_WARPS;

struct Fp8Src {
    const float* scale;      // [scale_rows][scale_cols] inverse scales; nullptr: plain float32 input
    int64_t scols, br, bc;   // scale columns, block rows, block columns
};

// SRC 0: x is float32 [rows][ld]; SRC 1: x is uint8 e4m3fn [rows][ld] with per-block scales
template <int SRC, bool EXACT_ABS>
__global__ void __launch_bounds__(F32_WARPS * 32, 3) stats_f32_kernel(const void* __restrict__ x, int64_t rows, int64_t cols, int64_t ld,
                                                                      int64_t tiles_w, int64_t chunks, int64_t item0, int64_t ntiles,
                                                                      uint32_t fmt_mask, Fp8Src src, double* __restrict__ table,
                                                                      unsigned long long* __restrict__ inexact) {
    __shared__ double part[F32_WARPS - 1][18][32];
    __shared__ float partmx[F32_WARPS - 1][NF][32];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int64_t item = blockIdx.x + item0;          // item0 > 0: a launch that covers a range of tile rows
    const int64_t tr = item / chunks, ck = item - tr * chunks;
    const int64_t col0 = ck * 512 + (int64_t)lane * GROUP;
    const int64_t row0 = tr * TILE + w * F32_RPW;
    const int nrows = (int)max((int64_t)0, min((int64_t)F32_RPW, rows - row0));
    TileAccF a;
    accf_zero(a);
    unsigned bad = 0;
    if (col0 < cols) {
        // fp8 source: a full, 16-byte aligned group is one LDG.128; the next row's is requested before this row is processed
        const uint8_t* p8 = reinterpret_cast<const uint8_t*>(x) + row0 * ld + col0;
        const bool full8 = SRC == 1 && col0 + GROUP <= cols && ((reinterpret_cast<uintptr_t>(p8) | (uintptr_t)ld) & 15) == 0;
        uint4 qn = make_uint4(0u, 0u, 0u, 0u);
        if (full8 && nrows > 0) qn = __ldg(reinterpret_cast<const uint4*>(p8));
        for (int r = 0; r < nrows; ++r) {
            const int64_t row = row0 + r;
            uint32_t u[GROUP];
            if (SRC == 0) {
                const uint32_t* p = reinterpret_cast<const uint32_t*>(x) + row * ld + col0;
                if (col0 + GROUP <= cols && (reinterpret_cast<uintptr_t>(p) & 31) == 0) {
                    uint32_t t8[8];
                    ldg256(p, t8);
#pragma unroll
                    for (int i = 0; i < 8; ++i) u[i] = t8[i];
                    ldg256(p + 8, t8);
#pragma unroll
                    for (int i = 0; i < 8; ++i) u[8 + i] = t8[i];
                } else {
#pragma unroll
                    for (int i = 0; i < GROUP; ++i) u[i] = col0 + i < cols ? p[i] : 0u;
                }
            } else {
                const uint8_t* p = p8 + (int64_t)r * ld;
                uint32_t wv[4];
                if (full8) {
                    wv[0] = qn.x; wv[1] = qn.y; wv[2] = qn.z; wv[3] = qn.w;
                    if (r + 1 < nrows) qn = __ldg(reinterpret_cast<const uint4*>(p + ld));
                } else {
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        wv[k] = 0;
#pragma unroll
                        for (int j = 0; j < 4; ++j)
                            if (col0 + 4 * k + j < cols) wv[k] |= (uint32_t)p[4 * k + j] << (8 * j);
                    }
                }
                // one inverse scale per 16-element group when the group lies inside one scale block (block widths are multiples
                // of 16 in every checkpoint format in use: 128); a group that straddles two blocks looks its scales up per element.
                // Columns past the end read as byte 0 = +0.0; a nan code stays a nan (any payload: only arithmetic sees it).
                const float* srow = src.scale + (row / src.br) * src.scols;
                const int64_t cb0 = col0 / src.bc, cb1 = min(col0 + GROUP - 1, cols - 1) / src.bc;
                const float sc0 = srow[cb0];
                if (cb0 == cb1) {
                    const float2 sc2 = make_float2(sc0, sc0);
#pragma unroll
                    for (int i = 0; i < GROUP; i += 2) {
                        const float2 v = __fmul2_rn(e4m3x2_f32(wv[i >> 2] >> (8 * (i & 3))), sc2);      // hf_model_utils.py:209-215
                        u[i] = __float_as_uint(v.x);
                        u[i + 1] = __float_as_uint(v.y);
                    }
                } else {
#pragma unroll
                    for (int i = 0; i < GROUP; i += 2) {
                        const float2 q = e4m3x2_f32(wv[i >> 2] >> (8 * (i & 3)));
                        u[i] = __float_as_uint(__fmul_rn(q.x, srow[min(col0 + i, cols - 1) / src.bc]));
                        u[i + 1] = __float_as_uint(__fmul_rn(q.y, srow[min(col0 + i + 1, cols - 1) / src.bc]));
                    }
                }
            }
            if (inexact) {
#pragma unroll
                for (int i = 0; i < GROUP; ++i) bad += (u[i] & 0xFFFFu) != 0u && (u[i] & 0x7FFFFFFFu) <= 0x7F800000u;   // a nan is not counted
            }
            groupf_fast<EXACT_ABS>(u, a);
        }
    }
    if (inexact) {
        bad = __reduce_add_sync(0xFFFFFFFFu, bad);
        if (lane == 0 && bad) atomicAdd(inexact, (unsigned long long)bad);
    }
    if (w > 0) {
        double (*p)[32] = part[w - 1];
        p[0][lane] = a.sx; p[1][lane] = a.sx2;
#pragma unroll
        for (int f = 0; f < NF; ++f) {
            p[2 + f][lane] = a.sy[f]; p[6 + f][lane] = a.sy2[f]; p[10 + f][lane] = a.sxy[f]; p[14 + f][lane] = a.sab[f];
            partmx[w - 1][f][lane] = a.amax[f];
        }
    }
    __syncthreads();
    if (w != 0) return;
#pragma unroll
    for (int q = 0; q < F32_WARPS - 1; ++q) {
        a.sx += part[q][0][lane]; a.sx2 += part[q][1][lane];
#pragma unroll
        for (int f = 0; f < NF; ++f) {
            a.sy[f] += part[q][2 + f][lane]; a.sy2[f] += part[q][6 + f][lane];
            a.sxy[f] += part[q][10 + f][lane]; a.sab[f] += part[q][14 + f][lane];
            a.amax[f] = nanmax(a.amax[f], partmx[q][f][lane]);
        }
    }
    a.sx += shfl_xor_df(a.sx, 1);
    a.sx2 += shfl_xor_df(a.sx2, 1);
#pragma unroll
    for (int f = 0; f < NF; ++f) {
        a.sy[f] += shfl_xor_df(a.sy[f], 1); a.sy2[f] += shfl_xor_df(a.sy2[f], 1);
        a.sxy[f] += shfl_xor_df(a.sxy[f], 1); a.sab[f] += shfl_xor_df(a.sab[f], 1);
        a.amax[f] = nanmax(a.amax[f], __shfl_xor_sync(0xFFFFFFFFu, a.amax[f], 1));
    }
    const int64_t tc = ck * 16 + (lane >> 1);
    if ((lane & 1) == 0 && tc < tiles_w) {
        const int64_t t = tr * tiles_w + tc;
        table[QA_STAT_SX * ntiles + t] = a.sx;
        table[QA_STAT_SX2 * ntiles + t] = a.sx2;
#pragma unroll
        for (int f = 0; f < NF; ++f) {
            if (fmt_mask & (1u << f)) {
                table[QA_STAT_FMT(f, 0) * ntiles + t] = a.sy[f];
                table[QA_STAT_FMT(f, 1) * ntiles + t] = a.sy2[f];
                table[QA_STAT_FMT(f, 2) * ntiles + t] = a.sxy[f];
                table[QA_STAT_FMT(f, 3) * ntiles + t] = a.sab[f];
                // the fast path's fmaxf maxima drop a nan that an earlier group of the lane left in amax; sum |x - y| is a
                // sum of terms >= 0, nan exactly when one of them is, so it restores np.max's nan
                table[QA_STAT_FMT(f, 4) * ntiles + t] = a.sab[f] != a.sab[f] ? a.sab[f] : (double)a.amax[f];
            }
        }
    }
}

}  // namespace qa

using namespace qa;

static int launch_f32(int src, const void* x, const float* scale, int64_t rows, int64_t cols, int64_t ld, int64_t scale_rows,
                      int64_t scale_cols, uint32_t fmt_mask, int mode, double* table, int64_t tile_row_begin, int64_t tile_row_end,
                      unsigned long long* inexact, cudaStream_t s, const char* who) {
    const int64_t tiles_h = cdiv(rows, TILE), tiles_w = cdiv(cols, TILE), ntiles = tiles_h * tiles_w;
    const int64_t chunks = cdiv(cols, 512);
    if (tile_row_end < 0) tile_row_end = tiles_h;
    if (tile_row_begin < 0 || tile_row_end <= tile_row_begin || tile_row_end > tiles_h) { set_error("%s: bad tile-row range", who); return 1; }
    Fp8Src fs{scale, scale_cols, 1, 1};
    if (src == 1) {
        fs.br = std::max<int64_t>(1, cdiv(rows, scale_rows));
        fs.bc = std::max<int64_t>(1, cdiv(cols, scale_cols));
        if (cdiv(rows, fs.br) > scale_rows || cdiv(cols, fs.bc) > scale_cols) { set_error("%s: scale shape too small", who); return 1; }
        if (inexact && tile_row_begin == 0 && cudaMemsetAsync(inexact, 0, sizeof(unsigned long long), s) != cudaSuccess) return check_launch(who);
    }
    const unsigned grid = (unsigned)((tile_row_end - tile_row_begin) * chunks);
    const int64_t item0 = tile_row_begin * chunks;
    const bool exact = mode == QA_STATS_FAST;
#define QA_F32_LAUNCH(SRC, EX) stats_f32_kernel<SRC, EX><<<grid, F32_WARPS * 32, 0, s>>>(x, rows, cols, ld, tiles_w, chunks, item0, ntiles, fmt_mask, fs, table, inexact)
    if (src == 0) { if (exact) QA_F32_LAUNCH(0, true); else QA_F32_LAUNCH(0, false); }
    else { if (exact) QA_F32_LAUNCH(1, true); else QA_F32_LAUNCH(1, false); }
#undef QA_F32_LAUNCH
    return check_launch(who);
}

extern "C" int qa_tile_stats_f32(const float* x, int64_t rows, int64_t cols, int64_t ld, uint32_t fmt_mask, int mode, double* table,
                                 int64_t tile_row_begin, int64_t tile_row_end, qa_stream_t stream) {
    if (!x || rows <= 0 || cols <= 0 || ld < cols || !table) { set_error("qa_tile_stats_f32: bad args"); return 1; }
    if (mode != QA_STATS_FAST && mode != QA_STATS_FAST_APPROX_ABS) { set_error("qa_tile_stats_f32: fast modes only"); return 1; }
    return launch_f32(0, x, nullptr, rows, cols, ld, 1, 1, fmt_mask & 0xFu, mode, table, tile_row_begin, tile_row_end, nullptr,
                      (cudaStream_t)stream, "qa_tile_stats_f32");
}

extern "C" int qa_tile_stats_fp8(const void* w_fp8, const float* scale_inv, int64_t rows, int64_t cols, int64_t ld, int64_t scale_rows,
                                 int64_t scale_cols, uint32_t fmt_mask, int mode, double* table, int64_t tile_row_begin,
                                 int64_t tile_row_end, unsigned long long* inexact_count, qa_stream_t stream) {
    if (!w_fp8 || !scale_inv || rows <= 0 || cols <= 0 || ld < cols || scale_rows <= 0 || scale_cols <= 0 || !table) {
        set_error("qa_tile_stats_fp8: bad args");
        return 1;
    }
    if (mode != QA_STATS_FAST && mode != QA_STATS_FAST_APPROX_ABS) { set_error("qa_tile_stats_fp8: fast modes only"); return 1; }
    return launch_f32(1, w_fp8, scale_inv, rows, cols, ld, scale_rows, scale_cols, fmt_mask & 0xFu, mode, table, tile_row_begin,
                      tile_row_end, inexact_count, (cudaStream_t)stream, "qa_tile_stats_fp8");
}
