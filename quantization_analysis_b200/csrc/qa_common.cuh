// Shared device helpers: bit-exact BFP quantizer, group loads, PCG64, error plumbing.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/qa_b200.h"

namespace qa {

constexpr int TILE = 32;
constexpr int GROUP = 16;

void set_error(const char* fmt, ...);
int check_launch(const char* what);

// qa_greedy_assign_sweep for atol (qa_assign.cu): the one-thread chain, one block per threshold.  Block k's scratch and
// end-of-stream slot lie k * stride bytes after work / rng_out; every chain starts from *rng.
int greedy_seq_sweep_launch(const double* table, int64_t ntiles, double numel, const double* thresholds, int nthr,
                            const int32_t* fmt_order, int nfmt, const qa_pcg64* rng, qa_pcg64* rng_out, int8_t* assignment,
                            int64_t* counts, double* state, void* work, int64_t stride, cudaStream_t stream);

__host__ __device__ inline int64_t cdiv(int64_t a, int64_t b) { return (a + b - 1) / b; }

// ---------------------------------------------------------------------------------------
// Bit-exact TTNN-style BFP reconstruction of one element (quantization_formats.py:121-158).
// u = float32 bit pattern, E = shared (max) biased exponent of its 16-element group.
// Returns the float32 bit pattern of the reconstruction (low 16 bits are always zero).
// ---------------------------------------------------------------------------------------
template <int MB>
__device__ __forceinline__ uint32_t bfp_recon_bits(uint32_t u, uint32_t E) {
    const uint32_t e = (u >> 23) & 0xFFu;
    const uint32_t d = E - e;                                  // >= 0: E is the group max
    const uint32_t m24 = (u & 0x7FFFFFu) | 0x800000u;
    const uint32_t m = d >= 24u ? 0u : (m24 >> d);             // :125-131 (shifts >= 24 clear it)
    constexpr uint32_t DROP = 24 - MB;
    constexpr uint32_t HALF = 1u << (DROP - 1);
    const uint32_t low = m & ((1u << DROP) - 1u);
    uint32_t q = m >> DROP;
    const uint32_t up = (low > HALF) | ((low == HALF) & (q & 1u));  // round half to even (:133-140)
    q = min(q + up, (1u << MB) - 1u);                          // clamp, no exponent bump (:141)
    if (e == 0u) q = 0u;                                       // zero / denormal inputs flush (:145)
    if (q == 0u) return 0u;                                    // sign dropped with the mantissa (:143)
    const uint32_t ls = (uint32_t)(MB - 1) - (uint32_t)(31 - __clz(q));  // decode table (:71-81)
    const uint32_t frac = (q << (ls + 1u)) & ((1u << MB) - 1u);
    const uint32_t eo = E - ls;                                // uint32 arithmetic as in :154
    return (u & 0x80000000u) | (eo << 23) | (frac << (23 - MB));
}

// bf16 round-to-nearest-even on the raw pattern, wrapping add (quantization_formats.py:29-35)
__device__ __forceinline__ uint32_t bf16_rne_bits(uint32_t u) {
    return ((u + 0x7FFFu + ((u >> 16) & 1u)) >> 16) << 16;
}

__device__ __forceinline__ uint32_t recon_bits(int fmt, uint32_t u, uint32_t E) {
    switch (fmt) {
        case 0: return bf16_rne_bits(u);
        case 1: return bfp_recon_bits<7>(u, E);
        case 2: return bfp_recon_bits<3>(u, E);
        default: return bfp_recon_bits<1>(u, E);
    }
}

__device__ __forceinline__ uint32_t group_max_exp(const uint32_t (&u)[GROUP]) {
    uint32_t m = 0;
#pragma unroll
    for (int i = 0; i < GROUP; ++i) m = max(m, u[i] & 0x7F800000u);
    return m >> 23;
}

// Load one 16-element group as float32 bit patterns; out-of-range columns read as +0.
template <int DT>
__device__ __forceinline__ void load_group_scalar(const void* x, int64_t row, int64_t col0,
                                                  int64_t cols, int64_t ld, uint32_t (&u)[GROUP]) {
#pragma unroll
    for (int i = 0; i < GROUP; ++i) {
        const int64_t c = col0 + i;
        uint32_t v = 0;
        if (c < cols) {
            if (DT == QA_DT_BF16)
                v = (uint32_t)reinterpret_cast<const uint16_t*>(x)[row * ld + c] << 16;
            else
                v = reinterpret_cast<const uint32_t*>(x)[row * ld + c];
        }
        u[i] = v;
    }
}

__device__ __forceinline__ void ldg256(const void* p, uint32_t (&r)[8]) {
    asm volatile("ld.global.nc.L1::no_allocate.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]),
                   "=r"(r[6]), "=r"(r[7])
                 : "l"(p));
}
__device__ __forceinline__ void stg256(void* p, const uint32_t (&r)[8]) {
    asm volatile("st.global.L1::no_allocate.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "r"(r[0]),
                 "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
                 : "memory");
}

// ---------------------------------------------------------------------------------------
// numpy.random PCG64 (XSL-RR 128/64) — SURVEY.md Appendix B3
// ---------------------------------------------------------------------------------------
struct u128 {
    uint64_t hi, lo;
};
__host__ __device__ inline u128 mul128(u128 a, u128 b) {
    u128 r;
    r.lo = a.lo * b.lo;
#ifdef __CUDA_ARCH__
    r.hi = __umul64hi(a.lo, b.lo) + a.hi * b.lo + a.lo * b.hi;
#else
    r.hi = (uint64_t)(((unsigned __int128)a.lo * b.lo) >> 64) + a.hi * b.lo + a.lo * b.hi;
#endif
    return r;
}
__host__ __device__ inline u128 add128(u128 a, u128 b) {
    u128 r;
    r.lo = a.lo + b.lo;
    r.hi = a.hi + b.hi + (r.lo < a.lo ? 1ull : 0ull);
    return r;
}
#define QA_PCG_MULT_HI 0x2360ED051FC65DA4ull
#define QA_PCG_MULT_LO 0x4385DF649FCCF645ull

struct Pcg {
    u128 s, inc;
    uint32_t has32, buf32;
    __device__ void load(const qa_pcg64* p) {
        s.hi = p->state_hi; s.lo = p->state_lo; inc.hi = p->inc_hi; inc.lo = p->inc_lo;
        has32 = p->has_uint32; buf32 = p->uinteger;
    }
    __device__ void store(qa_pcg64* p) const {
        p->state_hi = s.hi; p->state_lo = s.lo; p->has_uint32 = has32; p->uinteger = buf32;
    }
    __device__ __forceinline__ uint64_t next64() {
        s = add128(mul128(s, u128{QA_PCG_MULT_HI, QA_PCG_MULT_LO}), inc);
        const uint64_t x = s.hi ^ s.lo;
        const uint32_t rot = (uint32_t)(s.hi >> 58);
        return (x >> rot) | (x << ((64u - rot) & 63u));
    }
    __device__ __forceinline__ uint32_t next32() {
        if (has32) { has32 = 0; return buf32; }
        const uint64_t v = next64();
        has32 = 1; buf32 = (uint32_t)(v >> 32);
        return (uint32_t)v;
    }
    // advance the LCG by `delta` steps (no output)
    __device__ void advance(uint64_t delta) {
        u128 am{0, 1}, ap{0, 0}, cm{QA_PCG_MULT_HI, QA_PCG_MULT_LO}, cp = inc;
        while (delta) {
            if (delta & 1ull) { am = mul128(am, cm); ap = add128(mul128(ap, cm), cp); }
            cp = mul128(add128(cm, u128{0, 1}), cp);
            cm = mul128(cm, cm);
            delta >>= 1;
        }
        s = add128(mul128(am, s), ap);
    }
    // numpy random_interval(max) for max <= 0xffffffff: masked rejection on 32-bit draws
    __device__ __forceinline__ uint32_t interval(uint32_t mx) {
        if (mx == 0) return 0;
        const uint32_t mask = 0xFFFFFFFFu >> __clz(mx);
        uint32_t v;
        do { v = next32() & mask; } while (v > mx);
        return v;
    }
};

}  // namespace qa
