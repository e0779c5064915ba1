// Assignment kernels over the tile-stat table / tile-score arrays, and the NumPy RNG stream.
#include "qa_common.cuh"

namespace qa {

// ------------------------------------------------------------------------------------------
// NumPy Generator stream
// ------------------------------------------------------------------------------------------
// Fisher-Yates exactly as numpy's _shuffle_raw: for i = n-1 .. 1: j = interval(i); swap(i, j).
__device__ void permutation_seq(Pcg& g, int64_t n, int32_t* a) {
    for (int64_t i = 0; i < n; ++i) a[i] = (int32_t)i;
    for (int64_t i = n - 1; i >= 1; --i) {
        const uint32_t j = g.interval((uint32_t)i);
        const int32_t t = a[i];
        a[i] = a[j];
        a[j] = t;
    }
}

__global__ void permutation_kernel(qa_pcg64* rng, int64_t n, int32_t* out) {
    if (blockIdx.x || threadIdx.x) return;
    Pcg g;
    g.load(rng);
    permutation_seq(g, n, out);
    g.store(rng);
}

// integers(0, k, n): Lemire's method on 32-bit draws (numpy _bounded_uint32 path, rng = k-1)
__device__ __forceinline__ uint32_t bounded32(Pcg& g, uint32_t k) {
    uint64_t m = (uint64_t)g.next32() * k;
    uint32_t left = (uint32_t)m;
    if (left < k) {
        const uint32_t thr = (0u - k) % k;
        while (left < thr) {
            m = (uint64_t)g.next32() * k;
            left = (uint32_t)m;
        }
    }
    return (uint32_t)(m >> 32);
}

__global__ void integers_kernel(qa_pcg64* rng, uint32_t k, int64_t n, int8_t* out) {
    if (blockIdx.x || threadIdx.x) return;
    if (k <= 1) {
        for (int64_t i = 0; i < n; ++i) out[i] = 0;
        return;
    }
    Pcg g;
    g.load(rng);
    for (int64_t i = 0; i < n; ++i) out[i] = (int8_t)bounded32(g, k);
    g.store(rng);
}

// ------------------------------------------------------------------------------------------
// Greedy (sequential decision chain; mixed_tile_greedy.py:135-346)
// ------------------------------------------------------------------------------------------
struct OrderArg {
    int32_t fmt[QA_NFMT];
    int n;
};

struct GreedyWork {
    int32_t* perm;      // [n]
    int32_t* cand;      // [n]
    uint8_t* fixed;     // [n]
};

__device__ __forceinline__ double pcc_value(double n, double sx, double sx2, double sy, double sy2,
                                            double sxy, double sabs) {
    // mixed_tile_greedy.py:176-190 in Python-float evaluation order (no contraction)
    if (n == 0.0) return 1.0;
    const double mx = __ddiv_rn(sx, n);
    const double my = __ddiv_rn(sy, n);
    double am2 = __dsub_rn(sx2, __dmul_rn(__dmul_rn(n, mx), mx));
    double bm2 = __dsub_rn(sy2, __dmul_rn(__dmul_rn(n, my), my));
    if (am2 < 0.0) am2 = 0.0;
    if (bm2 < 0.0) bm2 = 0.0;
    const double den = __dsqrt_rn(__dmul_rn(am2, bm2));
    if (den == 0.0) return sabs == 0.0 ? 1.0 : 0.0;
    return __ddiv_rn(__dsub_rn(sxy, __dmul_rn(__dmul_rn(n, mx), my)), den);
}

__device__ __forceinline__ bool good(double v, int metric, double thr) {
    return metric == QA_METRIC_PCC ? v >= thr : v <= thr;
}

// The stream starts at *rng_in and its final position goes to *rng_out (the same pointer for a single run).
__device__ __forceinline__ void greedy_seq(const double* __restrict__ table, int64_t nt, double numel, int metric, double thr,
                                           OrderArg ord, const qa_pcg64* rng_in, qa_pcg64* rng_out, int8_t* assignment,
                                           int64_t* counts, double* state, GreedyWork w) {
    const int nfmt = ord.n;
    const int base = ord.fmt[0];
    int64_t cnt[QA_NFMT] = {0, 0, 0, 0};
    cnt[base] = nt;
    double sx = 0.0, sx2 = 0.0, sy = 0.0, sy2 = 0.0, sxy = 0.0, sabs = 0.0;
    double max_abs = 0.0;
    int64_t max_cnt = 0;
    const double* bsy = table + QA_STAT_FMT(base, 0) * nt;
    const double* bsy2 = table + QA_STAT_FMT(base, 1) * nt;
    const double* bsxy = table + QA_STAT_FMT(base, 2) * nt;
    const double* bsab = table + QA_STAT_FMT(base, 3) * nt;
    const double* bmax = table + QA_STAT_FMT(base, 4) * nt;
    // sequential float64 accumulation in tile order (:165-170)
    for (int64_t t = 0; t < nt; ++t) {
        assignment[t] = (int8_t)base;
        w.fixed[t] = 0;
        if (metric == QA_METRIC_PCC) {
            sx = __dadd_rn(sx, table[QA_STAT_SX * nt + t]);
            sx2 = __dadd_rn(sx2, table[QA_STAT_SX2 * nt + t]);
            sy = __dadd_rn(sy, bsy[t]);
            sy2 = __dadd_rn(sy2, bsy2[t]);
            sxy = __dadd_rn(sxy, bsxy[t]);
            sabs = __dadd_rn(sabs, bsab[t]);
        } else if (metric == QA_METRIC_MAE) {
            sabs = __dadd_rn(sabs, bsab[t]);
        } else {
            const double v = bmax[t];
            if (t == 0 || v > max_abs) { max_abs = v; max_cnt = 1; }
            else if (v == max_abs) ++max_cnt;
        }
    }
    Pcg g;
    g.load(rng_in);
    for (int fi = 0; fi < nfmt; ++fi) {
        const int fmt = ord.fmt[fi];
        int64_t m = 0;
        for (int64_t t = 0; t < nt; ++t)
            if (!w.fixed[t]) w.cand[m++] = (int32_t)t;
        if (m == 0) break;
        permutation_seq(g, m, w.perm);
        const double* fsy = table + QA_STAT_FMT(fmt, 0) * nt;
        const double* fsy2 = table + QA_STAT_FMT(fmt, 1) * nt;
        const double* fsxy = table + QA_STAT_FMT(fmt, 2) * nt;
        const double* fsab = table + QA_STAT_FMT(fmt, 3) * nt;
        const double* fmax = table + QA_STAT_FMT(fmt, 4) * nt;
        for (int64_t k = 0; k < m; ++k) {
            const int64_t t = w.cand[w.perm[k]];
            const int prev = assignment[t];
            if (prev == fmt) {
                double cur;
                if (metric == QA_METRIC_PCC) cur = pcc_value(numel, sx, sx2, sy, sy2, sxy, sabs);
                else if (metric == QA_METRIC_MAE) cur = numel != 0.0 ? __ddiv_rn(sabs, numel) : 0.0;
                else cur = max_abs;
                if (!good(cur, metric, thr)) w.fixed[t] = 1;
                continue;
            }
            bool accept;
            if (metric == QA_METRIC_PCC) {
                const double c_sy = __dadd_rn(sy, __dsub_rn(fsy[t], table[QA_STAT_FMT(prev, 0) * nt + t]));
                const double c_sy2 = __dadd_rn(sy2, __dsub_rn(fsy2[t], table[QA_STAT_FMT(prev, 1) * nt + t]));
                const double c_sxy = __dadd_rn(sxy, __dsub_rn(fsxy[t], table[QA_STAT_FMT(prev, 2) * nt + t]));
                const double c_sab = __dadd_rn(sabs, __dsub_rn(fsab[t], table[QA_STAT_FMT(prev, 3) * nt + t]));
                accept = good(pcc_value(numel, sx, sx2, c_sy, c_sy2, c_sxy, c_sab), metric, thr);
                if (accept) { sy = c_sy; sy2 = c_sy2; sxy = c_sxy; sabs = c_sab; }
            } else if (metric == QA_METRIC_MAE) {
                const double c_sab = __dadd_rn(sabs, __dsub_rn(fsab[t], table[QA_STAT_FMT(prev, 3) * nt + t]));
                accept = good(numel != 0.0 ? __ddiv_rn(c_sab, numel) : 0.0, metric, thr);
                if (accept) sabs = c_sab;
            } else {
                const double new_max = fmax[t];
                const double old_max = table[QA_STAT_FMT(prev, 4) * nt + t];
                double c_max = max_abs;
                int64_t c_cnt = max_cnt;
                bool rescan = false;
                if (new_max > max_abs) { c_max = new_max; c_cnt = 1; }
                else if (new_max == max_abs) { if (old_max != max_abs) c_cnt = max_cnt + 1; }
                else if (old_max == max_abs) {
                    if (max_cnt > 1) c_cnt = max_cnt - 1;
                    else rescan = true;
                }
                if (rescan) {  // the unique maximum tile shrinks: recompute over current per-tile maxima (:331-335)
                    c_max = new_max; c_cnt = 1;
                    bool first = true;
                    for (int64_t q = 0; q < nt; ++q) {
                        const double v = q == t ? new_max : table[QA_STAT_FMT(assignment[q], 4) * nt + q];
                        if (first || v > c_max) { c_max = v; c_cnt = 1; first = false; }
                        else if (v == c_max) ++c_cnt;
                    }
                }
                accept = good(c_max, metric, thr);
                if (accept) { max_abs = c_max; max_cnt = c_cnt; }
            }
            if (accept) {
                --cnt[prev];
                ++cnt[fmt];
                assignment[t] = (int8_t)fmt;
            } else {
                w.fixed[t] = 1;
            }
        }
    }
    g.store(rng_out);
    for (int f = 0; f < QA_NFMT; ++f) counts[f] = cnt[f];
    state[0] = sx; state[1] = sx2; state[2] = sy; state[3] = sy2; state[4] = sxy; state[5] = sabs;
    state[6] = max_abs;
    state[7] = metric == QA_METRIC_PCC ? pcc_value(numel, sx, sx2, sy, sy2, sxy, sabs)
             : metric == QA_METRIC_MAE ? (numel != 0.0 ? __ddiv_rn(sabs, numel) : 0.0) : max_abs;
}

__global__ void greedy_seq_kernel(const double* __restrict__ table, int64_t nt, double numel, int metric,
                                  double thr, OrderArg ord, qa_pcg64* rng,
                                  int8_t* assignment, int64_t* counts, double* state, GreedyWork w) {
    if (blockIdx.x || threadIdx.x) return;
    greedy_seq(table, nt, numel, metric, thr, ord, rng, rng, assignment, counts, state, w);
}

// atol sweep: block k runs the chain with thresholds[k] on its own slice of the work (`stride` bytes per block) and outputs
__global__ void greedy_seq_sweep_kernel(const double* __restrict__ table, int64_t nt, double numel, const double* __restrict__ thresholds,
                                        OrderArg ord, const qa_pcg64* rng, qa_pcg64* rng_out, int8_t* assignment, int64_t* counts,
                                        double* state, GreedyWork w, int64_t stride) {
    if (threadIdx.x) return;
    const int64_t k = blockIdx.x, off = k * stride;
    auto mine = [off](auto* p) { return reinterpret_cast<decltype(p)>(reinterpret_cast<char*>(p) + off); };
    w.perm = mine(w.perm); w.cand = mine(w.cand); w.fixed = mine(w.fixed);
    greedy_seq(table, nt, numel, QA_METRIC_ATOL, thresholds[k], ord, rng, mine(rng_out), assignment + k * nt, counts + k * QA_NFMT,
               state + k * 24, w);
}

// ------------------------------------------------------------------------------------------
// Threshold assignment (per tile, per threshold)
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) threshold_kernel(const float* __restrict__ scores, int64_t nt, OrderArg ord,
                                                        int is_pcc, const float* __restrict__ thr, int nthr,
                                                        int8_t* __restrict__ assignment,
                                                        unsigned long long* __restrict__ counts) {
    const int ti = blockIdx.y;
    const float th = thr[ti];
    unsigned int local[QA_NFMT] = {0, 0, 0, 0};
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < nt; t += (int64_t)gridDim.x * blockDim.x) {
        int pick = ord.fmt[ord.n - 1];
        for (int k = 0; k < ord.n; ++k) {
            const float s = scores[(int64_t)ord.fmt[k] * nt + t];
            const bool ok = is_pcc ? (s >= th) : (s <= th);   // float32 compare (NumPy 2 promotion)
            if (ok) { pick = ord.fmt[k]; break; }
        }
        assignment[(int64_t)ti * nt + t] = (int8_t)pick;
        ++local[pick];
    }
#pragma unroll
    for (int f = 0; f < QA_NFMT; ++f) {
        const unsigned int s = __reduce_add_sync(0xFFFFFFFFu, local[f]);
        if ((threadIdx.x & 31) == 0 && s) atomicAdd(&counts[(int64_t)ti * QA_NFMT + f], (unsigned long long)s);
    }
}

// ------------------------------------------------------------------------------------------
// Random assignment samples
// ------------------------------------------------------------------------------------------
constexpr int RB = 256;

__device__ __forceinline__ double block_sum(double v, double* sm) {
    // fixed-shape tree: deterministic for a given (ntiles, RB)
#pragma unroll
    for (int o = 16; o; o >>= 1)
        v += __hiloint2double(__shfl_xor_sync(0xFFFFFFFFu, __double2hiint(v), o),
                              __shfl_xor_sync(0xFFFFFFFFu, __double2loint(v), o));
    __syncthreads();
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = v;
    __syncthreads();
    double r = 0.0;
    for (int i = 0; i < RB / 32; ++i) r += sm[i];
    return r;
}

struct FmtIdxArg {
    int32_t idx[QA_NFMT];
    int n;
};

// one block per sample.  choice(s, t) is the (s*nt + t)-th bounded draw of the stream when k is
// a power of two (no rejection): each thread jumps the LCG to its contiguous tile range.
__global__ void __launch_bounds__(RB) random_samples_kernel(const double* __restrict__ table, int64_t nt, double numel,
                                                            FmtIdxArg fi, const qa_pcg64* __restrict__ rng,
                                                            int8_t* __restrict__ choices, int choices_ready,
                                                            double* __restrict__ metrics,
                                                            unsigned long long* __restrict__ counts) {
    __shared__ double sm[RB / 32];
    const int s = blockIdx.x;
    const int64_t per = cdiv(nt, (int64_t)RB);
    const int64_t t0 = min(nt, (int64_t)threadIdx.x * per), t1 = min(nt, t0 + per);
    double sy = 0.0, sy2 = 0.0, sxy = 0.0, sab = 0.0, amax = 0.0, sx = 0.0, sx2 = 0.0;
    unsigned int cnt[QA_NFMT] = {0, 0, 0, 0};
    Pcg g;
    const uint32_t k = (uint32_t)fi.n;
    const int shift = k == 4 ? 30 : k == 2 ? 31 : 32;
    if (!choices_ready && k > 1 && t0 < t1) {
        g.load(rng);
        // position of draw q = s*nt + t0 in the 32-bit stream
        uint64_t q = (uint64_t)s * (uint64_t)nt + (uint64_t)t0;
        if (g.has32) {
            if (q == 0) { /* first draw is the buffered half */ }
            else { q -= 1; g.has32 = 0; g.advance(q >> 1); if (q & 1ull) { const uint64_t v = g.next64(); g.has32 = 1; g.buf32 = (uint32_t)(v >> 32); } }
        } else {
            g.advance(q >> 1);
            if (q & 1ull) { const uint64_t v = g.next64(); g.has32 = 1; g.buf32 = (uint32_t)(v >> 32); }
        }
    }
    for (int64_t t = t0; t < t1; ++t) {
        int c;
        if (choices_ready) c = choices[(int64_t)s * nt + t];
        else {
            const uint32_t ci = k > 1 ? (g.next32() >> shift) : 0u;
            c = fi.idx[ci];
            choices[(int64_t)s * nt + t] = (int8_t)c;
        }
        ++cnt[c];
        sx += table[QA_STAT_SX * nt + t];
        sx2 += table[QA_STAT_SX2 * nt + t];
        sy += table[QA_STAT_FMT(c, 0) * nt + t];
        sy2 += table[QA_STAT_FMT(c, 1) * nt + t];
        sxy += table[QA_STAT_FMT(c, 2) * nt + t];
        sab += table[QA_STAT_FMT(c, 3) * nt + t];
        amax = fmax(amax, table[QA_STAT_FMT(c, 4) * nt + t]);
    }
    sx = block_sum(sx, sm); sx2 = block_sum(sx2, sm);
    sy = block_sum(sy, sm); sy2 = block_sum(sy2, sm); sxy = block_sum(sxy, sm); sab = block_sum(sab, sm);
#pragma unroll
    for (int o = 16; o; o >>= 1)
        amax = fmax(amax, __hiloint2double(__shfl_xor_sync(0xFFFFFFFFu, __double2hiint(amax), o),
                                           __shfl_xor_sync(0xFFFFFFFFu, __double2loint(amax), o)));
    __syncthreads();
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = amax;
    __syncthreads();
    amax = 0.0;
    for (int i = 0; i < RB / 32; ++i) amax = fmax(amax, sm[i]);
#pragma unroll
    for (int f = 0; f < QA_NFMT; ++f) {
        const unsigned int c = __reduce_add_sync(0xFFFFFFFFu, cnt[f]);
        if ((threadIdx.x & 31) == 0 && c) atomicAdd(&counts[(int64_t)s * QA_NFMT + f], (unsigned long long)c);
    }
    if (threadIdx.x == 0) {
        double pcc;
        const double am2 = fmax(sx2 - sx * sx / numel, 0.0), bm2 = fmax(sy2 - sy * sy / numel, 0.0);
        const double den = sqrt(am2 * bm2);
        if (den == 0.0) pcc = amax == 0.0 ? 1.0 : 0.0;
        else pcc = (sxy - sx * sy / numel) / den;
        metrics[s * 3 + 0] = pcc;
        metrics[s * 3 + 1] = sab / numel;
        metrics[s * 3 + 2] = amax;
    }
}

// advance *rng past `draws` 32-bit draws (after the sample kernel consumed them by jumping)
__global__ void rng_skip32_kernel(qa_pcg64* rng, uint64_t draws) {
    if (blockIdx.x || threadIdx.x || draws == 0) return;
    Pcg g;
    g.load(rng);
    uint64_t q = draws;
    if (g.has32) { g.has32 = 0; q -= 1; }
    g.advance(q >> 1);
    if (q & 1ull) { const uint64_t v = g.next64(); g.has32 = 1; g.buf32 = (uint32_t)(v >> 32); }
    g.store(rng);
}

// ------------------------------------------------------------------------------------------
// Whole-tensor sums for one assignment / one format (fixed reduction shape)
// ------------------------------------------------------------------------------------------
constexpr int SB = 1024;
__global__ void __launch_bounds__(SB) assignment_sums_kernel(const double* __restrict__ table, int64_t nt,
                                                             const int8_t* __restrict__ assignment, int fmt,
                                                             double* __restrict__ out) {
    // one block per assignment map: block b reduces map b (maps are [gridDim.x][nt]) into out[b][8]
    if (assignment) assignment += (int64_t)blockIdx.x * nt;
    out += (int64_t)blockIdx.x * 8;
    __shared__ double sm[7][SB / 32];
    double v[7] = {0, 0, 0, 0, 0, 0, 0};
    // thread t takes tiles t, t + SB, ...: coalesced column reads, and a fixed (deterministic) summation shape
#pragma unroll 2
    for (int64_t t = threadIdx.x; t < nt; t += SB) {
        int c = assignment ? (int)assignment[t] : fmt;
        v[0] += table[QA_STAT_SX * nt + t];
        v[1] += table[QA_STAT_SX2 * nt + t];
        if (c >= 0) {
            v[2] += table[QA_STAT_FMT(c, 0) * nt + t];
            v[3] += table[QA_STAT_FMT(c, 1) * nt + t];
            v[4] += table[QA_STAT_FMT(c, 2) * nt + t];
            v[5] += table[QA_STAT_FMT(c, 3) * nt + t];
            v[6] = fmax(v[6], table[QA_STAT_FMT(c, 4) * nt + t]);
        } else {  // "none": y == x
            v[2] += table[QA_STAT_SX * nt + t];
            v[3] += table[QA_STAT_SX2 * nt + t];
            v[4] += table[QA_STAT_SX2 * nt + t];
        }
    }
#pragma unroll
    for (int i = 0; i < 7; ++i) {
#pragma unroll
        for (int o = 16; o; o >>= 1) {
            const double other = __hiloint2double(__shfl_xor_sync(0xFFFFFFFFu, __double2hiint(v[i]), o),
                                                  __shfl_xor_sync(0xFFFFFFFFu, __double2loint(v[i]), o));
            v[i] = i == 6 ? fmax(v[i], other) : v[i] + other;
        }
        if ((threadIdx.x & 31) == 0) sm[i][threadIdx.x >> 5] = v[i];
    }
    __syncthreads();
    if (threadIdx.x < 7) {
        double r = 0.0;
        for (int w = 0; w < SB / 32; ++w) r = threadIdx.x == 6 ? fmax(r, sm[threadIdx.x][w]) : r + sm[threadIdx.x][w];
        out[threadIdx.x] = r;
    }
    if (threadIdx.x == 7) out[7] = 0.0;
}

// ------------------------------------------------------------------------------------------
// Whole-array pair sums for metrics.py (pearson_corr / metric_value on arbitrary float32 arrays)
// ------------------------------------------------------------------------------------------
constexpr int PS_BLOCKS = 592, PS_THREADS = 256;
__global__ void __launch_bounds__(PS_THREADS) pair_sums_kernel(const float* __restrict__ a, const float* __restrict__ b,
                                                               int64_t n, double* __restrict__ partial) {
    __shared__ double sm[7][PS_THREADS / 32];
    double v[7] = {0, 0, 0, 0, 0, 0, 0};
    const int64_t per = cdiv(n, (int64_t)gridDim.x * blockDim.x);
    const int64_t i0 = min(n, ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * per), i1 = min(n, i0 + per);
    for (int64_t i = i0; i < i1; ++i) {         // fixed element ranges and a fixed tree: deterministic
        const double x = (double)a[i], y = b ? (double)b[i] : 0.0;
        const double d = fabs((double)__fsub_rn(a[i], b ? b[i] : 0.f));     // float32 difference, as the reference forms it
        v[0] += x; v[1] = fma(x, x, v[1]); v[2] += y; v[3] = fma(y, y, v[3]); v[4] = fma(x, y, v[4]); v[5] += d;
        v[6] = fmax(v[6], d);
    }
#pragma unroll
    for (int k = 0; k < 7; ++k) {
#pragma unroll
        for (int o = 16; o; o >>= 1) {
            const double other = __hiloint2double(__shfl_xor_sync(0xFFFFFFFFu, __double2hiint(v[k]), o),
                                                  __shfl_xor_sync(0xFFFFFFFFu, __double2loint(v[k]), o));
            v[k] = k == 6 ? fmax(v[k], other) : v[k] + other;
        }
        if ((threadIdx.x & 31) == 0) sm[k][threadIdx.x >> 5] = v[k];
    }
    __syncthreads();
    if (threadIdx.x < 7) {
        double r = 0.0;
        for (int w = 0; w < PS_THREADS / 32; ++w) r = threadIdx.x == 6 ? fmax(r, sm[threadIdx.x][w]) : r + sm[threadIdx.x][w];
        partial[(int64_t)blockIdx.x * 8 + threadIdx.x] = r;
    }
}
__global__ void pair_sums_final_kernel(const double* __restrict__ partial, int nblocks, double* __restrict__ out) {
    const int k = threadIdx.x;
    if (k >= 8) return;
    double r = 0.0;
    if (k < 7)
        for (int b = 0; b < nblocks; ++b) r = k == 6 ? fmax(r, partial[(int64_t)b * 8 + k]) : r + partial[(int64_t)b * 8 + k];
    out[k] = r;
}

}  // namespace qa

using namespace qa;

extern "C" int64_t qa_pair_sums_work_bytes(void) { return (int64_t)PS_BLOCKS * 8 * sizeof(double); }

extern "C" int qa_pair_sums(const float* a, const float* b, int64_t n, double* out, void* work, qa_stream_t stream) {
    if (!a || n < 0 || !out || !work) { set_error("qa_pair_sums: bad args"); return 1; }
    cudaStream_t s = (cudaStream_t)stream;
    pair_sums_kernel<<<PS_BLOCKS, PS_THREADS, 0, s>>>(a, b, n, reinterpret_cast<double*>(work));
    pair_sums_final_kernel<<<1, 32, 0, s>>>(reinterpret_cast<const double*>(work), PS_BLOCKS, out);
    return check_launch("qa_pair_sums");
}

extern "C" int qa_numpy_permutation(qa_pcg64* rng, int64_t n, int32_t* out_perm, int32_t* work, qa_stream_t stream) {
    (void)work;
    if (!rng || n < 0 || (n > 0 && !out_perm)) { set_error("qa_numpy_permutation: bad args"); return 1; }
    if (n > 0xFFFFFFFFll) { set_error("qa_numpy_permutation: n too large"); return 1; }
    if (n == 0) return 0;
    permutation_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(rng, n, out_perm);
    return check_launch("qa_numpy_permutation");
}

extern "C" int qa_numpy_integers(qa_pcg64* rng, int k, int64_t n, int8_t* out_vals, qa_stream_t stream) {
    if (!rng || n < 0 || k < 1 || k > 127) { set_error("qa_numpy_integers: bad args"); return 1; }
    if (n == 0) return 0;
    integers_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(rng, (uint32_t)k, n, out_vals);
    return check_launch("qa_numpy_integers");
}

static inline int64_t align_up(int64_t v, int64_t a) { return (v + a - 1) / a * a; }

static GreedyWork carve_seq(void* work, int64_t ntiles) {
    GreedyWork w;
    char* p = reinterpret_cast<char*>(work);
    w.perm = reinterpret_cast<int32_t*>(p); p += align_up(ntiles * 4, 256);
    w.cand = reinterpret_cast<int32_t*>(p); p += align_up(ntiles * 4, 256);
    w.fixed = reinterpret_cast<uint8_t*>(p);
    return w;
}

extern "C" int64_t qa_greedy_work_bytes(int64_t ntiles) {
    return align_up(ntiles * 4, 256) * 2 + align_up(ntiles, 256) + 256;
}

extern "C" int qa_greedy_assign(const double* table, int64_t ntiles, double numel, int metric,
                                double threshold, const int32_t* fmt_order, int nfmt, qa_pcg64* rng,
                                int8_t* assignment, int64_t* counts, double* state, void* work,
                                qa_stream_t stream) {
    if (!table || ntiles <= 0 || !fmt_order || nfmt < 1 || nfmt > QA_NFMT || !rng || !assignment || !counts || !state || !work) {
        set_error("qa_greedy_assign: bad args");
        return 1;
    }
    if (metric < 0 || metric > 2) { set_error("qa_greedy_assign: bad metric"); return 1; }
    OrderArg ord;
    ord.n = nfmt;
    for (int i = 0; i < QA_NFMT; ++i) ord.fmt[i] = i < nfmt ? fmt_order[i] : 0;  // HOST array
    for (int i = 0; i < nfmt; ++i)
        if (ord.fmt[i] < 0 || ord.fmt[i] >= QA_NFMT) { set_error("qa_greedy_assign: bad format index"); return 1; }
    greedy_seq_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(table, ntiles, numel, metric, threshold, ord, rng,
                                                          assignment, counts, state, carve_seq(work, ntiles));
    return check_launch("qa_greedy_assign");
}

int qa::greedy_seq_sweep_launch(const double* table, int64_t ntiles, double numel, const double* thresholds, int nthr,
                                const int32_t* fmt_order, int nfmt, const qa_pcg64* rng, qa_pcg64* rng_out, int8_t* assignment,
                                int64_t* counts, double* state, void* work, int64_t stride, cudaStream_t stream) {
    OrderArg ord;       // fmt_order: checked by the caller
    ord.n = nfmt;
    for (int i = 0; i < QA_NFMT; ++i) ord.fmt[i] = i < nfmt ? fmt_order[i] : 0;
    greedy_seq_sweep_kernel<<<(unsigned)nthr, 32, 0, stream>>>(table, ntiles, numel, thresholds, ord, rng, rng_out, assignment, counts,
                                                               state, carve_seq(work, ntiles), stride);
    return check_launch("qa_greedy_assign_sweep");
}

extern "C" int qa_threshold_assign(const float* scores, int64_t ntiles, const int32_t* order, int norder,
                                   int is_pcc, const float* thresholds, int nthr, int8_t* assignment,
                                   int64_t* counts, qa_stream_t stream) {
    if (!scores || ntiles <= 0 || !order || norder < 1 || norder > QA_NFMT || !thresholds || nthr < 1 || !assignment || !counts) {
        set_error("qa_threshold_assign: bad args");
        return 1;
    }
    OrderArg o;
    o.n = norder;
    for (int i = 0; i < QA_NFMT; ++i) o.fmt[i] = i < norder ? order[i] : 0;  // `order` is a HOST array
    for (int i = 0; i < norder; ++i)
        if (o.fmt[i] < 0 || o.fmt[i] >= QA_NFMT) { set_error("qa_threshold_assign: bad format index"); return 1; }
    cudaStream_t s = (cudaStream_t)stream;
    cudaMemsetAsync(counts, 0, sizeof(int64_t) * QA_NFMT * nthr, s);
    int gx = (int)min((int64_t)148 * 4, cdiv(ntiles, 256));
    // one threshold per gridDim.y index, which CUDA caps at 65535: launch over threshold ranges of at most that many
    constexpr int max_y = 65535;
    for (int t0 = 0; t0 < nthr; t0 += max_y) {
        const int nt = min(nthr - t0, max_y);
        threshold_kernel<<<dim3(gx > 0 ? gx : 1, nt), 256, 0, s>>>(scores, ntiles, o, is_pcc, thresholds + t0, nt,
                                                                  assignment + (int64_t)t0 * ntiles,
                                                                  reinterpret_cast<unsigned long long*>(counts + (int64_t)t0 * QA_NFMT));
    }
    return check_launch("qa_threshold_assign");
}

extern "C" int qa_random_samples(const double* table, int64_t ntiles, double numel, const int32_t* fmt_indices,
                                 int nfmt, int iters, qa_pcg64* rng, int8_t* choices, int choices_ready,
                                 double* sample_metrics, int64_t* sample_counts, qa_stream_t stream) {
    if (!table || ntiles <= 0 || !fmt_indices || nfmt < 1 || nfmt > QA_NFMT || iters < 1 || !rng || !choices || !sample_metrics || !sample_counts) {
        set_error("qa_random_samples: bad args");
        return 1;
    }
    if (!choices_ready && nfmt == 3) { set_error("qa_random_samples: nfmt == 3 needs pre-drawn choices (rejection sampling)"); return 1; }
    FmtIdxArg fi;
    fi.n = nfmt;
    for (int i = 0; i < QA_NFMT; ++i) fi.idx[i] = i < nfmt ? fmt_indices[i] : 0;  // HOST array
    cudaStream_t s = (cudaStream_t)stream;
    cudaMemsetAsync(sample_counts, 0, sizeof(int64_t) * QA_NFMT * iters, s);
    random_samples_kernel<<<iters, RB, 0, s>>>(table, ntiles, numel, fi, rng, choices, choices_ready, sample_metrics,
                                               reinterpret_cast<unsigned long long*>(sample_counts));
    int rc = check_launch("qa_random_samples");
    if (rc) return rc;
    if (!choices_ready && nfmt > 1) {
        rng_skip32_kernel<<<1, 32, 0, s>>>(rng, (uint64_t)iters * (uint64_t)ntiles);
        rc = check_launch("qa_random_samples(skip)");
    }
    return rc;
}

extern "C" int qa_assignment_sums_batch(const double* table, int64_t ntiles, const int8_t* maps, int nmaps, double* out,
                                        qa_stream_t stream) {
    if (!table || ntiles <= 0 || !maps || nmaps < 0 || (nmaps > 0 && !out)) { set_error("qa_assignment_sums_batch: bad args"); return 1; }
    if (nmaps == 0) return 0;
    assignment_sums_kernel<<<(unsigned)nmaps, SB, 0, (cudaStream_t)stream>>>(table, ntiles, maps, -1, out);
    return check_launch("qa_assignment_sums_batch");
}

extern "C" int qa_assignment_sums(const double* table, int64_t ntiles, const int8_t* assignment, int fmt,
                                  double* out, qa_stream_t stream) {
    if (!table || ntiles <= 0 || !out || (!assignment && fmt >= QA_NFMT)) { set_error("qa_assignment_sums: bad args"); return 1; }
    assignment_sums_kernel<<<1, SB, 0, (cudaStream_t)stream>>>(table, ntiles, assignment, fmt, out);
    return check_launch("qa_assignment_sums");
}
