// Parallel, bit-faithful greedy assignment: one thread-block CLUSTER per tensor.
//
// The reference's greedy (mixed_tile_greedy.py:135-346) is three sequential chains:
//   (1) sequential float64 accumulation of the per-tile sums in tile order            (:165-170)
//   (2) numpy Generator.permutation of the candidate tiles, once per format           (:228-231)
//   (3) the accept/reject chain: cand = S + (new - old); accept iff metric(cand) passes (:234-346)
// All three are reproduced with the results of a one-thread loop, in parallel, by up to 16 CTAs
// of a cluster that exchange scan totals through distributed shared memory:
//
//  * Sequentially rounded float64 sums.  While a running sum S stays in one binade its ulp q is
//    fixed and S is an integer multiple m*q; adding t = (a + f)*q (a integer, 0 <= f < 1) gives
//    m + a rounded to nearest - up if f > 1/2, down if f < 1/2, and to the even neighbour if
//    f == 1/2.  The increment depends on the running state only through the parity of m at exact
//    ties, so a chunk of additions composes as pairs (increment if m even, increment if m odd):
//    an associative operator, i.e. a prefix scan over int64 pairs.  The first element that leaves
//    the binade [2^52, 2^53) q is itself still exact (it is a real float64 add from the exact
//    state before it); the chunk is cut after it and the next chunk starts with the new ulp.
//  * Decisions.  Within a chunk the accept flags F are guessed, the exact states before every
//    element follow from the masked scan, every decision D is re-evaluated in parallel with the
//    reference's float64 formula (behind an error-bounded multiplication-only filter), and F is
//    corrected from the first mismatch on; the fixed point is the sequential result.
//  * numpy permutation.  The 32-bit draw stream of PCG64 is generated in parallel by jumping the
//    LCG; the masked-rejection acceptance (draw & mask(i) <= i, i decreasing with every accept) is
//    a fixed point of  c = prefix_sum(accepts(c))  over per-thread accept counts; the Fisher-Yates
//    swap sequence is then applied in parallel by following, for every step, the chain of earlier
//    steps that last wrote the position it reads.
#include <cooperative_groups.h>

#include <cstdio>

#include <mutex>

#include "qa_common.cuh"

namespace cg = cooperative_groups;

namespace qa {

constexpr int GT = 256;           // threads per CTA
constexpr int NW = GT / 32;
constexpr int MAXR = 16;          // largest cluster
constexpr int DPT = 8;            // draws per thread per round (4 LCG outputs)
constexpr int EPS = 8;           // elements each thread streams through per chunk (scan works on thread totals)
constexpr int SEQ_TAIL = 96;      // last Fisher-Yates steps are drawn by one thread
constexpr long long M_LO = 1ll << 52, M_HI = 1ll << 53;

// Diagnostic timeline: first-start / last-end device timestamps (ns, %globaltimer) of the cluster kernels of this file,
// read back with qa_debug_times.  Slots: 0/1 resolve chain, 2/3 init sums, 4/5 chain launch with pass 0, 6/7 later launch.
// One row of 8 per cluster-size class (log2 of the cluster size, 0..4), so tensors of different sizes can be told apart.
// Diagnostic only: compiled in with -DQA_STAMP_TIMES (profiles/step_variants.py); the shipped library does no global
// atomics of its own in these kernels and qa_debug_times reports "not compiled in".
__device__ unsigned long long qa_times[5 * 8];
__device__ __forceinline__ void stamp(int slot, bool is_end) {
#ifndef QA_STAMP_TIMES
    (void)slot; (void)is_end;
    return;
#endif
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    unsigned nr;
    asm volatile("mov.u32 %0, %%cluster_nctaid.x;" : "=r"(nr));
    const int cls = 31 - __clz((int)(nr | 1u));
    if (is_end) atomicMax(&qa_times[cls * 8 + slot], t);
    else atomicMin(&qa_times[cls * 8 + slot], t);
}

struct ParOrder {
    int32_t fmt[QA_NFMT];
    int n;
};

struct ParWork {
    int32_t* order;   // [n]  candidates in visiting order
    int32_t* cand;    // [n]
    int32_t* jarr;    // [n]
    int32_t* off;     // [n+1]
    int32_t* cursor;  // [n]
    int32_t* bucket;  // [n]
    int32_t* succ;    // [n]
    int32_t* parent;  // [n]
    double* hdr;      // [32]    initial sums + diagnostics (greedy_init_kernel)
    double* res;      // [32]    running state handed from one launch of the chain to the next (pass ranges)
    double* delta;    // [3][n][4] per-tile deltas {sy, sy2, sxy, sabs} of the format transitions, tile order
    uint8_t* fixed;   // [n]
    const int32_t* pre_order;   // optional: permutations #2 (and #3) of n items, drawn ahead (qa_perm_resolve[_chain] + qa_perm_apply)
    const qa_pcg64* pre_rng;    //           and the stream states after permutation #2 (and #3)
    int npre;                   // how many permutations were drawn ahead (0, 2 or 3)
};
constexpr int HDR_DOUBLES = 32;
#ifdef QA_DBG_CHAIN
#define QA_PHASE_SYNC() __syncthreads()
#else
#define QA_PHASE_SYNC()
#endif

struct P2 {          // increment of m if the incoming m is even / odd
    long long d0, d1;
};

struct Sh {
    int i32[3 * NW + 8];
    long long i64[NW * 4 * 2 * 2 + 16];
    double f64[16];
    // cluster exchange (double buffered; written by remote CTAs through DSMEM)
    int xi[2][MAXR];
    long long xl[2][MAXR][12];
    double xd[2][MAXR];
    int cnt[QA_NFMT];
    unsigned tail_draws[256];    // permutation tail: one batch of 32-bit draws
    unsigned long long mbar;     // cluster exchange barrier: one arrival per CTA per exchange
};

struct Coop {
    Sh& sh;
    cg::cluster_group cl;
    unsigned rank, nr;
    int gtid, gth;       // cluster-wide thread id / thread count
    unsigned par;        // exchange counter (uniform): low bit = payload buffer and mbarrier phase parity
    long long cy_resolve = 0, cy_apply = 0; unsigned n_sweeps = 0, n_rounds = 0;   // diagnostics
    long long cy_i0 = 0, cy_i1 = 0, cy_i2 = 0; unsigned n_init_rounds = 0;
    __device__ Coop(Sh& s) : sh(s), cl(cg::this_cluster()) {
        rank = cl.block_rank();
        nr = cl.num_blocks();
        gtid = (int)rank * GT + (int)threadIdx.x;
        gth = (int)nr * GT;
        par = 0;
        if (nr > 1) {
            if (threadIdx.x == 0) {
                const uint32_t a = (uint32_t)__cvta_generic_to_shared(&sh.mbar);
                asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(a), "r"(nr));
                asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
            }
            cl.sync();
        }
    }
    // full cluster barrier (global-memory phases): orders global writes and invalidates L1
    __device__ __forceinline__ void sync() {
        __syncthreads();                 // every thread's writes happen-before the arrivals below (cumulativity)
        if (nr > 1) xarrive_wait();      // release / acquire at cluster scope; ~10x cheaper than barrier.cluster here
    }
    // Payload exchange barrier.  Call pattern inside a collective: thread r (r < nr) has just stored this
    // CTA's payload into CTA r's buffer `par & 1`; it then arrives on CTA r's mbarrier (release, cluster
    // scope), and every thread waits until all nr CTAs have arrived on the local one (acquire).  About an
    // order of magnitude cheaper than barrier.cluster with 16 x 512 threads.
    __device__ __forceinline__ void xarrive_wait() {
        const uint32_t local = (uint32_t)__cvta_generic_to_shared(&sh.mbar);
        if (threadIdx.x < nr) {
            uint32_t remote;
            asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(local), "r"(threadIdx.x));
            asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(remote) : "memory");
        }
        const uint32_t parity = par & 1u;
        uint32_t done = 0;
        while (!done) {
            asm volatile(
                "{\n\t.reg .pred p;\n\t"
                "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
                "selp.u32 %0, 1, 0, p;\n\t}"
                : "=r"(done)
                : "r"(local), "r"(parity)
                : "memory");
        }
        ++par;
    }
};

// ---------------------------------------------------------------------------------------------
// block / cluster collectives (every thread of the cluster calls them, values come back uniform)
// ---------------------------------------------------------------------------------------------
// warp-level helpers over a small array held one entry per lane
__device__ __forceinline__ int lanes_incl_scan(int x) {
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int y = __shfl_up_sync(0xFFFFFFFFu, x, o);
        if (lane >= o) x += y;
    }
    return x;
}

__device__ __forceinline__ int block_scan_excl(int v, int& total, Sh& sh) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int inc = lanes_incl_scan(v);
    if (lane == 31) sh.i32[w] = inc;
    __syncthreads();
    // every warp scans the NW warp totals itself (one entry per lane)
    const int wt = lanes_incl_scan(lane < NW ? sh.i32[lane] : 0);
    total = __shfl_sync(0xFFFFFFFFu, wt, NW - 1);
    const int before = __shfl_sync(0xFFFFFFFFu, wt, (w + 31) & 31);     // inclusive total of warp w-1
    __syncthreads();
    return (w ? before : 0) + inc - v;
}

// exchange of one int per CTA; returns (sum over CTAs before this one, sum over all); entries read one per lane
__device__ __forceinline__ void xchg_prefix(Coop& c, int mine, int& base, int& total) {
    const unsigned b = c.par & 1u;
    if (threadIdx.x < c.nr) *c.cl.map_shared_rank(&c.sh.xi[b][c.rank], threadIdx.x) = mine;
    c.xarrive_wait();
    const int lane = threadIdx.x & 31;
    const int sc = lanes_incl_scan(lane < (int)c.nr ? c.sh.xi[b][lane] : 0);
    total = __shfl_sync(0xFFFFFFFFu, sc, c.nr - 1);
    const int before = __shfl_sync(0xFFFFFFFFu, sc, (c.rank + 31) & 31);
    base = c.rank ? before : 0;
}

__device__ __forceinline__ int c_scan_excl(Coop& c, int v, int& total) {
    int bt;
    const int ex = block_scan_excl(v, bt, c.sh);
    if (c.nr == 1) { total = bt; return ex; }
    int base;
    xchg_prefix(c, bt, base, total);
    return base + ex;
}

// exclusive scan of v together with an OR-reduction of `flag`, one exchange (flag rides in bit 30 of the CTA total)
__device__ __forceinline__ int c_scan_excl_any(Coop& c, int v, int& total, bool flag, bool& any) {
    int bt;
    const int blk = __syncthreads_or(flag ? 1 : 0);
    const int ex = block_scan_excl(v, bt, c.sh);
    if (c.nr == 1) { total = bt; any = blk != 0; return ex; }
    const unsigned b = c.par & 1u;
    if (threadIdx.x < c.nr) {
        int* dst = c.cl.map_shared_rank(&c.sh.xi[b][c.rank], threadIdx.x);
        *dst = bt | (blk ? (1 << 30) : 0);
    }
    c.xarrive_wait();
    const int lane = threadIdx.x & 31;
    const int raw = lane < (int)c.nr ? c.sh.xi[b][lane] : 0;
    any = __any_sync(0xFFFFFFFFu, (raw >> 30) & 1);
    const int sc = lanes_incl_scan(raw & ~(1 << 30));
    total = __shfl_sync(0xFFFFFFFFu, sc, c.nr - 1);
    const int before = __shfl_sync(0xFFFFFFFFu, sc, (c.rank + 31) & 31);
    return (c.rank ? before : 0) + ex;
}

__device__ __forceinline__ int c_min(Coop& c, int v) {
    const int lane = threadIdx.x & 31;
    v = __reduce_min_sync(0xFFFFFFFFu, v);
    if (lane == 0) c.sh.i32[threadIdx.x >> 5] = v;
    __syncthreads();
    int r = __reduce_min_sync(0xFFFFFFFFu, lane < NW ? c.sh.i32[lane] : 0x7FFFFFFF);
    __syncthreads();
    if (c.nr == 1) return r;
    const unsigned b = c.par & 1u;
    if (threadIdx.x < c.nr) *c.cl.map_shared_rank(&c.sh.xi[b][c.rank], threadIdx.x) = r;
    c.xarrive_wait();
    return __reduce_min_sync(0xFFFFFFFFu, lane < (int)c.nr ? c.sh.xi[b][lane] : 0x7FFFFFFF);
}

__device__ __forceinline__ bool c_any(Coop& c, bool p) {
    const int blk = __syncthreads_or(p ? 1 : 0);
    if (c.nr == 1) return blk != 0;
    const unsigned b = c.par & 1u;
    if (threadIdx.x < c.nr) *c.cl.map_shared_rank(&c.sh.xi[b][c.rank], threadIdx.x) = blk;
    c.xarrive_wait();
    const int lane = threadIdx.x & 31;
    return __any_sync(0xFFFFFFFFu, lane < (int)c.nr ? c.sh.xi[b][lane] : 0);
}

// deterministic cluster-wide float64 sum / max (fixed tree: lanes, warps in order, CTAs in order)
template <bool MAX>
__device__ __forceinline__ double c_reduce_d(Coop& c, double v) {
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        const double y = __hiloint2double(__shfl_xor_sync(0xFFFFFFFFu, __double2hiint(v), o),
                                          __shfl_xor_sync(0xFFFFFFFFu, __double2loint(v), o));
        v = MAX ? fmax(v, y) : v + y;
    }
    if ((threadIdx.x & 31) == 0) c.sh.i64[threadIdx.x >> 5] = __double_as_longlong(v);
    __syncthreads();
    double r = __longlong_as_double(c.sh.i64[0]);
    for (int i = 1; i < NW; ++i) {
        const double y = __longlong_as_double(c.sh.i64[i]);
        r = MAX ? fmax(r, y) : r + y;
    }
    __syncthreads();
    if (c.nr == 1) return r;
    const unsigned b = c.par & 1u;
    if (threadIdx.x < c.nr) *c.cl.map_shared_rank(&c.sh.xd[b][c.rank], threadIdx.x) = r;
    c.xarrive_wait();
    double t = c.sh.xd[b][0];
    for (unsigned q = 1; q < c.nr; ++q) t = MAX ? fmax(t, c.sh.xd[b][q]) : t + c.sh.xd[b][q];
    return t;
}

// c_reduce_d<false> for NV values at once: the same fixed tree per value (lanes, warps in order, CTAs in order), one
// pair of CTA barriers and one exchange for all of them
template <int NV>
__device__ __forceinline__ void c_reduce_sum_multi(Coop& c, double (&v)[NV]) {
    static_assert(NV <= 12 && NW * NV <= NW * 4 * 2 * 2, "payload / staging slots");
#pragma unroll
    for (int k = 0; k < NV; ++k) {
#pragma unroll
        for (int o = 16; o; o >>= 1)
            v[k] = v[k] + __hiloint2double(__shfl_xor_sync(0xFFFFFFFFu, __double2hiint(v[k]), o),
                                           __shfl_xor_sync(0xFFFFFFFFu, __double2loint(v[k]), o));
        if ((threadIdx.x & 31) == 0) c.sh.i64[(threadIdx.x >> 5) * NV + k] = __double_as_longlong(v[k]);
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < NV; ++k) {
        double r = __longlong_as_double(c.sh.i64[k]);
        for (int i = 1; i < NW; ++i) r = r + __longlong_as_double(c.sh.i64[i * NV + k]);
        v[k] = r;
    }
    __syncthreads();
    if (c.nr == 1) return;
    const unsigned b = c.par & 1u;
    if (threadIdx.x < c.nr) {
        long long* dst = c.cl.map_shared_rank(&c.sh.xl[b][c.rank][0], threadIdx.x);
#pragma unroll
        for (int k = 0; k < NV; ++k) dst[k] = __double_as_longlong(v[k]);
    }
    c.xarrive_wait();
#pragma unroll
    for (int k = 0; k < NV; ++k) {
        double t = __longlong_as_double(c.sh.xl[b][0][k]);
        for (unsigned q = 1; q < c.nr; ++q) t = t + __longlong_as_double(c.sh.xl[b][q][k]);
        v[k] = t;
    }
}

// One thread of the cluster (owner) publishes n <= 8 doubles to every CTA; all threads read them back.
__device__ __forceinline__ void c_bcast_d(Coop& c, bool owner, const double* vals, int n, double* out) {
    const unsigned b = c.par & 1u;
    if (owner) {
        for (unsigned r = 0; r < c.nr; ++r) {
            double* dst = c.nr == 1 ? &c.sh.xd[b][0] : c.cl.map_shared_rank(&c.sh.xd[b][0], r);
            for (int i = 0; i < n; ++i) dst[i] = vals[i];
        }
    }
    __syncthreads();                 // the owner's stores happen-before this CTA's arrivals below
    if (c.nr == 1) ++c.par;
    else c.xarrive_wait();
    for (int i = 0; i < n; ++i) out[i] = c.sh.xd[b][i];
}

// c_bcast_d plus a cluster-wide sum of one double per thread (CTA partials in rank order), one exchange
__device__ __forceinline__ double c_bcast_sum_d(Coop& c, bool owner, const double* vals, int n, double* out, double part) {
#pragma unroll
    for (int o = 16; o; o >>= 1)
        part += __hiloint2double(__shfl_xor_sync(0xFFFFFFFFu, __double2hiint(part), o),
                                 __shfl_xor_sync(0xFFFFFFFFu, __double2loint(part), o));
    if ((threadIdx.x & 31) == 0) c.sh.i64[threadIdx.x >> 5] = __double_as_longlong(part);
    const unsigned b = c.par & 1u;
    if (owner) {
        for (unsigned r = 0; r < c.nr; ++r) {
            double* dst = c.nr == 1 ? &c.sh.xd[b][0] : c.cl.map_shared_rank(&c.sh.xd[b][0], r);
            for (int i = 0; i < n; ++i) dst[i] = vals[i];
        }
    }
    __syncthreads();
    double blk = 0.0;
    for (int i = 0; i < NW; ++i) blk += __longlong_as_double(c.sh.i64[i]);
    double tot = blk;
    if (c.nr == 1) ++c.par;
    else {
        if (threadIdx.x < c.nr) *c.cl.map_shared_rank(&c.sh.xl[b][c.rank][0], threadIdx.x) = __double_as_longlong(blk);
        c.xarrive_wait();
        tot = 0.0;
        for (unsigned r = 0; r < c.nr; ++r) tot += __longlong_as_double(c.sh.xl[b][r][0]);
    }
    for (int i = 0; i < n; ++i) out[i] = c.sh.xd[b][i];
    __syncthreads();
    return tot;
}

// ---------------------------------------------------------------------------------------------
// sequentially-rounded float64 accumulation as a scan
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ P2 p2_then(P2 a, P2 b) {   // apply a, then b
    P2 r;
    r.d0 = a.d0 + ((a.d0 & 1ll) ? b.d1 : b.d0);
    r.d1 = a.d1 + (((1ll + a.d1) & 1ll) ? b.d1 : b.d0);
    return r;
}

struct Grid {        // binade of the running sum at the start of a chunk
    double q;        // ulp (power of two); 0 => no grid (S == 0, inf/nan or denormal range)
    double invq;
    double sinvq;    // sign / q: maps an addend to signed grid units
    long long m0;    // |S| / q, in [2^52, 2^53)   (relaxed: S / q, signed, |m0| < 2^52)
    double sign;     // +1 / -1
    bool relaxed;    // fixed coarser grid that cannot be left: accurate (<= 1 ulp of the bound) but not the
                     // reference's rounding sequence; used for a signed sum that would hop between binades
};
__device__ __forceinline__ Grid make_grid(double S) {
    Grid g;
    const int e = (int)((__double2hiint(S) >> 20) & 0x7FF);
    g.relaxed = false;
    if (e < 64 || e > 1900) { g.q = 0.0; g.invq = 0.0; g.sinvq = 0.0; g.m0 = 0; g.sign = 1.0; return g; }
    g.q = __hiloint2double((e - 52) << 20, 0);
    g.invq = __hiloint2double((1023 + 1023 + 52 - e) << 20, 0);
    g.sign = S < 0.0 ? -1.0 : 1.0;
    g.sinvq = g.sign * g.invq;
    g.m0 = __double2ll_rn(fabs(S) * g.invq);
    return g;
}
// grid of the binade above |S| + bound: every state reachable by adding terms of total magnitude <= bound stays on it
__device__ __forceinline__ Grid make_grid_relaxed(double S, double bound) {
    Grid g;
    const double top = 2.0 * (fabs(S) + bound);
    int e = (int)((__double2hiint(top) >> 20) & 0x7FF);
    if (e < 64) e = 64;
    g.relaxed = true;
    g.sign = 1.0;
    if (e > 1900) { g.q = 0.0; g.invq = 0.0; g.sinvq = 0.0; g.m0 = 0; return g; }
    g.q = __hiloint2double((e - 52) << 20, 0);
    g.invq = __hiloint2double((1023 + 1023 + 52 - e) << 20, 0);
    g.sinvq = g.invq;
    g.m0 = __double2ll_rn(S * g.invq);
    return g;
}
// true when S +/- bound provably stays inside the binade of S (no grid change possible)
__device__ __forceinline__ bool stays_in_binade(double S, double bound) {
    const double lo = fabs(S) - bound, hi = fabs(S) + bound;
    if (!(lo > 0.0)) return false;
    return ((__double2hiint(lo) >> 20) & 0x7FF) == ((__double2hiint(hi) >> 20) & 0x7FF);
}
// classify one addend: returns false when it cannot be expressed on the grid (caller cuts the chunk)
__device__ __forceinline__ bool classify(const Grid& g, double t, P2& out) {
    if (t == 0.0) { out = P2{0, 0}; return true; }      // adding zero never moves the sum
    if (g.q == 0.0) return false;
    const double v = t * g.sinvq;                       // exact scaling by a power of two
    if (fabs(v) < 2251799813685248.0) {                 // |v| < 2^51: round to nearest-even integer with the 1.5 * 2^52 trick
        const double M = 6755399441055744.0;
        const double r = __dadd_rn(v, M);               // ulp(r) == 1, M even: r - M = v rounded to nearest, ties to even
        const long long rn = __double_as_longlong(r) - __double_as_longlong(M);
        const double fr = __dsub_rn(v, __dsub_rn(r, M));   // exact, in [-1/2, 1/2]
        out.d0 = rn;                                    // incoming m even: the tie goes to the even increment
        out.d1 = rn;
        if (fabs(fr) == 0.5) out.d1 = rn + (fr > 0.0 ? 1ll : -1ll);   // incoming m odd: to the odd increment
        return true;
    }
    if (!(fabs(v) < 4.0e18)) return false;
    const double fl = floor(v);
    const long long a = __double2ll_rd(v);
    if (fabs(v) >= 4503599627370496.0) { out.d0 = a; out.d1 = a; return true; }   // already an integer
    const double h = fl + 0.5;                          // exact; the comparisons below are exact too
    if (v < h) { out.d0 = a; out.d1 = a; }
    else if (v > h) { out.d0 = a + 1; out.d1 = a + 1; }
    else { out.d0 = a + (a & 1ll); out.d1 = a + 1 - (a & 1ll); }   // tie: to the even neighbour
    return true;
}
__device__ __forceinline__ long long m_after(const Grid& g, P2 p) { return g.m0 + ((g.m0 & 1ll) ? p.d1 : p.d0); }
__device__ __forceinline__ bool in_binade(long long m) { return m >= M_LO && m < M_HI; }
__device__ __forceinline__ double s_of(const Grid& g, long long m) {
    // m in [2^52, 2^53) is its own float64 mantissa: exponent field 1075, no int -> float conversion needed
    const double md = in_binade(m) ? __longlong_as_double(m + (1074ll << 52)) : (double)m;
    return g.sign * (md * g.q);
}
__device__ __forceinline__ bool left_grid(const Grid& g, long long m) { return g.q != 0.0 && !g.relaxed && !in_binade(m); }

__device__ __forceinline__ P2 shfl_up_p2(P2 v, int o) {
    P2 y;
    y.d0 = __shfl_up_sync(0xFFFFFFFFu, v.d0, o);
    y.d1 = __shfl_up_sync(0xFFFFFFFFu, v.d1, o);
    return y;
}

__device__ __forceinline__ long long lanes_incl_scan64(long long x) {
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const long long y = __shfl_up_sync(0xFFFFFFFFu, x, o);
        if (lane >= o) x += y;
    }
    return x;
}

__device__ __forceinline__ P2 lanes_incl_scan_p2(P2 v, int width) {       // inclusive pair scan over lanes [0, width)
    const int lane = threadIdx.x & 31;
    for (int o = 1; o < width; o <<= 1) {
        const P2 y = shfl_up_p2(v, o);
        if (lane >= o) v = p2_then(y, v);
    }
    return v;
}

// Exclusive cluster-wide scan (cluster thread order) of one P2 per stream per thread.
//  level 1  every warp scans its 32 thread totals.  Exact ties (an addend that ends exactly half an ulp of the
//           running sum) make the increment depend on the parity of the incoming state; a warp without one has
//           d0 == d1 everywhere and scans plain int64 sums instead of pairs.
//  level 2  warp s (s < NS) scans the NW warp totals of stream s and sends the CTA total to every CTA of the cluster.
//  level 3  after the exchange, warp s scans the CTA totals and publishes, per warp, the prefix of everything before it.
// Levels 2 and 3 run on NS warps only (one stream each) while the others wait at the closing barrier: the redundant
// per-warp copies of those scans used to cost more issue slots than the walks they serve.
template <int NS>
__device__ __forceinline__ void scan_totals(Coop& c, const P2 (&tot)[NS], P2 (&pre)[NS]) {
    Sh& sh = c.sh;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    static_assert(NS <= 4 && NS <= NW, "one warp per stream");
    long long* wt = sh.i64;                       // [NW][NS][2] warp totals
    long long* wp = sh.i64 + NW * 4 * 2;          // [NW][NS][2] prefix of everything before warp w (cluster-wide)
    bool tie = false;
#pragma unroll
    for (int s = 0; s < NS; ++s) tie = tie || (tot[s].d0 != tot[s].d1);
    P2 inc[NS];
    if (!__any_sync(0xFFFFFFFFu, tie)) {
#pragma unroll
        for (int s = 0; s < NS; ++s) {
            const long long v = lanes_incl_scan64(tot[s].d0);
            inc[s] = P2{v, v};
        }
    } else {
#pragma unroll
        for (int s = 0; s < NS; ++s) inc[s] = lanes_incl_scan_p2(tot[s], 32);
    }
#pragma unroll
    for (int s = 0; s < NS; ++s)
        if (lane == 31) { wt[(w * NS + s) * 2] = inc[s].d0; wt[(w * NS + s) * 2 + 1] = inc[s].d1; }
    P2 lanes_before[NS];
#pragma unroll
    for (int s = 0; s < NS; ++s) {
        lanes_before[s] = shfl_up_p2(inc[s], 1);
        if (lane == 0) lanes_before[s] = P2{0, 0};
    }
    __syncthreads();
    const unsigned b = c.par & 1u;
    if (w < NS) {
        const int s = w;
        P2 t{0, 0};
        if (lane < NW) { t.d0 = wt[(lane * NS + s) * 2]; t.d1 = wt[(lane * NS + s) * 2 + 1]; }
        t = lanes_incl_scan_p2(t, NW);
        P2 before = shfl_up_p2(t, 1);             // everything in this CTA before warp `lane`
        if (lane == 0) before = P2{0, 0};
        P2 cp{0, 0};                              // everything in the cluster before this CTA
        if (c.nr > 1) {
            P2 all;
            all.d0 = __shfl_sync(0xFFFFFFFFu, t.d0, NW - 1);
            all.d1 = __shfl_sync(0xFFFFFFFFu, t.d1, NW - 1);
            if (lane < (int)c.nr) {
                long long* dst = c.cl.map_shared_rank(&sh.xl[b][c.rank][0], lane);
                dst[2 * s] = all.d0;
                dst[2 * s + 1] = all.d1;
            }
            // the NS payload warps meet, then warp 0 signals every CTA; all NS warps wait for the cluster's arrivals
            asm volatile("bar.sync 1, %0;" ::"r"(32 * NS) : "memory");
            const uint32_t local = (uint32_t)__cvta_generic_to_shared(&sh.mbar);
            if (threadIdx.x < c.nr) {
                uint32_t remote;
                asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(local), "r"(threadIdx.x));
                asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(remote) : "memory");
            }
            const uint32_t parity = c.par & 1u;
            uint32_t done = 0;
            while (!done) {
                asm volatile(
                    "{\n\t.reg .pred p;\n\t"
                    "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
                    "selp.u32 %0, 1, 0, p;\n\t}"
                    : "=r"(done)
                    : "r"(local), "r"(parity)
                    : "memory");
            }
            P2 u{0, 0};
            if (lane < (int)c.nr) { u.d0 = sh.xl[b][lane][2 * s]; u.d1 = sh.xl[b][lane][2 * s + 1]; }
            u = lanes_incl_scan_p2(u, MAXR);
            cp.d0 = __shfl_sync(0xFFFFFFFFu, u.d0, (c.rank + 31) & 31);
            cp.d1 = __shfl_sync(0xFFFFFFFFu, u.d1, (c.rank + 31) & 31);
            if (c.rank == 0) cp = P2{0, 0};
        }
        const P2 pw = p2_then(cp, before);
        if (lane < NW) { wp[(lane * NS + s) * 2] = pw.d0; wp[(lane * NS + s) * 2 + 1] = pw.d1; }
    }
    ++c.par;                                      // one exchange, counted by every thread
    __syncthreads();
#pragma unroll
    for (int s = 0; s < NS; ++s) {
        P2 pw;
        pw.d0 = wp[(w * NS + s) * 2];
        pw.d1 = wp[(w * NS + s) * 2 + 1];
        pre[s] = p2_then(pw, lanes_before[s]);
    }
}

// three cluster-wide minima in one exchange
__device__ __forceinline__ void c_min3(Coop& c, int& v0, int& v1, int& v2) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    v0 = __reduce_min_sync(0xFFFFFFFFu, v0);
    v1 = __reduce_min_sync(0xFFFFFFFFu, v1);
    v2 = __reduce_min_sync(0xFFFFFFFFu, v2);
    if (lane == 0) { c.sh.i32[w] = v0; c.sh.i32[NW + w] = v1; c.sh.i32[2 * NW + w] = v2; }
    __syncthreads();
    int r0 = __reduce_min_sync(0xFFFFFFFFu, lane < NW ? c.sh.i32[lane] : 0x7FFFFFFF);
    int r1 = __reduce_min_sync(0xFFFFFFFFu, lane < NW ? c.sh.i32[NW + lane] : 0x7FFFFFFF);
    int r2 = __reduce_min_sync(0xFFFFFFFFu, lane < NW ? c.sh.i32[2 * NW + lane] : 0x7FFFFFFF);
    __syncthreads();
    if (c.nr > 1) {
        const unsigned b = c.par & 1u;
        if (threadIdx.x < c.nr) {
            long long* dst = c.cl.map_shared_rank(&c.sh.xl[b][c.rank][0], threadIdx.x);
            dst[0] = r0; dst[1] = r1; dst[2] = r2;
        }
        c.xarrive_wait();
        const bool on = lane < (int)c.nr;
        r0 = __reduce_min_sync(0xFFFFFFFFu, on ? (int)c.sh.xl[b][lane][0] : 0x7FFFFFFF);
        r1 = __reduce_min_sync(0xFFFFFFFFu, on ? (int)c.sh.xl[b][lane][1] : 0x7FFFFFFF);
        r2 = __reduce_min_sync(0xFFFFFFFFu, on ? (int)c.sh.xl[b][lane][2] : 0x7FFFFFFF);
    }
    v0 = r0; v1 = r1; v2 = r2;
}

// Cluster-wide minimum of one int per thread together with NV doubles held by the (unique) thread that attains it:
// one exchange.  Every thread returns the minimum and the winner's values.
template <int NV>
__device__ __forceinline__ int c_argmin_bcast(Coop& c, int e, const double (&v)[NV], double (&out)[NV]) {
    static_assert(NV + 1 <= 12 && NV <= 16, "payload slots");
    Sh& sh = c.sh;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int wm = __reduce_min_sync(0xFFFFFFFFu, e);
    if (lane == 0) sh.i32[w] = wm;
    __syncthreads();
    const int bm = __reduce_min_sync(0xFFFFFFFFu, lane < NW ? sh.i32[lane] : 0x7FFFFFFF);
    if (e == bm && e != 0x7FFFFFFF) {
#pragma unroll
        for (int s = 0; s < NV; ++s) sh.f64[s] = v[s];
    }
    __syncthreads();
    if (c.nr == 1) {
#pragma unroll
        for (int s = 0; s < NV; ++s) out[s] = sh.f64[s];
        return bm;
    }
    const unsigned b = c.par & 1u;
    if (threadIdx.x < c.nr) {
        long long* dst = c.cl.map_shared_rank(&sh.xl[b][c.rank][0], threadIdx.x);
        dst[0] = bm;
#pragma unroll
        for (int s = 0; s < NV; ++s) dst[1 + s] = __double_as_longlong(sh.f64[s]);
    }
    c.xarrive_wait();
    const int rm = lane < (int)c.nr ? (int)sh.xl[b][lane][0] : 0x7FFFFFFF;
    const int gm = __reduce_min_sync(0xFFFFFFFFu, rm);
    const int src = __ffs(__ballot_sync(0xFFFFFFFFu, rm == gm)) - 1;
#pragma unroll
    for (int s = 0; s < NV; ++s) out[s] = __longlong_as_double(sh.xl[b][src][1 + s]);
    return gm;
}

// ---------------------------------------------------------------------------------------------
// metric evaluation
// ---------------------------------------------------------------------------------------------
struct Consts {
    double n, sx, sx2, thr;
    int metric;
    // derived (pcc): reference intermediates and the filter's constants
    double mx, nmx, am2, inv_n, K;
    bool filter_ok;
};
__device__ __forceinline__ void consts_finish(Consts& c) {
    c.mx = c.n != 0.0 ? __ddiv_rn(c.sx, c.n) : 0.0;
    c.nmx = __dmul_rn(c.n, c.mx);
    double am2 = __dsub_rn(c.sx2, __dmul_rn(c.nmx, c.mx));
    if (am2 < 0.0) am2 = 0.0;
    c.am2 = am2;
    c.inv_n = c.n != 0.0 ? 1.0 / c.n : 0.0;
    c.K = c.thr * c.thr * am2;
    c.filter_ok = c.metric == QA_METRIC_PCC && c.thr > 0.0 && am2 > 0.0 && c.n > 0.0 && isfinite(c.K);
}
// mixed_tile_greedy.py:176-190 in Python-float order (no contraction); mx, n*mx and am2 are loop invariants
// (out of line: the division / square-root sequences are long and only run for near-ties and for the final report;
// keeping them out of the decision loop keeps its instruction footprint small)
__device__ __noinline__ double pcc_value_cold(double n, double am2, double nmx, double sy, double sy2, double sxy, double sabs) {
    if (n == 0.0) return 1.0;
    const double my = __ddiv_rn(sy, n);
    double bm2 = __dsub_rn(sy2, __dmul_rn(__dmul_rn(n, my), my));
    if (bm2 < 0.0) bm2 = 0.0;
    const double den = __dsqrt_rn(__dmul_rn(am2, bm2));
    if (den == 0.0) return sabs == 0.0 ? 1.0 : 0.0;
    return __ddiv_rn(__dsub_rn(sxy, __dmul_rn(nmx, my)), den);
}
__device__ __forceinline__ double pcc_value_par(const Consts& c, double sy, double sy2, double sxy, double sabs) {
    return pcc_value_cold(c.n, c.am2, c.nmx, sy, sy2, sxy, sabs);
}
// `mrg` collects the smallest relative distance of any evaluated decision from the threshold, |value - thr| / thr (for pcc
// through the gap: (num^2 - K bm2) / (num^2 + K bm2) ~ (value - thr) / thr).  It is taken over every evaluation, speculative
// ones included, so it is a lower bound of the real minimum: a caller that knows how far its sums may be from the
// reference's (the fast tile-stat kernel's sum x^2, tree-summed initial sums) can certify the map against it.
__device__ __forceinline__ bool good_par(const Consts& c, const double (&S)[4], double& mrg) {
    if (c.metric != QA_METRIC_PCC) {
        const double v = c.n != 0.0 ? __ddiv_rn(S[3], c.n) : 0.0;
        mrg = fmin(mrg, fabs(v - c.thr) / fmax(fabs(c.thr), 1e-300));
        return v <= c.thr;
    }
    if (c.filter_ok) {
        // value >= thr  <=>  num >= thr*den  <=>  num > 0 and num^2 >= thr^2 * am2 * bm2.
        // Evaluate both sides with multiplications only and decide when the gap exceeds a bound on
        // every rounding involved (here and in the reference formula): 512 ulp of the terms.
        const double my = S[0] * c.inv_n;
        const double t1 = c.nmx * my;
        const double num = S[2] - t1;
        const double t2 = (c.n * my) * my;
        const double bm2 = S[1] - t2;
        const double enum_ = 5.7e-14 * (fabs(S[2]) + fabs(t1));            // bound on the error of num
        const double ebm2 = 5.7e-14 * (fabs(S[1]) + fabs(t2));             // ... and of bm2
        if (bm2 > ebm2) {
            if (num < -enum_) return false;                                 // certainly negative correlation
            if (num > enum_) {
                const double lhs = num * num, rhs = c.K * bm2;
                const double gap = lhs - rhs;
                const double tol = 2.0 * enum_ * fabs(num) + c.K * ebm2 + 5.7e-14 * (lhs + rhs);
                if (fabs(gap) > tol) {
                    mrg = fmin(mrg, fabs(gap) / (lhs + rhs));
                    return gap > 0.0;
                }
            }
        }
    }
    const double v = pcc_value_par(c, S[0], S[1], S[2], S[3]);
    mrg = fmin(mrg, fabs(v - c.thr) / fmax(fabs(c.thr), 1e-300));
    return v >= c.thr;
}

// ---------------------------------------------------------------------------------------------
// numpy permutation, parallel
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t pcg_out(u128 s) {
    const uint64_t x = s.hi ^ s.lo;
    const uint32_t rot = (uint32_t)(s.hi >> 58);
    return (x >> rot) | (x << ((64u - rot) & 63u));
}
__device__ __forceinline__ u128 pcg_step(u128 s, u128 inc) {
    return add128(mul128(s, u128{QA_PCG_MULT_HI, QA_PCG_MULT_LO}), inc);
}
__device__ void lcg_jump_consts(u128 inc, uint64_t delta, u128& am, u128& ap) {
    am = u128{0, 1};
    ap = u128{0, 0};
    u128 cm{QA_PCG_MULT_HI, QA_PCG_MULT_LO}, cp = inc;
    while (delta) {
        if (delta & 1ull) { am = mul128(am, cm); ap = add128(mul128(ap, cm), cp); }
        cp = mul128(add128(cm, u128{0, 1}), cp);
        cm = mul128(cm, cm);
        delta >>= 1;
    }
}

// accepts among this thread's DPT raw draws when `c` accepts precede them: step i = T - c draws until
// (raw & mask(i)) <= i (numpy random_interval); at most L accepts in total.
__device__ __forceinline__ int local_accepts(const uint32_t (&raw)[DPT], uint32_t validmask, int c, int T, int L) {
    int a = 0;
#pragma unroll
    for (int j = 0; j < DPT; ++j) {
        const int i = T - (c + a);
        const uint32_t mask = i > 0 ? (0xFFFFFFFFu >> __clz((uint32_t)i)) : 0u;
        const bool ok = ((validmask >> j) & 1u) && (c + a < L) && ((raw[j] & mask) <= (uint32_t)i);
        a += ok ? 1 : 0;
    }
    return a;
}

// Generates numpy's permutation(m) from the stream in `g` (uniform: every thread of the cluster holds
// the same copy) and writes out[k] = cand ? cand[perm[k]] : perm[k].  apply == false only advances
// the stream (the visiting order is irrelevant when the running state cannot change).
// Part 1 (perm_resolve): the swap targets j[m-1..1] and the stream position after them.
// Part 2 (perm_apply):   the swap sequence applied to the identity, in parallel.
__device__ void perm_resolve(Coop& c, Pcg& g, int m, int32_t* jarr) {     // jarr == nullptr: stream position only
    const int tid = threadIdx.x;
    if (m <= 1) return;
    // jump constants: 4*gtid LCG steps (this thread's offset in a round) and one full round
    u128 am, ap, rm, rp;
    lcg_jump_consts(g.inc, 4ull * (uint64_t)c.gtid, am, ap);
    lcg_jump_consts(g.inc, 4ull * (uint64_t)c.gth, rm, rp);
    // uniform stream cursor: rs = LCG state at output index rk (out_k = pcg_out(state_k); the buffered
    // half, if any, is the high half of out_0); pnext = position (2*k + half) of the next unconsumed draw
    u128 rs = g.s;
    unsigned long long rk = 0ull, pnext = g.has32 ? 1ull : 2ull;
    int i_cur = m - 1;
    long long t0 = clock64();
#ifdef QA_DBG_PERM
    long long d_gen = 0, d_sw = 0, d_wr = 0, td;
    int d_sweeps = 0, d_rounds = 0;
#endif
    while (i_cur > SEQ_TAIL) {
        ++c.n_rounds;
#ifdef QA_DBG_PERM
        __syncthreads(); td = clock64(); ++d_rounds;
#endif
        const int L = i_cur - SEQ_TAIL;                      // accepts still wanted from the parallel part
        const unsigned long long kb = pnext >> 1;
        if (kb != rk) {
            if (kb - rk == 4ull * (unsigned long long)c.gth) rs = add128(mul128(rm, rs), rp);
            else { u128 a2, p2; lcg_jump_consts(g.inc, kb - rk, a2, p2); rs = add128(mul128(a2, rs), p2); }
            rk = kb;
        }
        u128 s = add128(mul128(am, rs), ap);                 // state at output index kb + 4*gtid
        uint32_t raw[DPT];
#pragma unroll
        for (int j = 0; j < DPT / 2; ++j) {
            const uint64_t o = pcg_out(s);
            raw[2 * j] = (uint32_t)o;
            raw[2 * j + 1] = (uint32_t)(o >> 32);
            s = pcg_step(s, g.inc);
        }
        const unsigned long long p0 = 2ull * (kb + 4ull * (unsigned long long)c.gtid);
        uint32_t validmask = 0;
#pragma unroll
        for (int j = 0; j < DPT; ++j)
            if (p0 + j >= pnext) validmask |= 1u << j;
        // fixed point of c_in = exclusive_prefix(accepts(c_in)); thread 0 is right from the start and
        // every sweep fixes at least one more thread (typically all of them within ~10 sweeps)
        // start from the expected accept count at the current acceptance rate (any start converges: the prefix of
        // thread 0 is exact from the first exchange on, and every sweep fixes at least one more thread)
#ifdef QA_DBG_PERM
        __syncthreads(); d_gen += clock64() - td; td = clock64();
#endif
        int c_in, total = 0, a_prev = -1;
        {
            // expected accepts among the valid draws before this thread's first one: within a mask bracket the rate is
            // (i + 1) / (mask + 1) with i falling by one per accept, so c(d) = (i + 1)(1 - exp(-d / (mask + 1)))
            double dd = (double)(p0 > pnext ? p0 - pnext : 0ull), acc = 0.0;
            int i = i_cur;
            while (dd > 0.0 && i > 0) {
                const uint32_t mk = 0xFFFFFFFFu >> __clz((uint32_t)i);
                const double mp1 = (double)mk + 1.0;
                const double A = (double)(i - (int)(mk >> 1));            // accepts until the mask halves
                const double d_full = -mp1 * log(1.0 - A / ((double)i + 1.0));
                if (dd >= d_full) { acc += A; i -= (int)A; dd -= d_full; }
                else { acc += ((double)i + 1.0) * (1.0 - exp(-dd / mp1)); break; }
            }
            c_in = min(L, (int)(acc + 0.5));
        }
        int a = local_accepts(raw, validmask, c_in, i_cur, L);
        for (;;) {
            // one exchange per sweep: prefix of the accept counts + "did any count change since the last sweep";
            // when none changed the prefix is the one the counts were computed from, i.e. the fixed point
            bool any;
            ++c.n_sweeps;
            const int c_new = c_scan_excl_any(c, a, total, a != a_prev, any);
            if (!any) break;
            a_prev = a;
            c_in = c_new;
            a = local_accepts(raw, validmask, c_in, i_cur, L);
        }
#ifdef QA_DBG_PERM
        __syncthreads(); d_sw += clock64() - td; td = clock64();
#endif
        // write j for the steps this thread resolved; find the draw that supplied the L-th accept
        int done_off = 0x7FFFFFFF;
        {
            int cc = c_in;
#pragma unroll
            for (int j = 0; j < DPT; ++j) {
                const int i = i_cur - cc;
                const uint32_t mask = i > 0 ? (0xFFFFFFFFu >> __clz((uint32_t)i)) : 0u;
                const bool ok = ((validmask >> j) & 1u) && (cc < L) && ((raw[j] & mask) <= (uint32_t)i);
                if (ok) {
                    if (jarr) jarr[i] = (int32_t)(raw[j] & mask);
                    ++cc;
                    if (cc == L) done_off = c.gtid * DPT + j;
                }
            }
        }
        if (total >= L) {
            const int off = c_min(c, done_off);
            pnext = 2ull * kb + (unsigned long long)off + 1ull;
        } else {
            pnext = 2ull * (kb + 4ull * (unsigned long long)c.gth);      // every draw of the round was consumed
        }
        i_cur -= total;
#ifdef QA_DBG_PERM
        __syncthreads(); d_wr += clock64() - td;
#endif
    }
#ifdef QA_DBG_PERM
    __syncthreads();
    const long long t_tail0 = clock64();
#endif
    // tail (the last <= SEQ_TAIL steps) and stream hand-back, by warp 0 of every CTA (redundantly, identically): the
    // lanes generate the next 256 draws in parallel (one LCG jump per lane), lane 0 consumes them in order.
    if (tid < 32) {
        const int lane = tid;
        unsigned long long pcur = pnext;                      // next unconsumed draw position
        unsigned long long k0 = pcur >> 1;                    // output index of the batch's first 64-bit draw
        u128 a2, p2, la, lp, ba, bp;
        lcg_jump_consts(g.inc, k0 - rk, a2, p2);
        u128 sb = add128(mul128(a2, rs), p2);                 // state at output index k0
        lcg_jump_consts(g.inc, 4ull * (uint64_t)lane, la, lp);
        lcg_jump_consts(g.inc, 128ull, ba, bp);
        long long* st = c.sh.i64;                             // [128][2] LCG states of the batch
        unsigned* dr = c.sh.tail_draws;                       // [256] 32-bit draws of the batch, in stream order
        int i = i_cur;
        for (;;) {
            u128 sl = add128(mul128(la, sb), lp);             // state at k0 + 4 * lane
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const uint64_t o = pcg_out(sl);
                const int idx = 4 * lane + q;
                dr[2 * idx] = (uint32_t)o;
                dr[2 * idx + 1] = (uint32_t)(o >> 32);
                st[2 * idx] = (long long)sl.hi;
                st[2 * idx + 1] = (long long)sl.lo;
                sl = pcg_step(sl, g.inc);
            }
            __syncwarp();
            int used = 0;
            if (lane == 0) {
                int off = (int)(pcur - 2ull * k0);            // 1 if the batch's first low half was consumed earlier
                while (i >= 1 && off < 256) {
                    const uint32_t mask = 0xFFFFFFFFu >> __clz((uint32_t)i);
                    const uint32_t v = dr[off++] & mask;
                    if (v <= (uint32_t)i) {
                        if (c.rank == 0 && jarr) jarr[i] = (int32_t)v;
                        --i;
                    }
                }
                used = off;
            }
            used = __shfl_sync(0xFFFFFFFFu, used, 0);
            i = __shfl_sync(0xFFFFFFFFu, i, 0);
            pcur = 2ull * k0 + (unsigned long long)used;
            if (i < 1) break;
            __syncwarp();
            k0 += 128ull;
            sb = add128(mul128(ba, sb), bp);
            pcur = 2ull * k0;
        }
        if (lane == 0) {
            const unsigned long long pl = pcur - 1ull;        // last consumed draw (the tail always consumes one)
            const int idx = (int)((pl >> 1) - k0);
            const long long shi = st[2 * idx], slo = st[2 * idx + 1];
            const unsigned hi_half = dr[2 * idx + 1];
            c.sh.i32[3 * NW + 2] = (pl & 1ull) == 0ull ? 1 : 0;     // a low half was consumed last: its high half is buffered
            c.sh.i32[3 * NW + 3] = (int)hi_half;
            c.sh.i64[256] = shi;
            c.sh.i64[257] = slo;
        }
    }
    __syncthreads();
    g.s.hi = (uint64_t)c.sh.i64[256];
    g.s.lo = (uint64_t)c.sh.i64[257];
    g.has32 = (uint32_t)c.sh.i32[3 * NW + 2];
    g.buf32 = (uint32_t)c.sh.i32[3 * NW + 3];
    c.sync();
#ifdef QA_DBG_PERM
    if (c.gtid == 0) printf("resolve m=%d rounds %d gen %lld sweeps %lld write+min %lld tail %lld total %lld\n", m, d_rounds, d_gen, d_sw, d_wr,
                            clock64() - t_tail0, clock64() - t0);
#endif
    c.cy_resolve += clock64() - t0;
}

__device__ void perm_apply(Coop& c, int m, const int32_t* cand, int32_t* out, const ParWork& w) {
    if (m <= 1) {
        if (m == 1 && c.gtid == 0) out[0] = cand ? cand[0] : 0;
        c.sync();
        return;
    }
    const long long t0 = clock64();
#ifdef QA_DBG_PERM
    long long tp[8]; int np_ = 0;
#define QA_TP() tp[np_++] = clock64()
#else
#define QA_TP()
#endif
    for (int p = c.gtid; p < m; p += c.gth) w.cursor[p] = 0;
    c.sync();
    QA_TP();
    for (int i = 1 + c.gtid; i < m; i += c.gth) atomicAdd(&w.cursor[w.jarr[i]], 1);
    c.sync();
    QA_TP();
    {   // exclusive scan of the per-position counts -> off[], contiguous range per thread
        const int per = (m + c.gth - 1) / c.gth;
        const int b = min(m, c.gtid * per), e = min(m, b + per);
        int local = 0;
        for (int p = b; p < e; ++p) local += w.cursor[p];
        int total;
        int run = c_scan_excl(c, local, total);
        for (int p = b; p < e; ++p) {
            const int cnt = w.cursor[p];
            w.off[p] = run;
            w.cursor[p] = run;
            run += cnt;
        }
        if (c.gtid == 0) w.off[m] = total;
    }
    c.sync();
    QA_TP();
    for (int i = 1 + c.gtid; i < m; i += c.gth) {
        const int slot = atomicAdd(&w.cursor[w.jarr[i]], 1);
        w.bucket[slot] = i;
    }
    c.sync();
    QA_TP();
    for (int p = c.gtid; p < m; p += c.gth) {
        const int b = w.off[p], e = w.off[p + 1];
        for (int a = b + 1; a < e; ++a) {          // insertion sort (buckets hold ~1 entry)
            const int key = w.bucket[a];
            int q = a - 1;
            while (q >= b && w.bucket[q] > key) { w.bucket[q + 1] = w.bucket[q]; --q; }
            w.bucket[q + 1] = key;
        }
        int par = -1;
        for (int a = b; a < e; ++a) {
            const int st = w.bucket[a];
            w.succ[st] = a + 1 < e ? w.bucket[a + 1] : -1;
            if (par < 0 && st != p) par = st;
        }
        w.parent[p] = par;       // first later-executed step that writes position p
    }
    c.sync();
    QA_TP();
    for (int i = c.gtid; i < m; i += c.gth) {
        // a[0] ends as the content of position 0 after all steps; a[i] (i >= 1) is what step i read
        const int start = i == 0 ? w.parent[0] : w.succ[i];
        int val;
        if (start < 0) val = i == 0 ? 0 : w.jarr[i];          // nobody wrote that position: initial content
        else {
            int cur = start;
            for (int pa = w.parent[cur]; pa >= 0; pa = w.parent[cur]) cur = pa;
            val = cur;
        }
        out[i] = cand ? cand[val] : val;
    }
    c.sync();
    QA_TP();
#ifdef QA_DBG_PERM
    if (c.gtid == 0) printf("apply m=%d zero %lld count %lld scan %lld fill %lld sort %lld follow %lld\n", m, tp[0] - t0, tp[1] - tp[0],
                            tp[2] - tp[1], tp[3] - tp[2], tp[4] - tp[3], tp[5] - tp[4]);
#endif
    c.cy_apply += clock64() - t0;
}

__device__ void permutation_par(Coop& c, Pcg& g, int m, const int32_t* cand, int32_t* out, const ParWork& w, bool apply) {
    perm_resolve(c, g, m, apply ? w.jarr : nullptr);
    if (apply) perm_apply(c, m, cand, out, w);
    else c.sync();
}

__global__ void __launch_bounds__(GT) permutation_par_kernel(qa_pcg64* rng, int m, int32_t* out, ParWork w) {
    __shared__ Sh sh;
    Coop c(sh);
    Pcg g;
    g.load(rng);
    c.sync();                       // everyone has read the stream before rank 0 overwrites it
    permutation_par(c, g, m, nullptr, out, w, true);
    if (c.gtid == 0) g.store(rng);
}

// One permutation's swap targets and the stream state after it (the apply runs as grid kernels, qa_perm_apply.cu)
__global__ void __launch_bounds__(GT) perm_resolve_kernel(const qa_pcg64* rng_in, int n, int32_t* jarr, qa_pcg64* rng_out) {
    __shared__ Sh sh;
    Coop c(sh);
    Pcg g;
    g.load(rng_in);
    c.sync();                       // rng_in may alias rng_out: everyone has read it before rank 0 overwrites it
    perm_resolve(c, g, n, jarr);
    if (c.gtid == 0) {
        rng_out->inc_hi = g.inc.hi;
        rng_out->inc_lo = g.inc.lo;
        g.store(rng_out);
    }
}

// `count` consecutive permutations of n items from one stream in ONE launch: the cluster keeps its SMs between them
// (a cluster that has to be re-placed while a streaming kernel floods the GPU waits for that kernel to drain).
__global__ void __launch_bounds__(GT) perm_resolve_chain_kernel(const qa_pcg64* rng_in, int n, int count, unsigned write_mask,
                                                                int32_t* jarr, qa_pcg64* rng_out) {
    __shared__ Sh sh;
    Coop c(sh);
    Pcg g;
    g.load(rng_in);
    if (c.gtid == 0) stamp(0, false);
    c.sync();
    for (int k = 0; k < count; ++k) {
        perm_resolve(c, g, n, ((write_mask >> k) & 1u) ? jarr + (size_t)k * n : nullptr);
        if (c.gtid == 0) {
            rng_out[k].inc_hi = g.inc.hi;
            rng_out[k].inc_lo = g.inc.lo;
            g.store(rng_out + k);
        }
    }
    if (c.gtid == 0) stamp(1, true);
}

// Per-thread staging of the chunk's addends in shared memory ([slot][thread] layout: conflict-free), so the
// walks of a round read them at shared-memory latency instead of re-fetching from L2.
constexpr int STAGE_SLOTS = 4 * EPS;                 // up to 4 streams x EPS elements per thread
extern __shared__ double qa_stage[];
__device__ __forceinline__ double& staged(int stream, int j) { return qa_stage[(stream * EPS + j) * GT + threadIdx.x]; }

// ---------------------------------------------------------------------------------------------
// faithful sequential sums of table columns (tile order): S_k = fl(S_{k-1} + t_k)
// ---------------------------------------------------------------------------------------------
// The first HEAD elements (a sum starting from zero changes binade at almost every step) are added
// by one thread; the rest rides the scan.  A column whose running sum keeps leaving its binade (a
// zero-mean random walk) is finished with a plain tree sum after max_events cuts and flagged.
template <int NC>
__device__ void faithful_init_sums(Coop& c, const double* const (&col)[NC], int pos_begin, int nt, double (&S)[NC],
                                   unsigned& degraded, int max_events) {
    // elements [pos_begin, nt) in order; pos_begin > 0 continues from the sums in S (the table may be produced in pieces)
    Sh& sh = c.sh;
    const int tid = threadIdx.x;
    constexpr int HEAD = 192;
    int events[NC];
#pragma unroll
    for (int s = 0; s < NC; ++s) events[s] = 0;
    degraded = 0;
    int pos = pos_begin;
    if (pos_begin == 0) {
#pragma unroll
    for (int s = 0; s < NC; ++s) S[s] = 0.0;
    pos = min(nt, HEAD);
    {   // stage the head in shared memory (parallel loads), then one thread per column adds it up in order
        static_assert(NC * HEAD <= STAGE_SLOTS * GT, "head staging does not fit");
        __syncthreads();
#pragma unroll
        for (int s = 0; s < NC; ++s)
            for (int i = tid; i < pos; i += GT) qa_stage[s * HEAD + i] = col[s][i];
        __syncthreads();
        if (tid < NC) {
            double acc = 0.0;
            for (int i = 0; i < pos; ++i) acc = __dadd_rn(acc, qa_stage[tid * HEAD + i]);
            sh.f64[tid] = acc;
        }
    }
    __syncthreads();
#pragma unroll
    for (int s = 0; s < NC; ++s) S[s] = sh.f64[s];
    __syncthreads();
    }
    const int CHc = c.gth * EPS;
    while (pos < nt) {
        ++c.n_init_rounds;
        // chunk length: a round ends at the first binade crossing anyway, so do not walk far past the point where
        // the fastest-growing column is expected to reach its next power of two (addends ~ S / pos each)
        double want = (double)CHc;
#pragma unroll
        for (int s = 0; s < NC; ++s) {
            const double a = fabs(S[s]);
            if (((degraded >> s) & 1u) || !(a > 0.0) || !(a < 1e300)) continue;
            const double top = __hiloint2double((__double2hiint(a) & 0x7FF00000) + 0x00100000, 0);   // next power of two
            want = fmin(want, (top - a) / a * (double)pos * 1.15 + 64.0);
        }
        const int len = min(max((int)want, c.gth), min(CHc, nt - pos));
        const int per = (len + c.gth - 1) / c.gth;                      // 1..EPS elements per thread
        const int lo = c.gtid * per, hi = min(len, lo + per);          // this thread streams elements [lo, hi)
        Grid g[NC];
#pragma unroll
        for (int s = 0; s < NC; ++s) g[s] = make_grid(S[s]);
        static_assert(NC <= 4, "staging holds four streams");
#pragma unroll
        for (int s = 0; s < NC; ++s)
#pragma unroll
            for (int j = 0; j < EPS; ++j) staged(s, j) = lo + j < hi ? col[s][pos + lo + j] : 0.0;
        // walk 1: compose this thread's additions (stop at the first one that cannot ride the grid)
        P2 tot[NC], pre0[NC];
#pragma unroll
        for (int s = 0; s < NC; ++s) tot[s] = P2{0, 0};
        int bad = 0x7FFFFFFF;
        for (int idx = lo; idx < hi && bad == 0x7FFFFFFF; ++idx) {
            P2 p[NC];
            bool ok = true;
#pragma unroll
            for (int s = 0; s < NC; ++s) {
                p[s] = P2{0, 0};
                if (!((degraded >> s) & 1u)) ok = classify(g[s], staged(s, idx - lo), p[s]) && ok;
            }
            if (!ok) { bad = idx; break; }
#pragma unroll
            for (int s = 0; s < NC; ++s) tot[s] = p2_then(tot[s], p[s]);
        }
        scan_totals<NC>(c, tot, pre0);
        // walk 2: this thread's first element that ends the chunk - one that cannot ride the grid, one whose result
        // leaves a binade, or the chunk's last element - and the state after it, fl(S_before + t): a real add from
        // the exact state before it.  The cluster-wide first such element wins.
        int e_l = 0x7FFFFFFF;
        double cand_nv[NC], nv[NC];
#pragma unroll
        for (int s = 0; s < NC; ++s) cand_nv[s] = 0.0;
        {
            P2 run[NC], prev[NC];
#pragma unroll
            for (int s = 0; s < NC; ++s) run[s] = prev[s] = pre0[s];
            for (int idx = lo; idx < hi; ++idx) {
#pragma unroll
                for (int s = 0; s < NC; ++s) prev[s] = run[s];
                if (idx == bad) { e_l = idx; break; }
                bool leaves = false;
#pragma unroll
                for (int s = 0; s < NC; ++s) {
                    if ((degraded >> s) & 1u) continue;
                    P2 p{0, 0};
                    classify(g[s], staged(s, idx - lo), p);
                    run[s] = p2_then(run[s], p);
                    if (g[s].q != 0.0 && !in_binade(m_after(g[s], run[s]))) leaves = true;
                }
                if (leaves || idx == len - 1) { e_l = idx; break; }
            }
            if (e_l != 0x7FFFFFFF) {
#pragma unroll
                for (int s = 0; s < NC; ++s) {
                    const double before = g[s].q != 0.0 ? s_of(g[s], m_after(g[s], prev[s])) : S[s];
                    cand_nv[s] = __dadd_rn(before, staged(s, e_l - lo));
                }
            }
        }
        const int cut = c_argmin_bcast<NC>(c, e_l, cand_nv, nv);
        const bool cut_short = cut < len - 1;
#pragma unroll
        for (int s = 0; s < NC; ++s) {
            if ((degraded >> s) & 1u) continue;
            if (cut_short) {
                const Grid gn = make_grid(nv[s]);
                if (gn.q != g[s].q || g[s].q == 0.0) ++events[s];      // this column left its grid here
            }
            S[s] = nv[s];
        }
        pos += cut + 1;
#pragma unroll
        for (int s = 0; s < NC; ++s) {
            if (!((degraded >> s) & 1u) && events[s] > max_events) {
                double part = 0.0;
                for (int i = pos + c.gtid; i < nt; i += c.gth) part += col[s][i];
                S[s] = S[s] + c_reduce_d<false>(c, part);
                degraded |= 1u << s;
            }
        }
        bool all_deg = true;
#pragma unroll
        for (int s = 0; s < NC; ++s) all_deg = all_deg && ((degraded >> s) & 1u);
        if (all_deg) break;
    }
}

// ---------------------------------------------------------------------------------------------
// init phase: initial sums and per-transition drift bounds (data-dependent, permutation-independent)
// ---------------------------------------------------------------------------------------------
// hdr: [0] sx  [1] sx2  [2..5] sy, sy2, sxy, sabs of the base format  [6] degraded bits  [7] cycles
//      [8] cycles of the non-negative columns  [9] cycles of the signed columns  [10] scan rounds
template <bool PCC>
__device__ void init_phase(Coop& c, const double* __restrict__ table, int nt, const ParOrder& ord, double* hdr, int t_begin,
                           int t_end) {
    // Tiles [t_begin, t_end) of the sequential sums; a call with t_end < nt only advances the sums of the non-negative
    // columns (kept in hdr[16..19]) so that it can run while the rest of the table is still being produced; the call that
    // reaches nt finishes everything else.
    const int base = ord.fmt[0];
    const long long t_start = clock64();
    double sx = 0.0, sx2 = 0.0;
    double S[4] = {0.0, 0.0, 0.0, 0.0};      // sy, sy2, sxy, sabs (mae uses S[3] only)
    double dr_sum[QA_NFMT - 1];              // per transition: sum |delta sy| over all tiles (pcc)
#pragma unroll
    for (int tr = 0; tr + 1 < QA_NFMT; ++tr) dr_sum[tr] = 0.0;
    unsigned degraded = 0;
    if (PCC) {
        {   // sums of non-negative terms: few binade changes, always carried faithfully
            const double* const cols[4] = {table + (size_t)QA_STAT_SX2 * nt, table + (size_t)QA_STAT_FMT(base, 1) * nt,
                                           table + (size_t)QA_STAT_FMT(base, 2) * nt, table + (size_t)QA_STAT_FMT(base, 3) * nt};
            double R[4] = {hdr[16], hdr[17], hdr[18], hdr[19]};      // only read when t_begin > 0
            unsigned dg;
            const long long ti = clock64();
            faithful_init_sums<4>(c, cols, t_begin, t_end, R, dg, 1 << 30);
            c.cy_i0 += clock64() - ti;
            if (t_end < nt) {
                if (c.gtid == 0) { hdr[16] = R[0]; hdr[17] = R[1]; hdr[18] = R[2]; hdr[19] = R[3]; hdr[20] = (double)c.n_init_rounds; }
                return;
            }
            sx2 = R[0]; S[1] = R[1]; S[2] = R[2]; S[3] = R[3];
        }
        {   // signed sums (means).  A sum with heavy cancellation (|sum t| << sum |t|: zero-mean weights) is a
            // random walk that changes binade all the time; it goes straight to a fixed-order tree sum and is
            // flagged (its rounding differences are ~1e-16 of a term that enters bm2 at the 1e-7 level).
            // Otherwise it is carried with the reference's rounding sequence like the other columns.
            const double* const cols[2] = {table + (size_t)QA_STAT_SX * nt, table + (size_t)QA_STAT_FMT(base, 0) * nt};
            double R[2];
            bool walk[2];
            const long long ti = clock64();
            // one pass over the tiles for everything that is a plain fixed-order sum: sum / sum|.| of the two signed
            // columns and, per format transition, sum |delta sy| (bounds how far sy can drift during that pass)
            double acc[4 + QA_NFMT - 1];
#pragma unroll
            for (int q = 0; q < 4 + QA_NFMT - 1; ++q) acc[q] = 0.0;
#pragma unroll 2
            for (int i = c.gtid; i < nt; i += c.gth) {
                const double vx = cols[0][i];
                double vy[QA_NFMT];
#pragma unroll
                for (int f = 0; f < QA_NFMT; ++f) vy[f] = f < ord.n ? table[(size_t)QA_STAT_FMT(ord.fmt[f], 0) * nt + i] : 0.0;
                acc[0] += vx; acc[1] += fabs(vx);
                acc[2] += vy[0]; acc[3] += fabs(vy[0]);
#pragma unroll
                for (int tr = 0; tr + 1 < QA_NFMT; ++tr)
                    if (tr + 1 < ord.n) acc[4 + tr] += fabs(__dsub_rn(vy[tr + 1], vy[tr]));
            }
            c_reduce_sum_multi<4 + QA_NFMT - 1>(c, acc);
            R[0] = acc[0]; R[1] = acc[2];
            walk[0] = fabs(R[0]) < 0.25 * acc[1];
            walk[1] = fabs(R[1]) < 0.25 * acc[3];
#pragma unroll
            for (int tr = 0; tr + 1 < QA_NFMT; ++tr) dr_sum[tr] = acc[4 + tr];
            if (walk[0] && walk[1]) degraded = 3u;
            else faithful_init_sums<2>(c, cols, 0, nt, R, degraded, 24);
            c.cy_i1 += clock64() - ti;
            sx = R[0]; S[0] = R[1];
        }
    } else {
        const double* const cols[1] = {table + (size_t)QA_STAT_FMT(base, 3) * nt};
        double R[1] = {hdr[16]};
        unsigned dg;
        faithful_init_sums<1>(c, cols, t_begin, t_end, R, dg, 1 << 30);
        if (t_end < nt) {
            if (c.gtid == 0) { hdr[16] = R[0]; hdr[20] = (double)c.n_init_rounds; }
            return;
        }
        S[3] = R[0];
    }
    if (c.gtid == 0) {
#pragma unroll
        for (int tr = 0; tr + 1 < QA_NFMT; ++tr) hdr[11 + tr] = dr_sum[tr];
        hdr[0] = sx; hdr[1] = sx2; hdr[2] = S[0]; hdr[3] = S[1]; hdr[4] = S[2]; hdr[5] = S[3];
        hdr[6] = (double)degraded;
        hdr[7] = (double)(clock64() - t_start);
        hdr[8] = (double)c.cy_i0; hdr[9] = (double)c.cy_i1; hdr[10] = (double)c.n_init_rounds + (t_begin > 0 ? hdr[20] : 0.0);
    }
}

template <bool PCC>
__global__ void __launch_bounds__(GT) greedy_init_kernel(const double* __restrict__ table, int nt, ParOrder ord, double* hdr,
                                                         int t_begin, int t_end) {
    __shared__ Sh sh;
    Coop c(sh);
    if (c.gtid == 0) stamp(2, false);
    init_phase<PCC>(c, table, nt, ord, hdr, t_begin, t_end);
    if (c.gtid == 0) stamp(3, true);
}

// delta[tr][t] = stats(fmt[tr+1]) - stats(fmt[tr]) of tile t: one 32-byte record per tile and transition, so the chain
// fetches a visited tile with one sector instead of eight
__device__ __forceinline__ void write_deltas(const double* __restrict__ table, int nt, const ParOrder& ord, double* delta, int t) {
    double v[QA_NFMT][4];
#pragma unroll
    for (int f = 0; f < QA_NFMT; ++f)
#pragma unroll
        for (int q = 0; q < 4; ++q) v[f][q] = f < ord.n ? table[(size_t)QA_STAT_FMT(ord.fmt[f], q) * nt + t] : 0.0;
#pragma unroll
    for (int tr = 0; tr + 1 < QA_NFMT; ++tr) {
        if (tr + 1 >= ord.n) break;
        double2* dst = reinterpret_cast<double2*>(delta + ((size_t)tr * nt + t) * 4);
        dst[0] = make_double2(__dsub_rn(v[tr + 1][0], v[tr][0]), __dsub_rn(v[tr + 1][1], v[tr][1]));
        dst[1] = make_double2(__dsub_rn(v[tr + 1][2], v[tr][2]), __dsub_rn(v[tr + 1][3], v[tr][3]));
    }
}

// delta records of every format transition, one thread per tile
__global__ void __launch_bounds__(256) greedy_delta_kernel(const double* __restrict__ table, int nt, ParOrder ord, double* delta) {
    const int t = blockIdx.x * 256 + threadIdx.x;
    if (t >= nt) return;
    write_deltas(table, nt, ord, delta, t);
}

// the same for a descriptor array of tensors: block b finds its tensor by bisection over the block prefix
__global__ void __launch_bounds__(256) greedy_delta_batch_kernel(const qa_batch_desc* __restrict__ descs, int n, ParOrder ord, int64_t hdr_bytes) {
    const int64_t b = blockIdx.x;
    int lo = 0, hi = n - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (__ldg(&descs[mid].block_begin) <= b) lo = mid; else hi = mid - 1;
    }
    const qa_batch_desc d = descs[lo];
    const int nt = (int)(cdiv(d.rows, TILE) * cdiv(d.cols, TILE));
    const int t = (int)(b - d.block_begin) * 256 + threadIdx.x;
    if (t >= nt) return;
    write_deltas(d.table, nt, ord, reinterpret_cast<double*>(reinterpret_cast<char*>(d.init) + hdr_bytes), t);
}

// ---------------------------------------------------------------------------------------------
// the greedy kernel
// ---------------------------------------------------------------------------------------------
// The chain kernel is capped at 128 registers (it wants 250): a 256-thread CTA then holds half of an SM's register file and
// two tile-stat CTAs of the next tensor lists fit beside it.  The cluster kernels issue on ~17 % of the cycles, the tile-stat
// kernel is pipe-bound, so sharing the SMs pays once enough lists are in flight: cfg2 step 0.286 -> 0.269 ms with 12 lists
// (profiles/r2_chain_regcap2.txt, r2_chain_regcap3.txt; 96 / 112 registers give the same, 168 nothing), at the price of a
// 13 % longer chain for a tensor processed alone (0.326 -> 0.369 ms).  -DQA_CHAIN_MAXNREG=0 restores the uncapped kernel.
#ifndef QA_CHAIN_MAXNREG
#define QA_CHAIN_MAXNREG 128
#endif
#if QA_CHAIN_MAXNREG > 0
#define QA_CHAIN_REGCAP __maxnreg__(QA_CHAIN_MAXNREG)
#else
#define QA_CHAIN_REGCAP __launch_bounds__(GT, 1)
#endif
// The chain body, shared by the single-run kernel and the sweep kernel.  The stream starts at *rng_in; its final position goes
// to *rng_out (the same pointer for a single run; a private slot for a sweep chain, whose starting state is shared).
template <bool PCC>
__device__ __forceinline__ void greedy_chain(const double* __restrict__ table, int nt, double numel, int metric, double thr,
                                             ParOrder ord, const qa_pcg64* rng_in, qa_pcg64* rng_out, int8_t* assignment,
                                             int64_t* counts, double* state, ParWork w, int fi_begin, int fi_end, int flags) {
    // Passes [fi_begin, fi_end) of the format order.  A run may be split into several launches (so that a later pass can
    // wait for a prefetched permutation that an earlier one does not need); the running state travels in w.res.  The
    // initial sums and delta records (w.hdr, w.delta) were written ahead of the chain by greedy_init_kernel and a delta kernel.
    __shared__ Sh sh;
    Coop c(sh);
    const int tid = threadIdx.x;
    const int base = ord.fmt[0];
    const bool first = fi_begin == 0, last = fi_end >= ord.n;
    if (c.gtid == 0) stamp(first ? 4 : 6, false);
    constexpr bool is_pcc = PCC;
    // running sums carried with the reference's exact rounding sequence: sy, sy2, sxy (pcc) | sabs (mae).
    // In pcc mode sum|x-y| only enters the degenerate den == 0 branch (mixed_tile_greedy.py:187-188): it is
    // tracked as a plain per-chunk sum (it starts at 0 and would change binade ~40 times on its way up).
    constexpr int NS = PCC ? 3 : 1;
    constexpr int S0 = PCC ? 0 : 3;       // first table statistic among them
    if (first) {
        for (int t = c.gtid; t < nt; t += c.gth) { assignment[t] = (int8_t)base; w.fixed[t] = 0; }
        if (c.gtid < QA_NFMT) counts[c.gtid] = c.gtid == base ? nt : 0;
    }
    if (tid < QA_NFMT) sh.cnt[tid] = 0;
    Pcg g;
    g.load(rng_in);
    c.sync();
    const long long t_start = clock64();

    // ---- (1) initial sums, sequentially rounded in tile order (greedy_init_kernel) ----
    Consts k;
    k.n = numel; k.thr = thr; k.metric = metric;
    k.sx = w.hdr[0]; k.sx2 = w.hdr[1];
    double S[4] = {w.hdr[2], w.hdr[3], w.hdr[4], w.hdr[5]};
    unsigned degraded = (unsigned)w.hdr[6];
    consts_finish(k);
    unsigned chain_rounds = 0;
    const int32_t* order_ptr = w.order;
    long long t_mark = clock64(), cyc_perm = 0, cyc_chain = 0;
    long long cy_load = 0, cy_scan = 0, cy_dec = 0, cy_min = 0, cy_commit = 0, cy_gather = 0, tq = 0;
    unsigned n_chunks = 0, n_cutshort = 0;
    const long long cyc_init = (long long)w.hdr[7];
    const int CHc = c.gth * EPS;
    bool base_failed = false, all_tiles_candidates = true, done = false;
    int accepted_last = nt;
    double min_margin = 1e300;          // smallest relative distance of an evaluated decision from the threshold (good_par)
    if (!first) {
        const double* r = w.res;
        min_margin = r[14];
        S[0] = r[0]; S[1] = r[1]; S[2] = r[2]; S[3] = r[3];
        degraded = (unsigned)r[4]; chain_rounds = (unsigned)r[5];
        base_failed = r[6] != 0.0; all_tiles_candidates = r[7] != 0.0; accepted_last = (int)r[8];
        cyc_perm = (long long)r[9]; cyc_chain = (long long)r[10]; done = r[11] != 0.0;
        n_chunks = (unsigned)r[12]; n_cutshort = (unsigned)r[13];
    }

    for (int fi = fi_begin; fi < fi_end && fi < ord.n && !done; ++fi) {
        const int fmt = ord.fmt[fi];
        // ---- candidates = not-fixed tiles in ascending order ------------------------------
        // The base pass fixes every tile or none, and a pass that accepted all of its candidates fixes none: as long
        // as that holds the candidates are the tiles 0..nt-1 themselves and no list is built (cand == nullptr).
        int m;
        const int32_t* cand = nullptr;
        if (fi == 0) m = nt;
        else if (fi == 1) m = base_failed ? 0 : nt;
        else if (all_tiles_candidates && accepted_last == nt) m = nt;
        else {
            all_tiles_candidates = false;
            const int lane = tid & 31;
            const int nwarps = c.gth >> 5, gw = c.gtid >> 5;
            const int per_w = (((nt + nwarps - 1) / nwarps) + 31) & ~31;        // a multiple of 32 tiles per warp
            const int b = min(nt, gw * per_w), e = min(nt, b + per_w);
            int cntw = 0;
            for (int t0 = b; t0 < e; t0 += 32) {
                const int t = t0 + lane;
                cntw += __popc(__ballot_sync(0xFFFFFFFFu, t < e && !w.fixed[t]));
            }
            int run = c_scan_excl(c, lane == 0 ? cntw : 0, m);                  // lane 0: candidates in earlier warps
            run = __shfl_sync(0xFFFFFFFFu, run, 0);
            for (int t0 = b; t0 < e; t0 += 32) {
                const int t = t0 + lane;
                const bool keep = t < e && !w.fixed[t];
                const unsigned bal = __ballot_sync(0xFFFFFFFFu, keep);
                if (keep) w.cand[run + __popc(bal & ((1u << lane) - 1u))] = t;
                run += __popc(bal);
            }
            cand = w.cand;
            c.sync();
        }
        if (m == 0) {
            // the base pass fixed every tile: only permutation #1 was consumed (rare; redo it if it was prefetched away)
            if (fi == 1 && w.pre_order != nullptr && w.npre >= 2 && ord.n >= 2) permutation_par(c, g, nt, nullptr, w.order, w, false);
            done = true;
            break;
        }
        int my_accepts = 0;                              // accepted by this thread during the pass
        const bool base_pass = fi == 0;
        // every candidate of pass fi was accepted in pass fi-1 (rejected tiles are fixed), so its
        // current format is the previous one in the order
        const int prev = base_pass ? base : ord.fmt[fi - 1];
        const double* dtab = w.delta + (size_t)(base_pass ? 0 : fi - 1) * nt * 4;      // {d sy, d sy2, d sxy, d sabs} per tile
        // sy is a signed sum near its mean: if the pass could carry it across a binade boundary (or zero),
        // run it on a fixed coarser grid instead of cutting a chunk at every hop
        bool relax_sy = false;
        double drift = 0.0;                              // sum |delta sy| over the candidates: how far sy can move
        if (PCC && !base_pass) {
            tq = clock64();
            if (cand == nullptr) drift = w.hdr[11 + fi - 1];      // every tile is a candidate: summed by the init phase
            else {
                for (int q = c.gtid; q < m; q += c.gth) drift += fabs(dtab[4 * (size_t)cand[q]]);
                drift = c_reduce_d<false>(c, drift);
            }
            relax_sy = !stays_in_binade(S[0], drift);
            if (relax_sy) degraded |= 4u;
            cy_gather += clock64() - tq;
        }
        // ---- (2) visiting order ----------------------------------------------------------
        t_mark = clock64();
        const bool have_pre = w.pre_order != nullptr && w.npre >= 2 && ord.n >= 2;
        order_ptr = w.order;
        if (have_pre && fi == 0) {
            // permutations #1 and #2 were drawn ahead of time; nothing to do for the base pass
        } else if (have_pre && fi == 1) {
            order_ptr = w.pre_order;          // m == nt here: candidates are 0..nt-1 in order, so perm[k] is the tile
            g.load(w.pre_rng);
        } else if (have_pre && fi == 2 && w.npre >= 3 && m == nt) {
            order_ptr = w.pre_order + nt;     // pass 2 accepted every tile: the speculative third permutation applies
            g.load(w.pre_rng + 1);
        } else {
            // Order-free shortcut: the state only changes on an accept, so if no candidate passes against the state at
            // the start of the pass, every candidate sees exactly that state whatever the visiting order and all are
            // rejected.  Then only the stream position of the permutation is needed, not the permutation itself.
            bool none = false;
            double sb0_start = S[0];
            if (!base_pass) {
                double sb0 = S[0];
                if (PCC && relax_sy) {
                    const Grid gx = make_grid_relaxed(S[0], drift);
                    if (gx.q != 0.0) sb0 = s_of(gx, gx.m0);          // the chain starts from the grid-rounded value
                    sb0_start = sb0;
                }
                auto passes = [&](int q) -> bool {
                    const double2* rec = reinterpret_cast<const double2*>(dtab) + 2 * (size_t)(cand ? cand[q] : q);
                    const double2 ra = rec[0], rb = rec[1];
                    double cnd[4] = {0.0, 0.0, 0.0, 0.0};
                    if (PCC) {
                        cnd[0] = __dadd_rn(sb0, ra.x); cnd[1] = __dadd_rn(S[1], ra.y); cnd[2] = __dadd_rn(S[2], rb.x);
                        cnd[3] = S[3] + rb.y;
                    } else cnd[3] = __dadd_rn(S[3], rb.y);
                    return good_par(k, cnd, min_margin);
                };
                bool acc = c.gtid < m && passes(c.gtid);              // a sample first: passes that do accept stop here
                if (!c_any(c, acc)) {
                    for (int q = c.gtid + c.gth; q < m && !acc; q += c.gth) acc = passes(q);
                    none = !c_any(c, acc);
                }
            }
            if (none) {
                if (PCC && relax_sy) S[0] = sb0_start;              // what an all-reject chain leaves behind
                // the permutation of an order-free pass only moves the stream; after the LAST pass nothing reads the
                // stream any more unless the caller wants its final position (QA_GREEDY_SKIP_FINAL_STREAM)
                if (!((flags & 1) && fi == ord.n - 1)) perm_resolve(c, g, m, nullptr);
                for (int q = c.gtid; q < m; q += c.gth) w.fixed[cand ? cand[q] : q] = 1;
                c.sync();
                cyc_perm += clock64() - t_mark;
                accepted_last = 0;
                continue;
            }
            permutation_par(c, g, m, cand, w.order, w, !base_pass);
        }
        cyc_perm += clock64() - t_mark;
        t_mark = clock64();
        if (base_pass) {
            // every candidate already has this format: the state cannot change, so all of them see the
            // same test (mixed_tile_greedy.py:238-241)
            if (!good_par(k, S, min_margin)) {
                for (int q = c.gtid; q < m; q += c.gth) w.fixed[q] = 1;
                base_failed = true;
            }
            c.sync();
            continue;
        }
        // ---- (3) accept / reject chain -------------------------------------------------------
        int pos = 0;
        bool guess = true;                      // initial guess for a chunk: accept everything
        while (pos < m) {
            const int len = min(CHc, m - pos);
            const int lo = c.gtid * EPS, hi = min(len, lo + EPS);      // this thread streams elements [lo, hi)
            const int cnt = max(0, hi - lo);
            tq = clock64();
            Grid gr[NS];
#pragma unroll
            for (int s = 0; s < NS; ++s) gr[s] = (PCC && s == 0 && relax_sy) ? make_grid_relaxed(S[0], drift) : make_grid(S[S0 + s]);
            unsigned F = guess && cnt > 0 ? (0xFFFFFFFFu >> (32 - cnt)) : 0u;     // accept flags, bit j <-> element lo + j
            unsigned D = 0;
            int valid = len;
            P2 pre0[NS];
            double st_rej[NS], st_take[NS];
#pragma unroll
            for (int s = 0; s < NS; ++s) st_rej[s] = st_take[s] = 0.0;
            bool pathological = false;
            bool any_flag = guess;             // uniform: does any element of the chunk carry an accept flag?
            int tl[EPS];                       // the tiles this thread visits in this chunk
#pragma unroll
            for (int j = 0; j < EPS; ++j) tl[j] = j < cnt ? order_ptr[pos + lo + j] : 0;
            {   // fetch the visited tiles' delta records (one 32-byte sector each)
                double2 da[EPS], db[EPS];
#pragma unroll
                for (int j = 0; j < EPS; ++j) {
                    da[j] = db[j] = make_double2(0.0, 0.0);
                    if (j < cnt) {
                        const double2* rec = reinterpret_cast<const double2*>(dtab) + 2 * (size_t)tl[j];
                        if (PCC) da[j] = rec[0];
                        db[j] = rec[1];
                    }
                }
#pragma unroll
                for (int j = 0; j < EPS; ++j) {
                    if (PCC) { staged(0, j) = da[j].x; staged(1, j) = da[j].y; staged(2, j) = db[j].x; staged(3, j) = db[j].y; }
                    else staged(0, j) = db[j].y;
                }
            }
            QA_PHASE_SYNC(); cy_load += clock64() - tq;
            for (int round = 0; round < 64; ++round) {
                ++chain_rounds;
                tq = clock64();
                // walk 1: compose the accepted elements of this thread
                P2 tot[NS];
#pragma unroll
                for (int s = 0; s < NS; ++s) tot[s] = P2{0, 0};
                int bad = 0x7FFFFFFF;           // first accepted element that cannot ride the grid
                for (int j = 0; j < cnt && lo + j < valid; ++j) {
                    if (!((F >> j) & 1u)) continue;
                    P2 p[NS];
                    bool ok = true;
#pragma unroll
                    for (int s = 0; s < NS; ++s) ok = classify(gr[s], staged(s, j), p[s]) && ok;
                    if (!ok) { bad = lo + j; break; }
#pragma unroll
                    for (int s = 0; s < NS; ++s) tot[s] = p2_then(tot[s], p[s]);
                }
                if (any_flag) scan_totals<NS>(c, tot, pre0);
                else {
#pragma unroll
                    for (int s = 0; s < NS; ++s) pre0[s] = P2{0, 0};
                }
                QA_PHASE_SYNC(); cy_scan += clock64() - tq; tq = clock64();
                // walk 2: exact state before every element -> decision; first wrong flag; first binade exit
                int mism = 0x7FFFFFFF, cut = 0x7FFFFFFF;
                D = 0;
                {
                    P2 run[NS];
#pragma unroll
                    for (int s = 0; s < NS; ++s) run[s] = pre0[s];
                    for (int j = 0; j < cnt && lo + j < valid; ++j) {
                        const int idx = lo + j;
                        double cnd[4] = {0.0, 0.0, 0.0, 0.0}, dl[NS];
#pragma unroll
                        for (int s = 0; s < NS; ++s) {
                            dl[s] = staged(s, j);
                            const double sb = gr[s].q != 0.0 ? s_of(gr[s], m_after(gr[s], run[s])) : S[S0 + s];
                            cnd[S0 + s] = __dadd_rn(sb, dl[s]);
                            st_rej[s] = sb;                 // state after this element if it is rejected / accepted:
                            st_take[s] = cnd[S0 + s];       // kept for the commit (the last element a thread walks)
                        }
                        if (PCC) cnd[3] = S[3] + staged(3, j);          // chunk-start value: only its zero test matters
                        const bool dj = good_par(k, cnd, min_margin);
                        const bool fj = (F >> j) & 1u;
                        D |= dj ? (1u << j) : 0u;
                        if (dj != fj) mism = min(mism, idx);
                        if (fj) {
                            if (idx == bad) { cut = min(cut, idx); break; }     // added for real; ends the chunk
#pragma unroll
                            for (int s = 0; s < NS; ++s) {
                                P2 p{0, 0};
                                classify(gr[s], dl[s], p);
                                run[s] = p2_then(run[s], p);
                                if (left_grid(gr[s], m_after(gr[s], run[s]))) cut = min(cut, idx);
                            }
                            if (cut == idx) break;
                        }
                    }
                }
                QA_PHASE_SYNC(); cy_dec += clock64() - tq; tq = clock64();
                // third slot: 0 if any element would carry an accept flag in the next round (F below mism, D from it on)
                const int nval = max(0, min(cnt, valid - lo));
                const int next_any = ((D | F) & (nval > 0 ? (0xFFFFFFFFu >> (32 - nval)) : 0u)) ? 0 : 0x7FFFFFFF;
                int next_any_io = next_any;
                c_min3(c, mism, cut, next_any_io);
                QA_PHASE_SYNC(); cy_min += clock64() - tq;
                cut = min(cut, valid - 1);
                if (mism > cut) { valid = cut + 1; break; }       // flags are consistent up to the cut
                if (round == 63) { valid = mism + 1; pathological = true; }   // commit up to the first wrong flag
                // fix the first wrong flag; later ones take the freshly computed decisions as the new guess
                for (int j = 0; j < cnt; ++j) {
                    const int idx = lo + j;
                    if (idx >= mism && idx < valid) F = (F & ~(1u << j)) | (D & (1u << j));
                }
                any_flag = next_any_io == 0;    // conservative (a superset of the flags actually set)
                if (round == 63) break;
            }
            // ---- commit [0, valid): D holds the decisions; pre0 the exact prefix of this thread ----
            tq = clock64();
            int loc = 0;
            bool owner = false;
            double vals[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
            double dabs = 0.0;
#pragma unroll
            for (int j = 0; j < EPS; ++j) {
                if (j < cnt && lo + j < valid) {
                    if ((D >> j) & 1u) {
                        assignment[tl[j]] = (int8_t)fmt;
                        ++loc;
                        if (PCC) dabs += staged(3, j);
                    } else w.fixed[tl[j]] = 1;
                }
            }
            if (valid - 1 >= lo && valid - 1 < lo + EPS) {       // owner of the last committed element
                owner = true;
                const int jl = valid - 1 - lo;
                const bool take = (D >> jl) & 1u;
                if (!pathological) {
                    // the last element this thread walked in the final round is valid - 1: its two outcomes are at hand
#pragma unroll
                    for (int s = 0; s < NS; ++s) vals[S0 + s] = take ? st_take[s] : st_rej[s];
                } else {
                    P2 run[NS];
#pragma unroll
                    for (int s = 0; s < NS; ++s) run[s] = pre0[s];
                    for (int j = 0; j < jl; ++j) {
                        if (!((D >> j) & 1u)) continue;
#pragma unroll
                        for (int s = 0; s < NS; ++s) {
                            P2 p{0, 0};
                            classify(gr[s], staged(s, j), p);
                            run[s] = p2_then(run[s], p);
                        }
                    }
#pragma unroll
                    for (int s = 0; s < NS; ++s) {
                        const double sb = gr[s].q != 0.0 ? s_of(gr[s], m_after(gr[s], run[s])) : S[S0 + s];
                        vals[S0 + s] = take ? __dadd_rn(sb, staged(s, jl)) : sb;
                    }
                }
                vals[4] = take ? 1.0 : 0.0;
            }
            my_accepts += loc;
            loc = __reduce_add_sync(0xFFFFFFFFu, loc);
            if ((tid & 31) == 0 && loc) { atomicAdd(&sh.cnt[fmt], loc); atomicAdd(&sh.cnt[prev], -loc); }
            double nv[5];
            const double dabs_all = c_bcast_sum_d(c, owner, vals, 5, nv, dabs);
#pragma unroll
            for (int s = 0; s < NS; ++s) S[S0 + s] = nv[S0 + s];
            if (PCC) S[3] += dabs_all;
            guess = nv[4] != 0.0;
            ++n_chunks;
            if (valid < len) ++n_cutshort;
            pos += valid;
            QA_PHASE_SYNC(); cy_commit += clock64() - tq;
        }
        if (fi + 1 < ord.n) accepted_last = (int)c_reduce_d<false>(c, (double)my_accepts);     // exact: counts < 2^53
        cyc_chain += clock64() - t_mark;
    }
    min_margin = -c_reduce_d<true>(c, -min_margin);
    if (!last) {
        // hand the running state to the next launch
        c.sync();
        if (tid < QA_NFMT && sh.cnt[tid] != 0)
            atomicAdd(reinterpret_cast<unsigned long long*>(&counts[tid]), (unsigned long long)(long long)sh.cnt[tid]);
        if (c.gtid == 0) {
            g.store(rng_out);
            double* r = w.res;
            r[0] = S[0]; r[1] = S[1]; r[2] = S[2]; r[3] = S[3];
            r[4] = (double)degraded; r[5] = (double)chain_rounds;
            r[6] = base_failed ? 1.0 : 0.0; r[7] = all_tiles_candidates ? 1.0 : 0.0; r[8] = (double)accepted_last;
            r[9] = (double)cyc_perm; r[10] = (double)cyc_chain; r[11] = done ? 1.0 : 0.0;
            r[12] = (double)n_chunks; r[13] = (double)n_cutshort; r[14] = min_margin;
            stamp(first ? 5 : 7, true);
        }
        return;
    }
    // max |x - y| of the final assignment (for the reported atol)
    c.sync();
    double amax = 0.0;
    for (int t = c.gtid; t < nt; t += c.gth) amax = fmax(amax, table[(size_t)QA_STAT_FMT(assignment[t], 4) * nt + t]);
    amax = c_reduce_d<true>(c, amax);
    __syncthreads();
    if (tid < QA_NFMT && sh.cnt[tid] != 0)
        atomicAdd(reinterpret_cast<unsigned long long*>(&counts[tid]), (unsigned long long)(long long)sh.cnt[tid]);
    if (c.gtid == 0) {
        g.store(rng_out);
        state[0] = k.sx; state[1] = k.sx2; state[2] = S[0]; state[3] = S[1]; state[4] = S[2]; state[5] = S[3];
        state[6] = (double)degraded + 65536.0 * (double)chain_rounds;
        state[7] = is_pcc ? pcc_value_par(k, S[0], S[1], S[2], S[3]) : (numel != 0.0 ? __ddiv_rn(S[3], numel) : 0.0);
        state[8] = (double)cyc_init; state[9] = (double)cyc_perm; state[10] = (double)cyc_chain;   // SM cycles per phase
        state[11] = amax;
        state[12] = (double)c.nr;
        state[13] = (double)cy_load + 1e-9 * 0; state[14] = (double)cy_scan; state[15] = (double)cy_dec;
        state[16] = (double)(clock64() - t_start); state[17] = (double)cy_commit; state[18] = (double)cy_gather;
        state[19] = (double)n_chunks; state[20] = min_margin;     // [20]: lower bound of min |value - thr| / thr over all decisions
        state[13] = w.hdr[8]; state[14] = w.hdr[9]; state[15] = w.hdr[10];
#ifdef QA_DBG_CHAIN
        printf("chain nt=%d load %lld walk1+scan %lld decide %lld min3 %lld commit %lld gather %lld | chunks %u rounds %u total %lld\n", nt, cy_load, cy_scan, cy_dec, cy_min, cy_commit, cy_gather, n_chunks, chain_rounds, (long long)(clock64() - t_start));
#endif
        state[21] = (double)c.cy_resolve; state[22] = (double)c.cy_apply; state[23] = (double)c.n_sweeps + 65536.0 * c.n_rounds;
        stamp(first ? 5 : 7, true);
    }
}

template <bool PCC>
__global__ void QA_CHAIN_REGCAP greedy_par_kernel(const double* __restrict__ table, int nt, double numel, int metric,
                                                        double thr, ParOrder ord, qa_pcg64* rng, int8_t* assignment,
                                                        int64_t* counts, double* state, ParWork w, int fi_begin, int fi_end,
                                                        int flags) {
    greedy_chain<PCC>(table, nt, numel, metric, thr, ord, rng, rng, assignment, counts, state, w, fi_begin, fi_end, flags);
}

// Sweep: cluster k runs the whole chain (passes [0, nfmt)) with thresholds[k].  Every cluster reads the one table, init
// (w.hdr / w.delta) and prefetched permutations (w.pre_order / w.pre_rng); its private buffers - the chain's scratch in w,
// its map, counts, state and the slot its stream ends in - lie `stride` bytes (work) or one row (outputs) per cluster apart,
// starting from cluster 0's.  The CTA rank inside the cluster comes from the cluster (Coop), never from blockIdx.
template <bool PCC>
__global__ void QA_CHAIN_REGCAP greedy_sweep_kernel(const double* __restrict__ table, int nt, double numel, int metric,
                                                          const double* __restrict__ thresholds, ParOrder ord, const qa_pcg64* rng,
                                                          qa_pcg64* rng_out, int8_t* assignment, int64_t* counts, double* state,
                                                          ParWork w, int64_t stride, int flags) {
    unsigned k;
    asm("mov.u32 %0, %%clusterid.x;" : "=r"(k));
    const int64_t off = (int64_t)k * stride;
    auto mine = [off](auto* p) { return reinterpret_cast<decltype(p)>(reinterpret_cast<char*>(p) + off); };
    w.order = mine(w.order); w.cand = mine(w.cand); w.jarr = mine(w.jarr); w.off = mine(w.off); w.cursor = mine(w.cursor);
    w.bucket = mine(w.bucket); w.succ = mine(w.succ); w.parent = mine(w.parent); w.res = mine(w.res); w.fixed = mine(w.fixed);
    greedy_chain<PCC>(table, nt, numel, metric, thresholds[k], ord, rng, mine(rng_out), assignment + (int64_t)k * nt,
                      counts + (int64_t)k * QA_NFMT, state + (int64_t)k * 24, w, 0, ord.n, flags);
}

// micro-benchmark of the collectives (cycles per call), for DESIGN.md / tuning
__global__ void __launch_bounds__(GT) collective_bench_kernel(double* out, int iters) {
    __shared__ Sh sh;
    Coop c(sh);
    int v = threadIdx.x & 3, tot = 0;
    bool any;
    long long t0 = clock64();
    for (int i = 0; i < iters; ++i) v = c_scan_excl_any(c, v & 3, tot, (v & 1) != 0, any) & 7;
    long long t1 = clock64();
    int a = v, b = v + 1, d = v + 2;
    for (int i = 0; i < iters; ++i) { c_min3(c, a, b, d); a += threadIdx.x & 1; }
    long long t2 = clock64();
    for (int i = 0; i < iters; ++i) c.sync();
    long long t3 = clock64();
    for (int i = 0; i < iters; ++i) __syncthreads();
    long long t4 = clock64();
    P2 tt[3] = {{v, v}, {1, 2}, {3, 3}}, pp[3];
    for (int i = 0; i < iters; ++i) { scan_totals<3>(c, tt, pp); tt[0].d0 = pp[0].d0 & 3; }
    long long t5 = clock64();
    if (c.gtid == 0) {
        out[0] = (double)(t1 - t0) / iters; out[1] = (double)(t2 - t1) / iters; out[2] = (double)(t3 - t2) / iters;
        out[3] = (double)(t4 - t3) / iters; out[4] = (double)(t5 - t4) / iters; out[5] = (double)(a + tot + pp[1].d0);
    }
}

static inline int64_t al(int64_t v) { return (v + 255) / 256 * 256; }

static ParWork carve(void* work, int64_t n) {
    ParWork w;
    char* p = reinterpret_cast<char*>(work);
    auto take = [&](int64_t bytes) { char* r = p; p += al(bytes); return r; };
    w.order = reinterpret_cast<int32_t*>(take(4 * (n + 1)));
    w.cand = reinterpret_cast<int32_t*>(take(4 * (n + 1)));
    w.jarr = reinterpret_cast<int32_t*>(take(4 * (n + 1)));
    w.off = reinterpret_cast<int32_t*>(take(4 * (n + 1)));
    w.cursor = reinterpret_cast<int32_t*>(take(4 * (n + 1)));
    w.bucket = reinterpret_cast<int32_t*>(take(4 * (n + 1)));
    w.succ = reinterpret_cast<int32_t*>(take(4 * (n + 1)));
    w.parent = reinterpret_cast<int32_t*>(take(4 * (n + 1)));
    w.fixed = reinterpret_cast<uint8_t*>(take(n));
    w.hdr = reinterpret_cast<double*>(take(8 * HDR_DOUBLES));
    w.res = reinterpret_cast<double*>(take(8 * HDR_DOUBLES));
    w.delta = reinterpret_cast<double*>(take(96 * n));
    w.pre_order = nullptr;
    w.pre_rng = nullptr;
    w.npre = 0;
    return w;
}

static thread_local int g_cluster_cap = 0;   // qa_greedy_cluster_cap: upper bound on the cluster size (0 = none), per calling thread

static int pick_cluster(int64_t n) {
    int r = 1;
    while (r < 8 && (int64_t)r * GT * DPT < n) r <<= 1;          // grow until one draw round covers the tensor
    if (n >= 65536) r = 16;                                      // opt-in (non-portable) size for the largest tensors
    return g_cluster_cap > 0 && r > g_cluster_cap ? g_cluster_cap : r;
}

// A grid of `nclusters` clusters of nr CTAs.  A grid with more clusters than can be resident at once queues: the probe below
// only asks whether one cluster of 16 fits.
template <typename... KArgs, typename... Args>
static int launch_cluster_dyn(int dyn, void (*kern)(KArgs...), int nr, int nclusters, cudaStream_t s, Args... args) {
    {   // attributes are set once per kernel (not a stream operation: keep it out of the per-launch path and of graph
        // captures); the same moment asks the occupancy calculator whether a 16-CTA cluster can be resident at all, so that
        // no launch ever has to fail and be retried (a failed launch would invalidate a stream capture)
        static std::mutex mu;
        static void* done[32];
        static bool ok16[32];
        static int ndone = 0;
        std::lock_guard<std::mutex> lock(mu);
        int idx = -1;
        for (int i = 0; i < ndone; ++i) if (done[i] == (void*)kern) idx = i;
        if (idx < 0) {
            cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
            cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, dyn);
            cudaLaunchConfig_t q = {};
            q.gridDim = dim3(16, 1, 1);
            q.blockDim = dim3(GT, 1, 1);
            q.dynamicSmemBytes = dyn;
            cudaLaunchAttribute qa_[1];
            qa_[0].id = cudaLaunchAttributeClusterDimension;
            qa_[0].val.clusterDim.x = 16;
            qa_[0].val.clusterDim.y = 1;
            qa_[0].val.clusterDim.z = 1;
            q.attrs = qa_;
            q.numAttrs = 1;
            int nclusters = 0;
            const bool fits = cudaOccupancyMaxActiveClusters(&nclusters, kern, &q) == cudaSuccess && nclusters > 0;
            (void)cudaGetLastError();
            if (ndone < 32) { done[ndone] = (void*)kern; ok16[ndone] = fits; idx = ndone++; }
            else if (!fits && nr > 8) nr = 8;
        }
        if (idx >= 0 && nr > 8 && !ok16[idx]) nr = 8;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(nr * nclusters), 1, 1);
    cfg.blockDim = dim3(GT, 1, 1);
    cfg.dynamicSmemBytes = dyn;
    cfg.stream = s;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = nr;
    at[0].val.clusterDim.y = 1;
    at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    cudaError_t e = cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
    if (e != cudaSuccess) {
        set_error("cluster launch (%d x %d CTAs): %s", nclusters, nr, cudaGetErrorString(e));
        return 2;
    }
    return 0;
}

// kernels that stage addends in dynamic shared memory (init / chain) vs. the ones that do not (permutation resolve:
// a smaller footprint is easier to place next to a streaming kernel)
template <typename... KArgs, typename... Args>
static int launch_cluster(void (*kern)(KArgs...), int nr, cudaStream_t s, Args... args) {
    return launch_cluster_dyn(STAGE_SLOTS * GT * (int)sizeof(double), kern, nr, 1, s, args...);
}
template <typename... KArgs, typename... Args>
static int launch_clusters(void (*kern)(KArgs...), int nr, int nclusters, cudaStream_t s, Args... args) {
    return launch_cluster_dyn(STAGE_SLOTS * GT * (int)sizeof(double), kern, nr, nclusters, s, args...);
}
template <typename... KArgs, typename... Args>
static int launch_cluster_nostage(void (*kern)(KArgs...), int nr, cudaStream_t s, Args... args) {
    return launch_cluster_dyn(0, kern, nr, 1, s, args...);
}

}  // namespace qa

using namespace qa;

extern "C" int qa_debug_times(unsigned long long* out8_host, int reset) {
#ifndef QA_STAMP_TIMES
    (void)out8_host; (void)reset;
    set_error("qa_debug_times: timestamps are not compiled in (build with -DQA_STAMP_TIMES)");
    return 3;
#endif
    if (out8_host && cudaMemcpyFromSymbol(out8_host, qa_times, sizeof(unsigned long long) * 40) != cudaSuccess) return check_launch("qa_debug_times");
    if (reset) {
        unsigned long long init[40];
        for (int i = 0; i < 40; ++i) init[i] = (i & 1) ? 0ull : ~0ull;
        if (cudaMemcpyToSymbol(qa_times, init, sizeof(init)) != cudaSuccess) return check_launch("qa_debug_times");
    }
    return 0;
}

extern "C" int qa_greedy_cluster_cap(int max_cluster) {
    const int prev = g_cluster_cap;
    g_cluster_cap = max_cluster < 0 ? 0 : (max_cluster > MAXR ? MAXR : max_cluster);
    return prev;
}

extern "C" int qa_collective_bench(double* out, int iters, int cluster, qa_stream_t stream) {
    return launch_cluster(collective_bench_kernel, cluster, (cudaStream_t)stream, out, iters);
}

extern "C" int64_t qa_greedy_par_work_bytes(int64_t n) { return al(4 * (n + 1)) * 8 + al(n) + 2 * al(8 * HDR_DOUBLES) + al(96 * n) + 512; }

extern "C" int64_t qa_greedy_init_bytes(int64_t n) { return al(8 * HDR_DOUBLES) + al(96 * n) + 256; }

extern "C" int qa_numpy_permutation_par(qa_pcg64* rng, int64_t n, int32_t* out_perm, void* work, qa_stream_t stream) {
    if (!rng || n < 0 || n > 0x3FFFFFFF || (n > 0 && (!out_perm || !work))) { set_error("qa_numpy_permutation_par: bad args"); return 1; }
    if (n == 0) return 0;
    return launch_cluster(permutation_par_kernel, pick_cluster(n), (cudaStream_t)stream, rng, (int)n, out_perm, carve(work, n));
}

extern "C" int qa_perm_resolve(const qa_pcg64* rng_in, int64_t n, int32_t* jarr, qa_pcg64* rng_out, qa_stream_t stream) {
    if (!rng_in || !rng_out || n <= 0 || n > 0x3FFFFFFF) { set_error("qa_perm_resolve: bad args"); return 1; }
    return launch_cluster_nostage(perm_resolve_kernel, pick_cluster(n), (cudaStream_t)stream, rng_in, (int)n, jarr, rng_out);
}

extern "C" int qa_perm_resolve_chain(const qa_pcg64* rng_in, int64_t n, int count, uint32_t write_mask, int32_t* jarr,
                                     qa_pcg64* rng_out, qa_stream_t stream) {
    if (!rng_in || !rng_out || n <= 0 || n > 0x3FFFFFFF || count < 1 || count > 32 || (write_mask && !jarr)) {
        set_error("qa_perm_resolve_chain: bad args");
        return 1;
    }
    return launch_cluster_nostage(perm_resolve_chain_kernel, pick_cluster(n), (cudaStream_t)stream, rng_in, (int)n, count, (unsigned)write_mask,
                          jarr, rng_out);
}

static int fill_order(const int32_t* fmt_order, int nfmt, ParOrder& ord, const char* who) {
    if (!fmt_order || nfmt < 1 || nfmt > QA_NFMT) { set_error("%s: bad format order", who); return 1; }
    ord.n = nfmt;
    for (int i = 0; i < QA_NFMT; ++i) ord.fmt[i] = i < nfmt ? fmt_order[i] : 0;
    for (int i = 0; i < nfmt; ++i)
        if (ord.fmt[i] < 0 || ord.fmt[i] >= QA_NFMT) { set_error("%s: bad format index", who); return 1; }
    return 0;
}

// an init buffer (qa_greedy_init_bytes) holds the header and then the delta records
static double* init_delta(const void* init) {
    return reinterpret_cast<double*>(static_cast<char*>(const_cast<void*>(init)) + al(8 * HDR_DOUBLES));
}

// On one stream: the delta records (a grid kernel) if delta != NULL, then the initial sums over tiles [t_begin, t_end) (one
// cluster) if hdr != NULL
static int greedy_init_launch(const double* table, int64_t ntiles, int metric, const int32_t* fmt_order, int nfmt, double* hdr,
                              double* delta, qa_stream_t stream, const char* who, int64_t t_begin = 0, int64_t t_end = -1) {
    if (t_end < 0) t_end = ntiles;
    if (t_begin < 0 || t_begin >= t_end || t_end > ntiles) { set_error("%s: bad tile range", who); return 1; }
    if (!table || ntiles <= 0 || ntiles > 0x3FFFFFFF || !(hdr || delta)) { set_error("%s: bad args", who); return 1; }
    if (metric != QA_METRIC_PCC && metric != QA_METRIC_MAE) { set_error("%s: metric must be pcc or mae", who); return 1; }
    ParOrder ord;
    if (fill_order(fmt_order, nfmt, ord, who)) return 1;
    cudaStream_t s = (cudaStream_t)stream;
    if (delta) {
        greedy_delta_kernel<<<(unsigned)cdiv(ntiles, 256), 256, 0, s>>>(table, (int)ntiles, ord, delta);
        if (int rc = check_launch(who)) return rc;
    }
    if (!hdr) return 0;
    if (metric == QA_METRIC_PCC)
        return launch_cluster(greedy_init_kernel<true>, pick_cluster(ntiles), s, table, (int)ntiles, ord, hdr, (int)t_begin, (int)t_end);
    return launch_cluster(greedy_init_kernel<false>, pick_cluster(ntiles), s, table, (int)ntiles, ord, hdr, (int)t_begin, (int)t_end);
}

extern "C" int qa_greedy_init_sums_range(const double* table, int64_t ntiles, int metric, const int32_t* fmt_order, int nfmt,
                                         void* init, int64_t tile_begin, int64_t tile_end, qa_stream_t stream) {
    return greedy_init_launch(table, ntiles, metric, fmt_order, nfmt, static_cast<double*>(init), nullptr, stream,
                              "qa_greedy_init_sums_range", tile_begin, tile_end);
}

extern "C" int qa_greedy_init_deltas(const double* table, int64_t ntiles, int metric, const int32_t* fmt_order, int nfmt, void* init,
                                     qa_stream_t stream) {
    return greedy_init_launch(table, ntiles, metric, fmt_order, nfmt, nullptr, init ? init_delta(init) : nullptr, stream,
                              "qa_greedy_init_deltas");
}

extern "C" int qa_greedy_init_deltas_batch(const qa_batch_desc* descs_dev, int n, int64_t total_blocks, const int32_t* fmt_order, int nfmt,
                                           qa_stream_t stream) {
    if (!descs_dev || n <= 0 || total_blocks <= 0 || total_blocks > 0x7FFFFFFF) { set_error("qa_greedy_init_deltas_batch: bad args"); return 1; }
    ParOrder ord;
    if (fill_order(fmt_order, nfmt, ord, "qa_greedy_init_deltas_batch")) return 1;
    greedy_delta_batch_kernel<<<(unsigned)total_blocks, 256, 0, (cudaStream_t)stream>>>(descs_dev, n, ord, al(8 * HDR_DOUBLES));
    return check_launch("qa_greedy_init_deltas_batch");
}

extern "C" int qa_greedy_assign_passes(const double* table, int64_t ntiles, double numel, int metric, double threshold,
                                       const int32_t* fmt_order, int nfmt, qa_pcg64* rng, int8_t* assignment,
                                       int64_t* counts, double* state, void* work, const int32_t* pre_order,
                                       const qa_pcg64* pre_rng, const void* init, int pass_begin, int pass_end, int flags,
                                       qa_stream_t stream) {
    if (pass_begin < 0 || pass_end <= pass_begin || pass_begin >= nfmt) { set_error("qa_greedy_assign_passes: bad pass range"); return 1; }
    if (!table || ntiles <= 0 || ntiles > 0x3FFFFFFF || !rng || !assignment || !counts || !state || !work) {
        set_error("qa_greedy_assign_par: bad args");
        return 1;
    }
    if (metric != QA_METRIC_PCC && metric != QA_METRIC_MAE) { set_error("qa_greedy_assign_par: metric must be pcc or mae"); return 1; }
    ParOrder ord;
    if (fill_order(fmt_order, nfmt, ord, "qa_greedy_assign_par")) return 1;
    ParWork pw = carve(work, ntiles);
    if (pre_order && pre_rng && nfmt >= 2) { pw.pre_order = pre_order; pw.pre_rng = pre_rng; pw.npre = nfmt >= 3 ? 3 : 2; }
    if (init) {
        pw.hdr = static_cast<double*>(const_cast<void*>(init));
        pw.delta = init_delta(init);
    } else if (pass_begin == 0) {
        // no init buffer: the call that runs pass 0 computes it into `work`, where the later pass ranges find it
        if (int rc = greedy_init_launch(table, ntiles, metric, fmt_order, nfmt, pw.hdr, pw.delta, stream, "qa_greedy_assign_par")) return rc;
    }
    const int nr = pick_cluster(ntiles);
    cudaStream_t cs = (cudaStream_t)stream;
    if (metric == QA_METRIC_PCC)
        return launch_cluster(greedy_par_kernel<true>, nr, cs, table, (int)ntiles, numel, metric, threshold, ord, rng, assignment, counts,
                              state, pw, pass_begin, pass_end, flags);
    return launch_cluster(greedy_par_kernel<false>, nr, cs, table, (int)ntiles, numel, metric, threshold, ord, rng, assignment, counts,
                          state, pw, pass_begin, pass_end, flags);
}

extern "C" int qa_greedy_assign_par(const double* table, int64_t ntiles, double numel, int metric, double threshold,
                                    const int32_t* fmt_order, int nfmt, qa_pcg64* rng, int8_t* assignment,
                                    int64_t* counts, double* state, void* work, qa_stream_t stream) {
    return qa_greedy_assign_passes(table, ntiles, numel, metric, threshold, fmt_order, nfmt, rng, assignment, counts, state, work,
                                   nullptr, nullptr, nullptr, 0, nfmt, 0, stream);
}

// per threshold: the chain's scratch (the single-run layout of the metric's kernel), then the slot its stream ends in
static int64_t sweep_chain_bytes(int64_t ntiles, int metric) {
    return al(metric == QA_METRIC_ATOL ? qa_greedy_work_bytes(ntiles) : qa_greedy_par_work_bytes(ntiles));
}

extern "C" int64_t qa_greedy_sweep_work_bytes(int64_t ntiles, int metric) {
    if (ntiles <= 0 || ntiles > 0x3FFFFFFF || metric < QA_METRIC_PCC || metric > QA_METRIC_ATOL) return -1;
    return sweep_chain_bytes(ntiles, metric) + al(sizeof(qa_pcg64));
}

extern "C" int qa_greedy_assign_sweep(const double* table, int64_t ntiles, double numel, int metric, const double* thresholds,
                                      int nthr, const int32_t* fmt_order, int nfmt, const qa_pcg64* rng, int8_t* assignment,
                                      int64_t* counts, double* state, void* work, const int32_t* pre_order, const qa_pcg64* pre_rng,
                                      const void* init, int flags, qa_stream_t stream) {
    const char* who = "qa_greedy_assign_sweep";
    if (!table || ntiles <= 0 || ntiles > 0x3FFFFFFF || !thresholds || nthr < 1 || !rng || !assignment || !counts || !state || !work) {
        set_error("%s: bad args", who);
        return 1;
    }
    if (metric < QA_METRIC_PCC || metric > QA_METRIC_ATOL) { set_error("%s: bad metric", who); return 1; }
    ParOrder ord;
    if (fill_order(fmt_order, nfmt, ord, who)) return 1;
    const int64_t stride = qa_greedy_sweep_work_bytes(ntiles, metric);
    char* rng_slot = static_cast<char*>(work) + sweep_chain_bytes(ntiles, metric);    // cluster / block 0's
    cudaStream_t cs = (cudaStream_t)stream;
    if (metric == QA_METRIC_ATOL)       // the one-thread chain, as for a single threshold: block k runs thresholds[k]
        return greedy_seq_sweep_launch(table, ntiles, numel, thresholds, nthr, fmt_order, nfmt, rng,
                                       reinterpret_cast<qa_pcg64*>(rng_slot), assignment, counts, state, work, stride, cs);
    const int nr = pick_cluster(ntiles);
    if ((int64_t)nthr * MAXR > 0x7FFFFFFF) { set_error("%s: too many thresholds", who); return 1; }
    ParWork pw = carve(work, ntiles);
    if (pre_order && pre_rng && nfmt >= 2) { pw.pre_order = pre_order; pw.pre_rng = pre_rng; pw.npre = nfmt >= 3 ? 3 : 2; }
    if (init) {
        pw.hdr = static_cast<double*>(const_cast<void*>(init));
        pw.delta = init_delta(init);
    } else if (int rc = greedy_init_launch(table, ntiles, metric, fmt_order, nfmt, pw.hdr, pw.delta, stream, who)) {
        return rc;       // computed once, into the first chain's work, where every chain reads it
    }
    if (metric == QA_METRIC_PCC)
        return launch_clusters(greedy_sweep_kernel<true>, nr, nthr, cs, table, (int)ntiles, numel, metric, thresholds, ord, rng,
                               reinterpret_cast<qa_pcg64*>(rng_slot), assignment, counts, state, pw, stride, flags);
    return launch_clusters(greedy_sweep_kernel<false>, nr, nthr, cs, table, (int)ntiles, numel, metric, thresholds, ord, rng,
                           reinterpret_cast<qa_pcg64*>(rng_slot), assignment, counts, state, pw, stride, flags);
}
