// Whole-tensor NumPy-float32-faithful scores: the numbers wq prints (wq:684-687), the sweep writes
// (scripts/sweep_mixed_tile_threshold.py:746-749) and mixed-tile-random records per sample
// (mixed_tile_random.py:137-141), i.e. metrics.py:6-27 on the flattened tensors, float32 end to end:
//
//   np.mean(a), np.mean(|a-b|) : np.add.reduce = pairwise sum.  Leaves of <= 128 elements with 8 strided accumulators,
//                                ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)), then the n%8 tail one by one; longer ranges split at
//                                n/2 rounded down to a multiple of 8.  The tree depends on n only: qa_pairwise_plan_build
//                                lays it out once per n on the host (leaves + internal nodes, deepest level first).
//   np.dot (OpenBLAS 0.3.30 SkylakeX sdot): n & -32 elements through the vector kernel - blocks of 64 into 64 FMA chains
//                                (element i -> chain i % 64), lanes l / l+8 added, an odd block of 32 as one more FMA into
//                                the 4 x 8 lanes, ((A0+A1)+A2)+A3, lanes l / l+4, (v0+v1)+(v2+v3) - and the last n % 32
//                                elements as float32 products accumulated in a double that starts at 0; float(tail + kernel).
//   pearson_corr               : am = a - mean(a), bm = b - mean(b) (float32), sqrt(dot(am,am)) * sqrt(dot(bm,bm)),
//                                dot(am,bm) / denom, all float32, with the denom == 0 branch on max|a-b|.
//
// The FMA chains are sequential by definition (one rounding per element): each of the 64 chains is one thread, the
// parallelism is across the three dot products, across tensors / formats / samples (the batch dimension), not inside a chain.
#include <vector>
#include <algorithm>

#include "qa_common.cuh"

namespace qa {

struct PlanNode { int64_t off, n; int32_t left, right, depth; };

static int32_t plan_rec(std::vector<PlanNode>& nodes, int64_t off, int64_t n, int depth) {
    const int32_t id = (int32_t)nodes.size();
    nodes.push_back(PlanNode{off, n, -1, -1, depth});
    if (n > 128) {
        int64_t n2 = n / 2;
        n2 -= n2 % 8;
        const int32_t l = plan_rec(nodes, off, n2, depth + 1);
        const int32_t r = plan_rec(nodes, off + n2, n - n2, depth + 1);
        nodes[id].left = l;
        nodes[id].right = r;
    }
    return id;
}

// plan words: [0] nleaves [1] nlevels [2] nnodes [3] ninternal [4 .. 4+nlevels] level offsets (nlevels+1 entries, into
// the internal arrays) | leaf_start8[nleaves] | leaf_len[nleaves] | left[ninternal] | right[ninternal]
// node ids: leaves 0..nleaves-1 in element order, internal nodes nleaves + k in evaluation order (deepest first); the
// root is the last node.
static void plan_counts(int64_t n, int64_t& nleaves, int64_t& ninternal, int& nlevels) {
    // the recursion is cheap enough to run twice (2 n / 100 nodes); keeps the size query allocation-free in spirit
    std::vector<PlanNode> nodes;
    nodes.reserve((size_t)(n / 40 + 8));
    plan_rec(nodes, 0, n, 0);
    nleaves = ninternal = 0;
    int maxd = 0;
    for (auto& nd : nodes) {
        if (nd.left < 0) ++nleaves; else { ++ninternal; maxd = std::max(maxd, nd.depth); }
    }
    nlevels = ninternal ? maxd + 1 : 0;
}

template <int DT>
__device__ __forceinline__ float ld_elem(const void* p, int64_t i) {
    if (DT == QA_DT_BF16) return __uint_as_float((uint32_t)reinterpret_cast<const uint16_t*>(p)[i] << 16);
    return reinterpret_cast<const float*>(p)[i];
}
__device__ __forceinline__ float ld_any(const void* p, int dt, int64_t i) {
    if (!p) return 0.f;
    return dt == QA_DT_BF16 ? ld_elem<QA_DT_BF16>(p, i) : ld_elem<QA_DT_F32>(p, i);
}

// ---- pairwise leaves: 8 lanes per leaf, 4 leaves per warp ------------------------------------------------
__global__ void __launch_bounds__(256) pw_leaf_kernel(const void* __restrict__ x, int xdt, const void* __restrict__ ybase, int ydt,
                                                      int64_t y_stride, int64_t nleaves, int64_t nnodes,
                                                      const int32_t* __restrict__ leaf_start8, const int32_t* __restrict__ leaf_len,
                                                      float* __restrict__ vals, unsigned* __restrict__ maxbits, int b0) {
    const int b = b0 + (int)blockIdx.y;
    const char* yb = reinterpret_cast<const char*>(ybase);
    const void* y = ybase ? (const void*)(yb + (size_t)b * (size_t)y_stride * (ydt == QA_DT_BF16 ? 2 : 4)) : nullptr;
    float* v = vals + (size_t)b * 3 * nnodes;
    const int lane = threadIdx.x & 31, k = lane & 7;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    float mx = 0.f;
    bool mxnan = false;
    for (int64_t base = warp * 4; base < nleaves; base += nwarps * 4) {
        const int64_t leaf = base + (lane >> 3);
        const bool live = leaf < nleaves;
        const int64_t s = live ? (int64_t)leaf_start8[leaf] * 8 : 0;
        const int len = live ? leaf_len[leaf] : 0;
        float rx = 0.f, ry = 0.f, rd = 0.f;
        if (len >= 8) {
            const int len8 = len - (len & 7);
            for (int i = 0; i < len8; i += 8) {
                const float xv = ld_any(x, xdt, s + i + k), yv = ld_any(y, ydt, s + i + k);
                const float d = fabsf(__fsub_rn(xv, yv));
                if (i == 0) { rx = xv; ry = yv; rd = d; }
                else { rx = __fadd_rn(rx, xv); ry = __fadd_rn(ry, yv); rd = __fadd_rn(rd, d); }
                if (d != d) mxnan = true;
                mx = fmaxf(mx, d);
            }
        }
        // ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)): butterfly over the 8 lanes of the leaf (same order on every lane)
#pragma unroll
        for (int o = 1; o < 8; o <<= 1) {
            const float ox = __shfl_xor_sync(0xFFFFFFFFu, rx, o), oy = __shfl_xor_sync(0xFFFFFFFFu, ry, o),
                        od = __shfl_xor_sync(0xFFFFFFFFu, rd, o);
            // lower lane holds the left operand: a + b with a from the lane whose bit o is clear
            const bool lo = !(k & o);
            rx = lo ? __fadd_rn(rx, ox) : __fadd_rn(ox, rx);
            ry = lo ? __fadd_rn(ry, oy) : __fadd_rn(oy, ry);
            rd = lo ? __fadd_rn(rd, od) : __fadd_rn(od, rd);
        }
        if (live && k == 0) {
            int i0 = len - (len & 7);
            if (len < 8) { rx = ry = rd = 0.f; i0 = 0; }
            for (int i = i0; i < len; ++i) {      // tail (and the n < 8 case) one by one
                const float xv = ld_any(x, xdt, s + i), yv = ld_any(y, ydt, s + i);
                const float d = fabsf(__fsub_rn(xv, yv));
                rx = __fadd_rn(rx, xv); ry = __fadd_rn(ry, yv); rd = __fadd_rn(rd, d);
                if (d != d) mxnan = true;
                mx = fmaxf(mx, d);
            }
            v[leaf] = rx; v[nnodes + leaf] = ry; v[2 * nnodes + leaf] = rd;
        }
    }
    // np.max propagates NaN; as unsigned bit patterns a (positive) NaN orders above +inf
    unsigned mb = mxnan ? 0x7FC00000u : __float_as_uint(mx);
#pragma unroll
    for (int o = 16; o; o >>= 1) mb = max(mb, __shfl_xor_sync(0xFFFFFFFFu, mb, o));
    if (lane == 0 && mb) atomicMax(&maxbits[b], mb);
}

// ---- pairwise leaves, vector form: one thread per leaf, 8 elements (= the 8 strided accumulators) per load --------------
// Used when every operand is 16-byte aligned at every leaf start (leaf starts are multiples of 8 elements).  YDT == 2: y = 0.
template <int DT>
__device__ __forceinline__ void ld8(const void* p, int64_t i, float (&v)[8]) {
    if (DT == QA_DT_BF16) {
        const uint4 w = __ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const uint16_t*>(p) + i));
        const uint32_t u[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) { v[2 * k] = __uint_as_float(u[k] << 16); v[2 * k + 1] = __uint_as_float(u[k] & 0xFFFF0000u); }
    } else {
        const float4 a = __ldg(reinterpret_cast<const float4*>(reinterpret_cast<const float*>(p) + i));
        const float4 b = __ldg(reinterpret_cast<const float4*>(reinterpret_cast<const float*>(p) + i) + 1);
        v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
    }
}
template <int XDT, int YDT>
__global__ void __launch_bounds__(128) pw_leaf_vec_kernel(const void* __restrict__ x, const void* __restrict__ ybase, int64_t y_stride,
                                                          int64_t nleaves, int64_t nnodes, const int32_t* __restrict__ leaf_start8,
                                                          const int32_t* __restrict__ leaf_len, float* __restrict__ vals,
                                                          unsigned* __restrict__ maxbits, int b0) {
    const int b = b0 + (int)blockIdx.y;
    const void* y = YDT == 2 ? nullptr
                             : (const void*)(reinterpret_cast<const char*>(ybase) + (size_t)b * (size_t)y_stride * (YDT == QA_DT_BF16 ? 2 : 4));
    float* v = vals + (size_t)b * 3 * nnodes;
    unsigned mb = 0;
    for (int64_t leaf = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; leaf < nleaves; leaf += (int64_t)gridDim.x * blockDim.x) {
        const int64_t s = (int64_t)leaf_start8[leaf] * 8;
        const int len = leaf_len[leaf];
        const int len8 = len - (len & 7);
        float rx[8], ry[8], rd[8];
        float sx = 0.f, sy = 0.f, sd = 0.f;
        if (len8) {
            for (int i = 0; i < len8; i += 8) {
                float xv[8], yv[8];
                ld8<XDT>(x, s + i, xv);
                if (YDT == 2) {
#pragma unroll
                    for (int k = 0; k < 8; ++k) yv[k] = 0.f;
                } else ld8<YDT == 2 ? QA_DT_F32 : YDT>(y, s + i, yv);
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    const float d = fabsf(__fsub_rn(xv[k], yv[k]));
                    mb = max(mb, __float_as_uint(d));                     // NaN patterns order above +inf: np.max propagates them
                    if (i == 0) { rx[k] = xv[k]; ry[k] = yv[k]; rd[k] = d; }
                    else { rx[k] = __fadd_rn(rx[k], xv[k]); ry[k] = __fadd_rn(ry[k], yv[k]); rd[k] = __fadd_rn(rd[k], d); }
                }
            }
            sx = __fadd_rn(__fadd_rn(__fadd_rn(rx[0], rx[1]), __fadd_rn(rx[2], rx[3])), __fadd_rn(__fadd_rn(rx[4], rx[5]), __fadd_rn(rx[6], rx[7])));
            sy = __fadd_rn(__fadd_rn(__fadd_rn(ry[0], ry[1]), __fadd_rn(ry[2], ry[3])), __fadd_rn(__fadd_rn(ry[4], ry[5]), __fadd_rn(ry[6], ry[7])));
            sd = __fadd_rn(__fadd_rn(__fadd_rn(rd[0], rd[1]), __fadd_rn(rd[2], rd[3])), __fadd_rn(__fadd_rn(rd[4], rd[5]), __fadd_rn(rd[6], rd[7])));
        }
        for (int i = len < 8 ? 0 : len8; i < len; ++i) {                 // tail (and the n < 8 case) one by one
            const float xv = ld_elem<XDT>(x, s + i);
            const float yv = YDT == 2 ? 0.f : ld_elem<YDT == 2 ? QA_DT_F32 : YDT>(y, s + i);
            const float d = fabsf(__fsub_rn(xv, yv));
            mb = max(mb, __float_as_uint(d));
            sx = __fadd_rn(sx, xv); sy = __fadd_rn(sy, yv); sd = __fadd_rn(sd, d);
        }
        v[leaf] = sx; v[nnodes + leaf] = sy; v[2 * nnodes + leaf] = sd;
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) mb = max(mb, __shfl_xor_sync(0xFFFFFFFFu, mb, o));
    if ((threadIdx.x & 31) == 0 && mb) atomicMax(&maxbits[b], mb);
}

// ---- pairwise tree: one CTA per batch item, deepest level first -------------------------------------------
__global__ void __launch_bounds__(1024) pw_tree_kernel(int64_t nleaves, int64_t nnodes, int nlevels, const int32_t* __restrict__ level_off,
                                                       const int32_t* __restrict__ left, const int32_t* __restrict__ right,
                                                       float* __restrict__ vals) {
    float* v = vals + (size_t)blockIdx.x * 3 * nnodes;
    for (int L = 0; L < nlevels; ++L) {
        const int32_t e = level_off[L + 1];
        for (int32_t i = level_off[L] + threadIdx.x; i < e; i += blockDim.x) {
            const int32_t l = left[i], r = right[i];
#pragma unroll
            for (int q = 0; q < 3; ++q) v[q * nnodes + nleaves + i] = __fadd_rn(v[q * nnodes + l], v[q * nnodes + r]);
        }
        __syncthreads();
    }
}

// ---- sdot chains: block = 64 threads = the 64 accumulators of one dot product ------------------------------
template <int XDT, int YDT>
__global__ void __launch_bounds__(64) sdot_kernel(const void* __restrict__ x, const void* __restrict__ ybase, int64_t y_stride,
                                                  int64_t n, int64_t nnodes, const float* __restrict__ vals, float* __restrict__ dots,
                                                  int b0) {
    const int kind = blockIdx.x;     // 0: (am, am)  1: (bm, bm)  2: (am, bm)
    const int b = b0 + (int)blockIdx.y;
    if (kind == 0 && b > 0) return;  // x is shared by the batch
    const void* y = ybase ? (const void*)(reinterpret_cast<const char*>(ybase) + (size_t)b * (size_t)y_stride * (YDT == QA_DT_BF16 ? 2 : 4))
                          : nullptr;
    const float fn = (float)n;
    const float mean_x = __fdiv_rn(vals[nnodes - 1], fn);
    const float mean_y = __fdiv_rn(vals[(size_t)b * 3 * nnodes + nnodes + nnodes - 1], fn);
    const int t = threadIdx.x;
    const int64_t n1 = n & ~(int64_t)31, n64 = n1 & ~(int64_t)63;
    auto U = [&](int64_t i) -> float {
        if (kind == 1) return __fsub_rn(y ? ld_elem<YDT>(y, i) : 0.f, mean_y);
        return __fsub_rn(ld_elem<XDT>(x, i), mean_x);
    };
    auto V = [&](int64_t i) -> float {
        if (kind == 0) return __fsub_rn(ld_elem<XDT>(x, i), mean_x);
        return __fsub_rn(y ? ld_elem<YDT>(y, i) : 0.f, mean_y);
    };
    float acc = 0.f;
    int64_t i = t;
    constexpr int UN = 8;
    for (; i + (UN - 1) * 64 < n64; i += UN * 64) {
        float u[UN], v[UN];
#pragma unroll
        for (int k = 0; k < UN; ++k) { u[k] = U(i + k * 64); v[k] = V(i + k * 64); }
#pragma unroll
        for (int k = 0; k < UN; ++k) acc = __fmaf_rn(u[k], v[k], acc);
    }
    for (; i < n64; i += 64) acc = __fmaf_rn(U(i), V(i), acc);
    __shared__ float sacc[64];
    __shared__ float sh[32];
    sacc[t] = acc;
    __syncthreads();
    if (t < 32) {
        const int a = t >> 3, l = t & 7;
        float h = __fadd_rn(sacc[a * 16 + l], sacc[a * 16 + l + 8]);
        if (n1 - n64 == 32) h = __fmaf_rn(U(n64 + 8 * a + l), V(n64 + 8 * a + l), h);
        sh[t] = h;
    }
    __syncthreads();
    if (t == 0) {
        float s[8];
#pragma unroll
        for (int l = 0; l < 8; ++l) s[l] = __fadd_rn(__fadd_rn(__fadd_rn(sh[l], sh[8 + l]), sh[16 + l]), sh[24 + l]);
        float q[4];
#pragma unroll
        for (int l = 0; l < 4; ++l) q[l] = __fadd_rn(s[l], s[l + 4]);
        const float kern = __fadd_rn(__fadd_rn(q[0], q[1]), __fadd_rn(q[2], q[3]));
        float res = kern;
        if (n1 < n) {
            double tail = 0.0;
            for (int64_t j = n1; j < n; ++j) tail = __dadd_rn(tail, (double)__fmul_rn(V(j), U(j)));
            res = (float)__dadd_rn(tail, (double)kern);
        }
        dots[(size_t)b * 4 + kind] = res;
    }
}

// ---- sdot chains, pipelined.  The 64 chains of one dot product are sequential by definition (element i feeds chain i % 64 with
// one fused multiply-add), so a dot product is one CTA of 64 threads whatever the tensor size, and the job is to keep those two
// warps issuing nothing but the chain's own work: LDS, unpack, centre (x - mean in float32, the reference's `a - np.mean(a)`),
// FFMA - seven instructions per element for a bf16 pair.  Operands arrive through the TMA engine: thread 0 issues one bulk copy
// (cp.async.bulk, 8 - 16 KB) per operand and 4096-element stage into a shared-memory ring and every stage completes on its own
// mbarrier, so no warp spends issue slots on address arithmetic or per-16-byte copy requests, and up to eight stages are in
// flight.  Measured per SM on o_proj-size operands: LDGSTS (cp.async) streaming sustains 38 GB/s = 840 cycles per bf16-pair
// stage, the bulk copies 56 GB/s = 570 cycles, the chains themselves 1 250 cycles (see sd_stage): 33 -> 20 ms per call.
constexpr int SD_TE = 4096;                 // elements per stage (64 chain steps)
constexpr int SD_MAX_STAGES = 8;

__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_wait(unsigned bar, unsigned parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "SD_WAIT:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra SD_DONE;\n\t"
        "bra SD_WAIT;\n\t"
        "SD_DONE:\n\t}" ::"r"(bar), "r"(parity) : "memory");
}
template <int DT>
__device__ __forceinline__ float lds_elem(const unsigned char* base, int i) {
    if (DT == QA_DT_BF16) return __uint_as_float((uint32_t)reinterpret_cast<const uint16_t*>(base)[i] << 16);
    return reinterpret_cast<const float*>(base)[i];
}

// One 4096-element stage of one chain: 64 dependent FFMAs; the operands of the next 16 steps are requested before the chain
// runs through the present 16.  SAME: both operands are the same tensor (a.a, b.b); ZERO_V: the second operand is all zeros
// (fp0).  Measured (profiles/r2_scorer_time.txt): 18 - 20 cycles per step for a bf16 pair - a lone warp per SM sub-partition
// issues its seven instructions per step at about one every two cycles, and ptxas keeps only ~6 shared-memory loads in flight
// (one per scoreboard), whatever order the source asks for (an explicit volatile-asm pipeline compiled to the same schedule).
template <int UDT, int VDT, bool SAME, bool ZERO_V>
__device__ __forceinline__ float sd_stage(const unsigned char* su, const unsigned char* sv, int t, float mean_u, float mean_v, float acc) {
    constexpr int BL = 16;
    float ru[BL], rv[BL];
#pragma unroll
    for (int k = 0; k < BL; ++k) {
        ru[k] = lds_elem<UDT>(su, k * 64 + t);
        rv[k] = (SAME || ZERO_V) ? 0.f : lds_elem<VDT>(sv, k * 64 + t);
    }
#pragma unroll
    for (int blk = 0; blk < SD_TE / 64 / BL; ++blk) {
        float u[BL], v[BL];
#pragma unroll
        for (int k = 0; k < BL; ++k) {
            u[k] = __fsub_rn(ru[k], mean_u);
            v[k] = SAME ? u[k] : __fsub_rn(rv[k], mean_v);
        }
        if (blk + 1 < SD_TE / 64 / BL) {
#pragma unroll
            for (int k = 0; k < BL; ++k) {
                ru[k] = lds_elem<UDT>(su, ((blk + 1) * BL + k) * 64 + t);
                rv[k] = (SAME || ZERO_V) ? 0.f : lds_elem<VDT>(sv, ((blk + 1) * BL + k) * 64 + t);
            }
        }
#pragma unroll
        for (int k = 0; k < BL; ++k) acc = __fmaf_rn(u[k], v[k], acc);
    }
    return acc;
}

template <int XDT, int YDT>      // YDT == 2: y is all zeros (never loaded)
__global__ void __launch_bounds__(64, 1) sdot_pipe_kernel(const void* __restrict__ x, const void* __restrict__ ybase, int64_t y_stride, int64_t n,
                                                       int64_t nnodes, int nstages, const float* __restrict__ vals,
                                                       float* __restrict__ dots, int b0) {
    extern __shared__ __align__(128) unsigned char sd_smem[];
    __shared__ __align__(8) unsigned long long full[SD_MAX_STAGES];
    const int kind = blockIdx.x;     // 0: (am, am)  1: (bm, bm)  2: (am, bm)
    const int b = b0 + (int)blockIdx.y;
    if (kind == 0 && b > 0) return;  // x is shared by the batch
    constexpr int XB = XDT == QA_DT_BF16 ? 2 : 4, YB = YDT == QA_DT_BF16 ? 2 : 4;
    constexpr bool HAVE_Y = YDT != 2;
    constexpr int YD = HAVE_Y ? YDT : QA_DT_F32;
    const unsigned char* xg = reinterpret_cast<const unsigned char*>(x);
    const unsigned char* yg = HAVE_Y ? reinterpret_cast<const unsigned char*>(ybase) + (size_t)b * (size_t)y_stride * YB : nullptr;
    const bool need_x = kind != 1, need_y = HAVE_Y && kind != 0;
    const int stage_bytes = SD_TE * (XB + (HAVE_Y ? YB : 0));
    const float fn = (float)n;
    const float mean_x = __fdiv_rn(vals[nnodes - 1], fn);
    const float mean_y = __fdiv_rn(vals[(size_t)b * 3 * nnodes + nnodes + nnodes - 1], fn);
    const int t = threadIdx.x;
    const int64_t n1 = n & ~(int64_t)31, n64 = n1 & ~(int64_t)63;
    const int64_t ntile = n64 / SD_TE;
    float acc = 0.f;
    if (kind == 1 && !HAVE_Y) {
        // y = 0: b - mean(b) = 0 everywhere, the chains stay at 0
    } else {
        if (t == 0) {
            for (int s_ = 0; s_ < nstages; ++s_) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&full[s_])) : "memory");
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        }
        __syncthreads();
        // thread 0: arm the stage's barrier with its byte count, then one bulk copy per operand
        auto issue = [&](int64_t tile) {
            const int slot = (int)(tile % nstages);
            const unsigned bar = smem_u32(&full[slot]);
            unsigned char* st = sd_smem + (size_t)slot * stage_bytes;
            const unsigned bytes = (need_x ? SD_TE * XB : 0) + (need_y ? SD_TE * YB : 0);
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
            if (need_x)
                asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(st)),
                             "l"(xg + (size_t)tile * SD_TE * XB), "r"((unsigned)(SD_TE * XB)), "r"(bar)
                             : "memory");
            if (need_y)
                asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                                 smem_u32(st + SD_TE * XB)),
                             "l"(yg + (size_t)tile * SD_TE * YB), "r"((unsigned)(SD_TE * YB)), "r"(bar)
                             : "memory");
        };
        if (t == 0)
            for (int p = 0; p < nstages && p < ntile; ++p) issue(p);
        int slot = 0;
        unsigned parity = 0;
        for (int64_t tile = 0; tile < ntile; ++tile) {
            mbar_wait(smem_u32(&full[slot]), parity);      // the stage's bytes have landed
            const unsigned char* st = sd_smem + (size_t)slot * stage_bytes;
            if (kind == 0) acc = sd_stage<XDT, XDT, true, false>(st, st, t, mean_x, mean_x, acc);
            else if (kind == 1) acc = sd_stage<YD, YD, true, false>(st + SD_TE * XB, st + SD_TE * XB, t, mean_y, mean_y, acc);
            else acc = HAVE_Y ? sd_stage<XDT, YD, false, false>(st, st + SD_TE * XB, t, mean_x, mean_y, acc)
                              : sd_stage<XDT, YD, false, true>(st, st, t, mean_x, mean_y, acc);
            __syncthreads();                               // both warps are done with the slot
            if (t == 0 && tile + nstages < ntile) issue(tile + nstages);
            if (++slot == nstages) { slot = 0; parity ^= 1u; }
        }
    }
    auto U = [&](int64_t i) -> float {
        if (kind == 1) return __fsub_rn(HAVE_Y ? ld_elem<YD>(yg, i) : 0.f, mean_y);
        return __fsub_rn(ld_elem<XDT>(xg, i), mean_x);
    };
    auto V = [&](int64_t i) -> float {
        if (kind == 0) return __fsub_rn(ld_elem<XDT>(xg, i), mean_x);
        return __fsub_rn(HAVE_Y ? ld_elem<YD>(yg, i) : 0.f, mean_y);
    };
    __shared__ float sacc[64];
    __shared__ float sh[32];
    for (int64_t i = ntile * SD_TE + t; i < n64; i += 64) acc = __fmaf_rn(U(i), V(i), acc);     // < 64 leftover steps
    sacc[t] = acc;
    __syncthreads();
    if (t < 32) {
        const int a = t >> 3, l = t & 7;
        float h = __fadd_rn(sacc[a * 16 + l], sacc[a * 16 + l + 8]);
        if (n1 - n64 == 32) h = __fmaf_rn(U(n64 + 8 * a + l), V(n64 + 8 * a + l), h);
        sh[t] = h;
    }
    __syncthreads();
    if (t == 0) {
        float s8[8];
#pragma unroll
        for (int l = 0; l < 8; ++l) s8[l] = __fadd_rn(__fadd_rn(__fadd_rn(sh[l], sh[8 + l]), sh[16 + l]), sh[24 + l]);
        float q[4];
#pragma unroll
        for (int l = 0; l < 4; ++l) q[l] = __fadd_rn(s8[l], s8[l + 4]);
        const float kern = __fadd_rn(__fadd_rn(q[0], q[1]), __fadd_rn(q[2], q[3]));
        float res = kern;
        if (n1 < n) {
            double tail = 0.0;
            for (int64_t j = n1; j < n; ++j) tail = __dadd_rn(tail, (double)__fmul_rn(V(j), U(j)));
            res = (float)__dadd_rn(tail, (double)kern);
        }
        dots[(size_t)b * 4 + kind] = res;
    }
}

__global__ void scores_final_kernel(int nbatch, int64_t n, int64_t nnodes, const float* __restrict__ vals, const float* __restrict__ dots,
                                    const unsigned* __restrict__ maxbits, float* __restrict__ out) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nbatch) return;
    const float amax = __uint_as_float(maxbits[b]);
    const float na = __fsqrt_rn(dots[0]), nb = __fsqrt_rn(dots[(size_t)b * 4 + 1]);
    const float denom = __fmul_rn(na, nb);
    float pcc;
    if (denom == 0.f) pcc = (amax == 0.f) ? 1.f : 0.f;
    else pcc = __fdiv_rn(dots[(size_t)b * 4 + 2], denom);
    out[(size_t)b * 4 + 0] = pcc;
    out[(size_t)b * 4 + 1] = __fdiv_rn(vals[(size_t)b * 3 * nnodes + 2 * nnodes + nnodes - 1], (float)n);
    out[(size_t)b * 4 + 2] = amax;
    out[(size_t)b * 4 + 3] = __fdiv_rn(vals[(size_t)b * 3 * nnodes + nnodes + nnodes - 1], (float)n);   // mean(b), for reference
}

}  // namespace qa

using namespace qa;

extern "C" int64_t qa_pairwise_plan_words(int64_t n) {
    if (n <= 0) return 0;
    int64_t nl, ni;
    int lv;
    plan_counts(n, nl, ni, lv);
    return 4 + (lv + 1) + 2 * nl + 2 * ni;
}

extern "C" int qa_pairwise_plan_build(int64_t n, int32_t* plan) {
    if (n <= 0 || !plan) { set_error("qa_pairwise_plan_build: bad args"); return 1; }
    if (n / 8 > 0x7FFFFFFFll) { set_error("qa_pairwise_plan_build: n too large"); return 1; }
    std::vector<PlanNode> nodes;
    nodes.reserve((size_t)(n / 40 + 8));
    plan_rec(nodes, 0, n, 0);
    std::vector<int32_t> leaf_ids, internal;
    int maxd = 0;
    for (int32_t i = 0; i < (int32_t)nodes.size(); ++i) {
        if (nodes[i].left < 0) leaf_ids.push_back(i);
        else { internal.push_back(i); maxd = std::max(maxd, nodes[i].depth); }
    }
    // leaves are created in element order by the pre-order recursion (left before right)
    std::stable_sort(internal.begin(), internal.end(), [&](int32_t a, int32_t b) { return nodes[a].depth > nodes[b].depth; });
    const int64_t nl = (int64_t)leaf_ids.size(), ni = (int64_t)internal.size();
    const int lv = ni ? maxd + 1 : 0;
    std::vector<int32_t> newid(nodes.size());
    for (int64_t i = 0; i < nl; ++i) newid[leaf_ids[i]] = (int32_t)i;
    for (int64_t i = 0; i < ni; ++i) newid[internal[i]] = (int32_t)(nl + i);
    plan[0] = (int32_t)nl; plan[1] = lv; plan[2] = (int32_t)(nl + ni); plan[3] = (int32_t)ni;
    int32_t* loff = plan + 4;
    int32_t* ls = loff + lv + 1;
    int32_t* ll = ls + nl;
    int32_t* lf = ll + nl;
    int32_t* rt = lf + ni;
    for (int64_t i = 0; i < nl; ++i) { ls[i] = (int32_t)(nodes[leaf_ids[i]].off / 8); ll[i] = (int32_t)nodes[leaf_ids[i]].n; }
    int level = 0;
    loff[0] = 0;
    for (int64_t i = 0; i < ni; ++i) {
        const int d = maxd - nodes[internal[i]].depth;       // evaluation level 0 = deepest
        while (level < d) loff[++level] = (int32_t)i;
        lf[i] = newid[nodes[internal[i]].left];
        rt[i] = newid[nodes[internal[i]].right];
    }
    while (level < lv) loff[++level] = (int32_t)ni;
    return 0;
}

extern "C" int64_t qa_tensor_scores_work_bytes(int64_t plan_nnodes, int nbatch) {
    if (plan_nnodes <= 0 || nbatch <= 0) return 0;
    return (int64_t)nbatch * (3 * plan_nnodes * 4 + 32);
}

extern "C" int qa_tensor_scores_f32(const void* x, int x_dtype, const void* y, int y_dtype, int64_t y_stride, int nbatch, int64_t n,
                                    const int32_t* plan_dev, const int32_t* plan_head_host, float* out, void* work, qa_stream_t stream) {
    if (!x || n <= 0 || nbatch <= 0 || !plan_dev || !plan_head_host || !out || !work) { set_error("qa_tensor_scores_f32: bad args"); return 1; }
    if ((x_dtype != QA_DT_BF16 && x_dtype != QA_DT_F32) || (y && y_dtype != QA_DT_BF16 && y_dtype != QA_DT_F32)) {
        set_error("qa_tensor_scores_f32: bad dtype");
        return 1;
    }
    cudaStream_t s = (cudaStream_t)stream;
    const int64_t nl = plan_head_host[0], nnodes = plan_head_host[2];
    const int lv = plan_head_host[1];
    const int32_t* loff = plan_dev + 4;
    const int32_t* ls = loff + lv + 1;
    const int32_t* ll = ls + nl;
    const int32_t* lf = ll + nl;
    const int32_t* rt = lf + plan_head_host[3];
    float* vals = reinterpret_cast<float*>(work);
    float* dots = vals + (size_t)nbatch * 3 * nnodes;
    unsigned* maxbits = reinterpret_cast<unsigned*>(dots + (size_t)nbatch * 4);
    cudaMemsetAsync(dots, 0, (size_t)nbatch * 32, s);
    const size_t ybytes = y_dtype == QA_DT_BF16 ? 2 : 4;
    const bool aligned = reinterpret_cast<uintptr_t>(x) % 32 == 0 &&
                         (!y || (reinterpret_cast<uintptr_t>(y) % 32 == 0 && ((size_t)y_stride * ybytes) % 32 == 0));
    // The leaf and chain kernels put the batch on gridDim.y, which CUDA caps at 65535: they are launched over batch ranges
    // [b0, b0 + nb) of at most that many items.  pw_tree_kernel and scores_final_kernel put the batch on gridDim.x.
    constexpr int max_y = 65535;
    const int yk = y ? y_dtype : 2;
    if (aligned) {
        const unsigned gx = (unsigned)std::max<int64_t>(1, std::min<int64_t>(cdiv(nl, 128), 148 * 16));
        for (int b0 = 0; b0 < nbatch; b0 += max_y) {
            const dim3 gv(gx, std::min(nbatch - b0, max_y));
#define QA_LEAF(XD, YD) pw_leaf_vec_kernel<XD, YD><<<gv, 128, 0, s>>>(x, y, y_stride, nl, nnodes, ls, ll, vals, maxbits, b0)
            if (x_dtype == QA_DT_BF16) { if (yk == QA_DT_BF16) QA_LEAF(QA_DT_BF16, QA_DT_BF16); else if (yk == QA_DT_F32) QA_LEAF(QA_DT_BF16, QA_DT_F32); else QA_LEAF(QA_DT_BF16, 2); }
            else { if (yk == QA_DT_BF16) QA_LEAF(QA_DT_F32, QA_DT_BF16); else if (yk == QA_DT_F32) QA_LEAF(QA_DT_F32, QA_DT_F32); else QA_LEAF(QA_DT_F32, 2); }
#undef QA_LEAF
        }
    } else {
        const int64_t warps_needed = cdiv(nl, 4);
        const unsigned gx = (unsigned)std::max<int64_t>(1, std::min<int64_t>(cdiv(warps_needed, 8), 148 * 8));
        for (int b0 = 0; b0 < nbatch; b0 += max_y)
            pw_leaf_kernel<<<dim3(gx, std::min(nbatch - b0, max_y)), 256, 0, s>>>(x, x_dtype, y, y_dtype, y_stride, nl, nnodes, ls, ll,
                                                                                  vals, maxbits, b0);
    }
    if (lv) pw_tree_kernel<<<nbatch, 1024, 0, s>>>(nl, nnodes, lv, loff, lf, rt, vals);
    const int ydt = y ? y_dtype : QA_DT_F32;
    if (aligned && n >= 4 * (int64_t)SD_TE) {
        // pipelined chains: shared-memory ring of 4096-element stages
        const int stage_bytes = SD_TE * ((x_dtype == QA_DT_BF16 ? 2 : 4) + (yk == 2 ? 0 : (yk == QA_DT_BF16 ? 2 : 4)));
        // one dot product alone wants a deep ring (latency); a batch larger than the GPU wants many CTAs per SM instead - a lone
        // warp per sub-partition issues at half rate - so the ring shrinks to what lets 4 - 7 CTAs share an SM's shared memory
        const int64_t nctas = 2 * (int64_t)nbatch + 1;
        const int deep = std::max(2, std::min(SD_MAX_STAGES, 196608 / stage_bytes));
        const int nst = nctas >= 4 * 148 ? 2 : nctas > 148 ? std::min(deep, 3) : deep;
        const int dyn = nst * stage_bytes;
#define QA_SDOT(XD, YD)                                                                                              \
    do {                                                                                                             \
        if (cudaFuncSetAttribute(sdot_pipe_kernel<XD, YD>, cudaFuncAttributeMaxDynamicSharedMemorySize, 196608) != cudaSuccess) \
            return check_launch("qa_tensor_scores_f32 (shared memory attribute)");                                   \
        for (int b0 = 0; b0 < nbatch; b0 += max_y)                                                                   \
            sdot_pipe_kernel<XD, YD><<<dim3(3, std::min(nbatch - b0, max_y)), 64, dyn, s>>>(x, y, y_stride, n, nnodes, nst, vals, dots, b0); \
    } while (0)
        if (x_dtype == QA_DT_BF16) { if (yk == QA_DT_BF16) QA_SDOT(QA_DT_BF16, QA_DT_BF16); else if (yk == QA_DT_F32) QA_SDOT(QA_DT_BF16, QA_DT_F32); else QA_SDOT(QA_DT_BF16, 2); }
        else { if (yk == QA_DT_BF16) QA_SDOT(QA_DT_F32, QA_DT_BF16); else if (yk == QA_DT_F32) QA_SDOT(QA_DT_F32, QA_DT_F32); else QA_SDOT(QA_DT_F32, 2); }
#undef QA_SDOT
    } else {
        for (int b0 = 0; b0 < nbatch; b0 += max_y) {
            const dim3 g(3, std::min(nbatch - b0, max_y));
            if (x_dtype == QA_DT_BF16 && ydt == QA_DT_BF16) sdot_kernel<QA_DT_BF16, QA_DT_BF16><<<g, 64, 0, s>>>(x, y, y_stride, n, nnodes, vals, dots, b0);
            else if (x_dtype == QA_DT_BF16) sdot_kernel<QA_DT_BF16, QA_DT_F32><<<g, 64, 0, s>>>(x, y, y_stride, n, nnodes, vals, dots, b0);
            else if (ydt == QA_DT_BF16) sdot_kernel<QA_DT_F32, QA_DT_BF16><<<g, 64, 0, s>>>(x, y, y_stride, n, nnodes, vals, dots, b0);
            else sdot_kernel<QA_DT_F32, QA_DT_F32><<<g, 64, 0, s>>>(x, y, y_stride, n, nnodes, vals, dots, b0);
        }
    }
    scores_final_kernel<<<(unsigned)cdiv((int64_t)nbatch, 128), 128, 0, s>>>(nbatch, n, nnodes, vals, dots, maxbits, out);
    return check_launch("qa_tensor_scores_f32");
}
