// Out-of-place 2-D transposition of 1-, 2- or 4-byte elements: out[cols][rows] = x[rows][cols] (leading dimension ld).
// The mixed-tile algorithms run in the device layout (W^T) by transposing the checkpoint's W once and then using every
// row-major kernel unchanged; this kernel is that copy (bf16 / float32 weights, fp8 bytes and their scale grid, and y back).
//
// A CTA moves one 64 x 64 tile through shared memory: coalesced row reads of x, coalesced row writes of out.  Each thread
// moves V consecutive elements per access (4 B for bytes, 8 B for bf16, 16 B for float32) when the base pointers and the
// leading dimensions allow it, else one element.  The shared row stride is padded to an odd number of 4 B-words, so that
// the column reads of the store phase spread over the banks (at most 2-way conflicts with V = 4).
#include "qa_common.cuh"

namespace qa {
namespace {

constexpr int TD = 64;          // tile edge (elements)
constexpr int THREADS = 256;

template <typename T, int V>
struct alignas(sizeof(T) * V) Vec {
    T v[V];
};

template <typename T, int V>
__global__ void __launch_bounds__(THREADS) transpose_kernel(const T* __restrict__ x, int64_t rows, int64_t cols, int64_t ld,
                                                            T* __restrict__ out, int64_t tiles_c, int64_t ntiles) {
    constexpr int PAD = 4 / (int)sizeof(T);              // one 4 B-word: an odd row stride in words
    __shared__ T tile[TD][TD + PAD];
    constexpr int TPR = TD / V;                           // threads per tile row
    constexpr int RPP = THREADS / TPR;                    // tile rows per pass
    const int tx = threadIdx.x % TPR, ty = threadIdx.x / TPR;
    for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const int64_t r0 = (t / tiles_c) * TD, c0 = (t % tiles_c) * TD;
        const int nr = rows - r0 < TD ? (int)(rows - r0) : TD, nc = cols - c0 < TD ? (int)(cols - c0) : TD;
        // load: tile[i][j] = x[r0 + i][c0 + j]
        for (int i = ty; i < nr; i += RPP) {
            const int j = tx * V;
            const T* src = x + (r0 + i) * ld + c0 + j;
            if (j + V <= nc) {
                const Vec<T, V> w = *reinterpret_cast<const Vec<T, V>*>(src);
#pragma unroll
                for (int k = 0; k < V; ++k) tile[i][j + k] = w.v[k];
            } else {
#pragma unroll
                for (int k = 0; k < V; ++k)
                    if (j + k < nc) tile[i][j + k] = src[k];
            }
        }
        __syncthreads();
        // store: out[c0 + j][r0 + i] = tile[i][j]
        for (int j = ty; j < nc; j += RPP) {
            const int i = tx * V;
            T* dst = out + (c0 + j) * rows + r0 + i;
            if (i + V <= nr) {
                Vec<T, V> w;
#pragma unroll
                for (int k = 0; k < V; ++k) w.v[k] = tile[i + k][j];
                *reinterpret_cast<Vec<T, V>*>(dst) = w;
            } else {
#pragma unroll
                for (int k = 0; k < V; ++k)
                    if (i + k < nr) dst[k] = tile[i + k][j];
            }
        }
        __syncthreads();
    }
}

template <typename T>
int launch(const void* x, int64_t rows, int64_t cols, int64_t ld, void* out, cudaStream_t s) {
    constexpr int V = 4;
    constexpr uintptr_t VB = sizeof(T) * V;
    // the vector path needs every row start of x (stride ld) and of out (stride rows) on a V-element boundary
    const bool vec = ((uintptr_t)x % VB == 0) && ((uintptr_t)out % VB == 0) && (ld % V == 0) && (rows % V == 0);
    const int64_t tiles_c = cdiv(cols, TD), ntiles = cdiv(rows, TD) * tiles_c;
    const int grid = (int)(ntiles < 148 * 16 ? ntiles : 148 * 16);       // 148 SMs x 16 resident CTAs; larger tensors loop
    const T* xp = reinterpret_cast<const T*>(x);
    T* op = reinterpret_cast<T*>(out);
    if (vec) transpose_kernel<T, V><<<grid, THREADS, 0, s>>>(xp, rows, cols, ld, op, tiles_c, ntiles);
    else transpose_kernel<T, 1><<<grid, THREADS, 0, s>>>(xp, rows, cols, ld, op, tiles_c, ntiles);
    return check_launch("qa_transpose_2d");
}

}  // namespace
}  // namespace qa

using namespace qa;

extern "C" int qa_transpose_2d(const void* x, int elem_bytes, int64_t rows, int64_t cols, int64_t ld, void* out,
                               qa_stream_t stream) {
    if (elem_bytes != 1 && elem_bytes != 2 && elem_bytes != 4) {
        set_error("qa_transpose_2d: elem_bytes must be 1, 2 or 4 (got %d)", elem_bytes);
        return 1;
    }
    if (rows < 0 || cols < 0 || ld < cols) { set_error("qa_transpose_2d: bad shape"); return 1; }
    if (rows == 0 || cols == 0) return 0;
    if (!x || !out) { set_error("qa_transpose_2d: null pointer"); return 1; }
    cudaStream_t s = (cudaStream_t)stream;
    if (elem_bytes == 1) return launch<uint8_t>(x, rows, cols, ld, out, s);
    if (elem_bytes == 2) return launch<uint16_t>(x, rows, cols, ld, out, s);
    return launch<uint32_t>(x, rows, cols, ld, out, s);
}
