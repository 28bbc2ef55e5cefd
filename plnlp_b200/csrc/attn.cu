// Per-destination softmax over the stored entries of a CSR row (forward and backward): the attention weights of
// PyG's TransformerConv, the conv of the reference's `Transformer` encoder (/root/reference/plnlp/layer.py:57-63).
//   alpha[e] = exp(s[e] - max_row) / sum_row exp(s - max_row)           for e in [rowptr[r], rowptr[r+1])
//   ds[e]    = alpha[e] * (dalpha[e] - sum_row alpha * dalpha)
// One warp per row; entries are walked 32 at a time, reductions by shuffle in a fixed order (deterministic).
// Latency bound (8 B per entry); the heavy parts of the conv are the edge-dot and SpMM kernels.
//
// The row-partitioned conv (layer.TransformerConv on a parallel.ShardedAdj) scores its row block with
// attn_score_csr_kernel: score[e] = <q[row(e)], k[col(e)]> for every stored entry of a CSR block whose queries and
// keys are two separate tables (q: the block's own rows, k: all gathered rows).  Same lane split and reduction order
// as edge_dot_kernel (csrc/edge.cu), so every score is bit-identical to the edge-dot kernel over the pair list
// (row, n_q + col) of the stacked table [q; k] -- without building that table or the pair list.
#include "common.cuh"

namespace plnlp {

__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

__global__ void __launch_bounds__(256) segment_softmax_fwd_kernel(const int64_t* __restrict__ rowptr, int64_t n_rows,
                                                                  const float* __restrict__ s, float scale,
                                                                  float* __restrict__ alpha) {
    const int lane = threadIdx.x & 31;
    const int64_t r = static_cast<int64_t>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (r >= n_rows) return;
    const int64_t e0 = __ldg(rowptr + r), e1 = __ldg(rowptr + r + 1);
    float m = -INFINITY;
    for (int64_t e = e0 + lane; e < e1; e += 32) m = fmaxf(m, __ldg(s + e) * scale);
    m = warp_max(m);
    float z = 0.0f;
    for (int64_t e = e0 + lane; e < e1; e += 32) z += expf(__ldg(s + e) * scale - m);
    z = warp_sum(z);
    const float inv = 1.0f / z;
    for (int64_t e = e0 + lane; e < e1; e += 32) alpha[e] = expf(__ldg(s + e) * scale - m) * inv;
}

__global__ void __launch_bounds__(256) segment_softmax_bwd_kernel(const int64_t* __restrict__ rowptr, int64_t n_rows,
                                                                  const float* __restrict__ alpha,
                                                                  const float* __restrict__ dalpha, float scale,
                                                                  float* __restrict__ ds) {
    const int lane = threadIdx.x & 31;
    const int64_t r = static_cast<int64_t>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (r >= n_rows) return;
    const int64_t e0 = __ldg(rowptr + r), e1 = __ldg(rowptr + r + 1);
    float dot = 0.0f;
    for (int64_t e = e0 + lane; e < e1; e += 32) dot = fmaf(__ldg(alpha + e), __ldg(dalpha + e), dot);
    dot = warp_sum(dot);
    for (int64_t e = e0 + lane; e < e1; e += 32) ds[e] = __ldg(alpha + e) * (__ldg(dalpha + e) - dot) * scale;
}

// One warp per work item of the block's SpMM plan (graph.build_plan: a row, or a <= chunk slice of a hub row), so no
// warp walks a whole hub row.  The lane's slice of q[row] stays in registers across the item (ATTN_QREG floats per
// lane: F <= 512 at VEC = 4; wider rows read the rest from L1); entries go ATTN_U at a time so that many key rows are
// in flight.
constexpr int ATTN_QREG = 16;                 // floats of q per lane held in registers
constexpr int ATTN_U = 4;

template <int VEC, int NREG, int U>
__device__ __forceinline__ void attn_score_entries(const float (&qv)[NREG][VEC], const float* __restrict__ qr,
                                                   const float* __restrict__ k, int64_t ldk,
                                                   const int32_t* __restrict__ col, int e, int H, int lane,
                                                   float* __restrict__ score) {
    const float* kr[U];
#pragma unroll
    for (int u = 0; u < U; ++u) kr[u] = k + static_cast<int64_t>(__ldg(col + e + u)) * ldk;
    float acc[U];
#pragma unroll
    for (int u = 0; u < U; ++u) acc[u] = 0.0f;
    // feature order f = lane * VEC + c * 32 * VEC, c ascending, then the VEC lanes of a chunk: edge_dot_kernel's order
#pragma unroll
    for (int c = 0; c < NREG; ++c) {
        const int f = (c * 32 + lane) * VEC;
        if (f < H) {
#pragma unroll
            for (int u = 0; u < U; ++u) {
                float b[VEC];
                load_vec<VEC>(b, kr[u] + f);
#pragma unroll
                for (int j = 0; j < VEC; ++j) acc[u] = fmaf(qv[c][j], b[j], acc[u]);
            }
        }
    }
    for (int f = (NREG * 32 + lane) * VEC; f < H; f += 32 * VEC) {      // features past the register slice
        float a[VEC];
        load_vec<VEC>(a, qr + f);
#pragma unroll
        for (int u = 0; u < U; ++u) {
            float b[VEC];
            load_vec<VEC>(b, kr[u] + f);
#pragma unroll
            for (int j = 0; j < VEC; ++j) acc[u] = fmaf(a[j], b[j], acc[u]);
        }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) acc[u] = warp_sum(acc[u]);
    if (lane == 0) {
#pragma unroll
        for (int u = 0; u < U; ++u) score[e + u] = acc[u];
    }
}

template <int VEC>
__global__ void __launch_bounds__(256) attn_score_csr_kernel(const int32_t* __restrict__ item_ptr,
                                                             const int32_t* __restrict__ item_row, int64_t n_items,
                                                             const int32_t* __restrict__ col,
                                                             const float* __restrict__ q, int64_t ldq,
                                                             const float* __restrict__ k, int64_t ldk, int H,
                                                             float* __restrict__ score) {
    constexpr int NREG = ATTN_QREG / VEC;
    const int lane = threadIdx.x & 31;
    const int64_t it = static_cast<int64_t>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (it >= n_items) return;
    const int e0 = __ldg(item_ptr + it), e1 = __ldg(item_ptr + it + 1);
    if (e0 >= e1) return;
    const float* qr = q + static_cast<int64_t>(__ldg(item_row + it)) * ldq;
    float qv[NREG][VEC];
#pragma unroll
    for (int c = 0; c < NREG; ++c) {
        const int f = (c * 32 + lane) * VEC;
        if (f < H) {
            load_vec<VEC>(qv[c], qr + f);
        } else {
#pragma unroll
            for (int j = 0; j < VEC; ++j) qv[c][j] = 0.0f;
        }
    }
    int e = e0;
    for (; e + ATTN_U <= e1; e += ATTN_U) attn_score_entries<VEC, NREG, ATTN_U>(qv, qr, k, ldk, col, e, H, lane, score);
    for (; e < e1; ++e) attn_score_entries<VEC, NREG, 1>(qv, qr, k, ldk, col, e, H, lane, score);
}

}  // namespace plnlp

extern "C" int plnlp_attn_score_csr_f32(const int32_t* item_ptr, const int32_t* item_row, int64_t n_items,
                                        const int32_t* col, const float* q, int64_t ldq, const float* k, int64_t ldk,
                                        int64_t F, float* score, void* stream) {
    using namespace plnlp;
    PLNLP_REQUIRE(n_items >= 0 && F > 0 && F < (int64_t{1} << 30), PLNLP_E_SIZE);
    if (n_items == 0) return 0;
    PLNLP_REQUIRE(item_ptr && item_row && col && q && k && score, PLNLP_E_NULL);
    PLNLP_REQUIRE(ldq >= F && ldk >= F, PLNLP_E_SIZE);
    const int vec = pick_vec(F, {ldq, ldk}, {q, k});
    const unsigned grid = static_cast<unsigned>(ceil_div(n_items, 8));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
#define CALL(V) attn_score_csr_kernel<V><<<grid, 256, 0, st>>>(item_ptr, item_row, n_items, col, q, ldq, k, ldk, \
                                                               static_cast<int>(F), score)
    if (vec == 4) CALL(4);
    else if (vec == 2) CALL(2);
    else CALL(1);
#undef CALL
    PLNLP_LAUNCH_CHECK();
    return 0;
}

extern "C" int plnlp_segment_softmax_fwd_f32(const int64_t* rowptr, int64_t n_rows, const float* s, float scale,
                                             float* alpha, void* stream) {
    using namespace plnlp;
    PLNLP_REQUIRE(n_rows >= 0, PLNLP_E_SIZE);
    if (n_rows == 0) return 0;
    PLNLP_REQUIRE(rowptr && s && alpha, PLNLP_E_NULL);
    segment_softmax_fwd_kernel<<<static_cast<unsigned>(ceil_div(n_rows, 8)), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        rowptr, n_rows, s, scale, alpha);
    PLNLP_LAUNCH_CHECK();
    return 0;
}

extern "C" int plnlp_segment_softmax_bwd_f32(const int64_t* rowptr, int64_t n_rows, const float* alpha,
                                             const float* dalpha, float scale, float* ds, void* stream) {
    using namespace plnlp;
    PLNLP_REQUIRE(n_rows >= 0, PLNLP_E_SIZE);
    if (n_rows == 0) return 0;
    PLNLP_REQUIRE(rowptr && alpha && dalpha && ds, PLNLP_E_NULL);
    segment_softmax_bwd_kernel<<<static_cast<unsigned>(ceil_div(n_rows, 8)), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        rowptr, n_rows, alpha, dalpha, scale, ds);
    PLNLP_LAUNCH_CHECK();
    return 0;
}
