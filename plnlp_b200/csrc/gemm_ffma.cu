// Exact-fp32 GEMM on the CUDA cores (FFMA, fp32 accumulate) with fused epilogues.
//
// Replaces torch.nn.Linear -> cuBLAS sgemm at /root/reference/plnlp/layer.py:20,23,82-86 and the
// two backward GEMMs autograd derives from it.  This is the parity-exact dense path; the
// tensor-core (tcgen05, 3xTF32) path lives in gemm_tcgen05.cu and is validated against this one.
//
//   C = act( op(A) . op(B) + beta*C + bias )
//
// 128x128x16 CTA tile, 256 threads, 8x8 register micro-tile per thread (2x2 groups of 4x4 so
// that shared-memory reads are 16-byte and conflict-free), register-staged double buffering:
// the next k-slab is fetched from global memory while the current one is multiplied.
#include "common.cuh"

namespace plnlp {

constexpr int BM = 128, BN = 128, BK = 16, PAD = 4;

struct GemmParams {
    int64_t M, N, K;
    const float* A; int64_t lda;
    const float* B; int64_t ldb;
    float* C; int64_t ldc;
    float beta;
    const float* bias;
    int act;
    const float* aux; int64_t ldaux;
    float drop_p; uint64_t seed;
    float* ws;       // split-k partials [split][M][N]
    int split_k;
    int64_t k_per_split;
    bool vec_c;
};

__device__ __forceinline__ float epilogue_one(const GemmParams& p, int64_t r, int64_t c, float v) {
    if (p.beta != 0.0f) v += p.beta * p.C[r * p.ldc + c];
    if (p.bias) v += __ldg(p.bias + c);
    if (p.act == PLNLP_ACT_RELU) {
        v = fmaxf(v, 0.0f);
        if (p.drop_p > 0.0f)
            v = dropout_keep(p.seed, static_cast<uint64_t>(r) * p.N + c, p.drop_p) ? v * (1.0f / (1.0f - p.drop_p)) : 0.0f;
    } else if (p.act == PLNLP_ACT_RELU_GRAD) {
        v = (__ldg(p.aux + r * p.ldaux + c) > 0.0f) ? v * (1.0f / (1.0f - p.drop_p)) : 0.0f;
    }
    return v;
}

// Global -> register fetch of this thread's share of one operand slab.
// KCONTIG: the operand is contiguous along k (A non-transposed / B transposed).
//   tile is [128 rows][16 k]; float4 i = tid + 256*r -> row = i/4, kq = i%4
// else: contiguous along the row index (A transposed / B non-transposed)
//   tile is [16 k][128 rows]; float4 i -> k = i/32, rq = i%32
template <bool KCONTIG, bool VEC>
__device__ __forceinline__ void fetch(const float* __restrict__ base, int64_t ld, int64_t row0, int64_t nrows,
                                      int64_t k0, int64_t kend, int tid, float (&reg)[2][4]) {
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        const int i = tid + 256 * r;
        if (KCONTIG) {
            const int64_t row = row0 + (i >> 2);
            const int64_t k = k0 + (i & 3) * 4;
            const float* src = base + row * ld + k;
            if (VEC) {
                if (row < nrows && k < kend) {
                    const float4 t = __ldg(reinterpret_cast<const float4*>(src));
                    reg[r][0] = t.x; reg[r][1] = t.y; reg[r][2] = t.z; reg[r][3] = t.w;
                } else {
                    reg[r][0] = reg[r][1] = reg[r][2] = reg[r][3] = 0.0f;
                }
            } else {
#pragma unroll
                for (int e = 0; e < 4; ++e) reg[r][e] = (row < nrows && k + e < kend) ? __ldg(src + e) : 0.0f;
            }
        } else {
            const int64_t k = k0 + (i >> 5);
            const int64_t row = row0 + (i & 31) * 4;
            const float* src = base + k * ld + row;
            if (VEC) {
                if (k < kend && row < nrows) {
                    const float4 t = __ldg(reinterpret_cast<const float4*>(src));
                    reg[r][0] = t.x; reg[r][1] = t.y; reg[r][2] = t.z; reg[r][3] = t.w;
                } else {
                    reg[r][0] = reg[r][1] = reg[r][2] = reg[r][3] = 0.0f;
                }
            } else {
#pragma unroll
                for (int e = 0; e < 4; ++e) reg[r][e] = (k < kend && row + e < nrows) ? __ldg(src + e) : 0.0f;
            }
        }
    }
}

// register -> shared, always producing the k-major layout S[k][row] (row padded by PAD)
template <bool KCONTIG>
__device__ __forceinline__ void stash(float (*S)[BM + PAD], int tid, const float (&reg)[2][4]) {
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        const int i = tid + 256 * r;
        if (KCONTIG) {
            const int row = i >> 2, kq = (i & 3) * 4;
#pragma unroll
            for (int e = 0; e < 4; ++e) S[kq + e][row] = reg[r][e];
        } else {
            const int k = i >> 5, rq = (i & 31) * 4;
            *reinterpret_cast<float4*>(&S[k][rq]) = make_float4(reg[r][0], reg[r][1], reg[r][2], reg[r][3]);
        }
    }
}

template <bool TA, bool TB, bool VA, bool VB>
__global__ void __launch_bounds__(256) gemm_ffma_kernel(const GemmParams p) {
    __shared__ __align__(16) float As[2][BK][BM + PAD];
    __shared__ __align__(16) float Bs[2][BK][BN + PAD];
    const int tid = threadIdx.x;
    const int tx = tid & 15, ty = tid >> 4;
    const int64_t m0 = static_cast<int64_t>(blockIdx.y) * BM, n0 = static_cast<int64_t>(blockIdx.x) * BN;
    const int64_t kbeg = static_cast<int64_t>(blockIdx.z) * p.k_per_split;
    const int64_t kend = min(p.K, kbeg + p.k_per_split);

    float acc[8][8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = 0.0f;

    float ra[2][4], rb[2][4];
    // A is k-contiguous when NOT transposed; B is k-contiguous when transposed.
    fetch<!TA, VA>(p.A, p.lda, m0, p.M, kbeg, kend, tid, ra);
    fetch<TB, VB>(p.B, p.ldb, n0, p.N, kbeg, kend, tid, rb);
    stash<!TA>(As[0], tid, ra);
    stash<TB>(Bs[0], tid, rb);
    __syncthreads();

    int buf = 0;
    for (int64_t k0 = kbeg; k0 < kend; k0 += BK) {
        const bool more = (k0 + BK) < kend;
        if (more) {
            fetch<!TA, VA>(p.A, p.lda, m0, p.M, k0 + BK, kend, tid, ra);
            fetch<TB, VB>(p.B, p.ldb, n0, p.N, k0 + BK, kend, tid, rb);
        }
#pragma unroll
        for (int k = 0; k < BK; ++k) {
            const float4 a0 = *reinterpret_cast<const float4*>(&As[buf][k][ty * 4]);
            const float4 a1 = *reinterpret_cast<const float4*>(&As[buf][k][64 + ty * 4]);
            const float4 b0 = *reinterpret_cast<const float4*>(&Bs[buf][k][tx * 4]);
            const float4 b1 = *reinterpret_cast<const float4*>(&Bs[buf][k][64 + tx * 4]);
            const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
            const float b[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
        }
        if (more) {
            stash<!TA>(As[buf ^ 1], tid, ra);
            stash<TB>(Bs[buf ^ 1], tid, rb);
            __syncthreads();
            buf ^= 1;
        }
    }

    // epilogue
    const bool split = p.split_k > 1;
    float* wsz = split ? p.ws + static_cast<int64_t>(blockIdx.z) * p.M * p.N : nullptr;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int64_t r = m0 + (i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4));
        if (r >= p.M) continue;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int64_t c = n0 + h * 64 + tx * 4;
            if (c >= p.N) continue;
            float v[4] = {acc[i][h * 4 + 0], acc[i][h * 4 + 1], acc[i][h * 4 + 2], acc[i][h * 4 + 3]};
            if (split) {
#pragma unroll
                for (int e = 0; e < 4; ++e)
                    if (c + e < p.N) wsz[r * p.N + c + e] = v[e];
            } else {
#pragma unroll
                for (int e = 0; e < 4; ++e)
                    if (c + e < p.N) v[e] = epilogue_one(p, r, c + e, v[e]);
                if (p.vec_c && c + 3 < p.N) {
                    *reinterpret_cast<float4*>(p.C + r * p.ldc + c) = make_float4(v[0], v[1], v[2], v[3]);
                } else {
#pragma unroll
                    for (int e = 0; e < 4; ++e)
                        if (c + e < p.N) p.C[r * p.ldc + c + e] = v[e];
                }
            }
        }
    }
}

__global__ void __launch_bounds__(256) splitk_reduce_kernel(const GemmParams p) {
    const int64_t total = p.M * p.N;
    for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
         i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        float v = 0.0f;
        for (int z = 0; z < p.split_k; ++z) v += p.ws[static_cast<int64_t>(z) * total + i];
        const int64_t r = i / p.N, c = i % p.N;
        p.C[r * p.ldc + c] = epilogue_one(p, r, c, v);
    }
}

template <bool TA, bool TB>
static void launch_variant(const GemmParams& p, bool va, bool vb, dim3 grid, cudaStream_t st) {
    if (va && vb)       gemm_ffma_kernel<TA, TB, true, true><<<grid, 256, 0, st>>>(p);
    else if (va && !vb) gemm_ffma_kernel<TA, TB, true, false><<<grid, 256, 0, st>>>(p);
    else if (!va && vb) gemm_ffma_kernel<TA, TB, false, true><<<grid, 256, 0, st>>>(p);
    else                gemm_ffma_kernel<TA, TB, false, false><<<grid, 256, 0, st>>>(p);
}

}  // namespace plnlp

extern "C" int plnlp_gemm_f32(int transa, int transb, int64_t M, int64_t N, int64_t K, const float* A,
                              int64_t lda, const float* B, int64_t ldb, float* C, int64_t ldc, float beta,
                              const float* bias, int act, const float* aux, int64_t ldaux, float drop_p,
                              uint64_t seed, float* workspace, int64_t workspace_bytes, int split_k,
                              void* stream) {
    using namespace plnlp;
    PLNLP_REQUIRE(M >= 0 && N >= 0 && K >= 0, PLNLP_E_SIZE);
    if (M == 0 || N == 0) return 0;
    PLNLP_REQUIRE(C && (K == 0 || (A && B)), PLNLP_E_NULL);     // K = 0 reads neither operand (empty tensors: NULL)
    PLNLP_REQUIRE(lda >= (transa ? M : K) && ldb >= (transb ? K : N) && ldc >= N, PLNLP_E_SIZE);
    PLNLP_REQUIRE(act >= 0 && act <= 2 && drop_p >= 0.0f && drop_p < 1.0f, PLNLP_E_SIZE);
    if (act == PLNLP_ACT_RELU_GRAD) PLNLP_REQUIRE(aux && ldaux >= N, PLNLP_E_NULL);
    if (split_k < 1) split_k = 1;
    if (K == 0) split_k = 1;
    GemmParams p{};
    p.M = M; p.N = N; p.K = K; p.A = A; p.lda = lda; p.B = B; p.ldb = ldb; p.C = C; p.ldc = ldc;
    p.beta = beta; p.bias = bias; p.act = act; p.aux = aux; p.ldaux = ldaux; p.drop_p = drop_p; p.seed = seed;
    p.split_k = split_k;
    int64_t kper = ceil_div(ceil_div(K, split_k), BK) * BK;
    if (kper == 0) kper = BK;
    p.k_per_split = kper;
    p.split_k = split_k = static_cast<int>(K == 0 ? 1 : ceil_div(K, kper));
    p.ws = workspace;
    if (split_k > 1) {
        PLNLP_REQUIRE(workspace, PLNLP_E_NULL);
        PLNLP_REQUIRE(workspace_bytes >= static_cast<int64_t>(split_k) * M * N * 4, PLNLP_E_WORKSPACE);
    }
    p.vec_c = (ldc % 4 == 0) && aligned(C, 16);
    // a 16-byte fetch is legal when the contiguous extent is a multiple of 4 and rows stay aligned
    const bool va = aligned(A, 16) && (lda % 4 == 0) && ((transa ? M : K) % 4 == 0) && (kper % 4 == 0);
    const bool vb = aligned(B, 16) && (ldb % 4 == 0) && ((transb ? K : N) % 4 == 0);
    const dim3 grid(static_cast<unsigned>(ceil_div(N, BN)), static_cast<unsigned>(ceil_div(M, BM)),
                    static_cast<unsigned>(split_k));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (!transa && !transb)      launch_variant<false, false>(p, va, vb, grid, st);
    else if (!transa && transb)  launch_variant<false, true>(p, va, vb, grid, st);
    else if (transa && !transb)  launch_variant<true, false>(p, va, vb, grid, st);
    else                         launch_variant<true, true>(p, va, vb, grid, st);
    PLNLP_LAUNCH_CHECK();
    if (split_k > 1) {
        const int64_t total = M * N;
        const unsigned blocks = static_cast<unsigned>(std::min<int64_t>(ceil_div(total, 256), 148 * 8));
        splitk_reduce_kernel<<<blocks, 256, 0, st>>>(p);
        PLNLP_LAUNCH_CHECK();
    }
    return 0;
}
