// Tensor-core GEMM for sm_100a: tcgen05.mma kind::tf32, operands staged in shared memory in the
// canonical no-swizzle core-matrix layout, fp32 accumulator in TMEM, fused epilogue.
//
// Replaces torch.nn.Linear -> cuBLAS sgemm at /root/reference/plnlp/layer.py:20,23,82-86 and its two
// backward GEMMs on the tensor pipe while keeping fp32 parity:
//
//   passes = 3 ("3xTF32", error-compensated):  A = Ah + Al, B = Bh + Bl with Ah = rn_tf32(A),
//            Al = A - Ah (exact in fp32);  A.B ~= Ah.Bh + Ah.Bl + Al.Bh, all accumulated in fp32 in
//            TMEM.  The dropped Al.Bl term is 2^-22 relative.  The tensor core accumulates with
//            round-toward-zero, so the error grows linearly with the number of accumulation steps
//            (K/8): callers keep K per accumulator <= 1024 (split-k, partials reduced with RN adds on
//            the CUDA cores) which keeps the result within ~4e-6 relative -- inside the 1e-5 bar.
//   passes = 1: plain TF32 (~1e-3 relative), the stated fast path.
//
// CTA = 128 x BN output tile, 9 warps: warps 0-7 load A/B slabs from global memory (any of the four
// transpose combinations), split them into hi/lo parts and write the UMMA layout; warp 8 allocates
// TMEM and its elected lane issues the MMAs; full/empty mbarriers form a STAGES-deep ring
// (loaders -> MMA via fence.proxy.async + arrive, MMA -> loaders via tcgen05.commit).  Global loads
// run two slabs ahead of the shared-memory stores (two register buffers).  The shared-memory footprint
// is held to ~165 KB on purpose: the global loads travel through L1, and with a full 227 KB carve-out
// the ~7 KB of L1 left throttles the loads in flight (measured: 4x slower).  After the last k-slab the
// same 8 warps read the accumulator (tcgen05.ld 32x32b) and apply the epilogue (split-k partial store,
// or beta*C + bias -> relu -> dropout / relu-grad mask).
//
// Shared-memory operand layout: BOTH operands are staged K-major, whatever their layout in global
// memory (MN-major tf32 operands need the special 128B_BASE32B swizzle on this hardware; transposing in
// the loader keeps one well-understood layout).  Slab tile [R rows][16 k] (64 B of K per row), made of
// 8-row x 16-byte core matrices:
//     byte(r, k) = (k/4)*LBO + (r/8)*SBO + (r%8)*16 + (k%4)*4,   SBO = 144, LBO = 18*R + 32
//   SBO = 128 + 16 and LBO = 2 (mod 8) x 16 bytes skew successive row-groups / k-chunks by one / two 16-byte bank
//   groups, so both store patterns below are bank-conflict free:
//     K-contiguous source : a quarter-warp writes the k-chunks of two rows           (16-byte stores)
//     MN-contiguous source: a thread loads a 4(k) x 4(mn) block with four 16-byte loads, transposes it
//                           in registers and writes four 16-byte chunks (rows r..r+3 of one k-chunk);
//                           a quarter-warp covers 8 consecutive 4-row groups.
#include "gemm_tc_common.cuh"

namespace plnlp {

namespace {

using namespace tcgemm;

template <bool SPLIT>
struct Cfg {
    static constexpr int STAGES = SPLIT ? 2 : 4;      // 2 CTAs per SM share the 227 KB
};

// BN: CTA tile columns (UMMA N, TMEM columns); AMN/BMN: operand is MN-contiguous in global memory
// (A: transa = 1, B: transb = 0); VA/VB: 16-byte global loads legal; SPLIT: 3xTF32.
template <int BN, bool AMN, bool BMN, bool VA, bool VB, bool SPLIT>
__global__ void __launch_bounds__(NTHREADS, 2) gemm_tcgen05_kernel(const TcGemmParams p) {
    constexpr int STAGES = Cfg<SPLIT>::STAGES;
    constexpr int A_SLOT = slot_bytes(TBM), B_SLOT = slot_bytes(BN);
    constexpr int STAGE_BYTES = (SPLIT ? 2 : 1) * (A_SLOT + B_SLOT);
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ __align__(8) uint64_t full_bar[STAGES], empty_bar[STAGES], accum_bar;
    __shared__ uint32_t tmem_holder;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t m0 = static_cast<int64_t>(blockIdx.y) * TBM, n0 = static_cast<int64_t>(blockIdx.x) * BN;
    const int64_t kbeg = static_cast<int64_t>(blockIdx.z) * p.k_per_split;
    const int64_t kend = min(p.K, kbeg + p.k_per_split);
    const int n_iter = static_cast<int>((kend - kbeg + TBK - 1) / TBK);
    // columns actually multiplied: N remainder rounded up to the UMMA granularity (16)
    const int64_t n_rem = ((p.N - n0 + 15) / 16) * 16;
    const int n_mma = n_rem < BN ? static_cast<int>(n_rem) : BN;

    if (tid == 0) {
        for (int s = 0; s < STAGES; ++s) {
            tc::mbar_init(&full_bar[s], LOADERS);
            tc::mbar_init(&empty_bar[s], 1);
        }
        tc::mbar_init(&accum_bar, 1);
        tc::mbar_fence_init();
    }
    if (warp == 8) tc::tmem_alloc<BN>(&tmem_holder);
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    const uint32_t tmem_d = tmem_holder;

    auto stage_ptr = [&](int s, int which) -> uint8_t* {  // which: 0 A.hi, 1 B.hi, 2 A.lo, 3 B.lo
        uint8_t* base = smem + s * STAGE_BYTES;
        return base + (which & 1 ? A_SLOT : 0) + (which & 2 ? (A_SLOT + B_SLOT) : 0);
    };

    if (warp < 8) {
        // ============================ loaders ============================
        float ra[2][nreg(TBM, AMN)][4], rb[2][nreg(BN, BMN)][4];
        Loader<TBM, AMN, VA> la;
        Loader<BN, BMN, VB> lb;
        la.init(p.A, p.lda, m0, p.M, kbeg, tid);
        lb.init(p.B, p.ldb, n0, p.N, kbeg, tid);
        const int ktot = static_cast<int>(kend - kbeg);
        auto fetch = [&](int it, float (&a)[nreg(TBM, AMN)][4], float (&b)[nreg(BN, BMN)][4]) {
            if (it < n_iter) {                            // called with it = 0, 1, 2, ... in order
                la.fetch(ktot - it * TBK, a);
                lb.fetch(ktot - it * TBK, b);
            }
        };
        auto publish = [&](int it, const float (&a)[nreg(TBM, AMN)][4], const float (&b)[nreg(BN, BMN)][4]) {
            const int s = it % STAGES;
            const uint32_t ph = (it / STAGES) & 1;
            tc::mbar_wait(&empty_bar[s], ph ^ 1);         // slot free (first round passes immediately)
            la.template stash<SPLIT>(stage_ptr(s, 0), stage_ptr(s, 2), a);
            lb.template stash<SPLIT>(stage_ptr(s, 1), stage_ptr(s, 3), b);
        };
        fetch(0, ra[0], rb[0]);
        fetch(1, ra[1], rb[1]);
        // NOTE the order: the proxy fence waits for every memory operation the thread has in flight,
        // including global loads, so it must come BEFORE the next prefetch is issued (measured: with
        // the prefetch first every slab paid a full global-load latency).
        for (int it = 0; it < n_iter; it += 2) {
            publish(it, ra[0], rb[0]);
            tc::fence_proxy_async_smem();
            tc::mbar_arrive(&full_bar[it % STAGES]);
            fetch(it + 2, ra[0], rb[0]);                  // two slabs ahead of the stores
            if (it + 1 < n_iter) {
                publish(it + 1, ra[1], rb[1]);
                tc::fence_proxy_async_smem();
                tc::mbar_arrive(&full_bar[(it + 1) % STAGES]);
                fetch(it + 3, ra[1], rb[1]);
            }
        }
    } else {
        // ============================ MMA issuer ============================
        const uint32_t idesc = tc::make_idesc_tf32(TBM, n_mma, 0, 0);      // both operands K-major in smem
        constexpr uint32_t A_LBO = tile_lbo(TBM), B_LBO = tile_lbo(BN), A_SBO = TILE_SBO, B_SBO = TILE_SBO;
        // one UMMA consumes K = 8 (32 bytes) = two 16-byte k-chunks, i.e. 2*LBO per step
        constexpr uint32_t A_STEP = 2 * A_LBO, B_STEP = 2 * B_LBO;
        for (int it = 0; it < n_iter; ++it) {
            const int s = it % STAGES;
            const uint32_t ph = (it / STAGES) & 1;
            tc::mbar_wait(&full_bar[s], ph);
            tc::fence_after_sync();
            if (lane == 0) {
                const uint32_t a_hi = tc::smem_u32(stage_ptr(s, 0)), b_hi = tc::smem_u32(stage_ptr(s, 1));
                const uint32_t a_lo = tc::smem_u32(stage_ptr(s, 2)), b_lo = tc::smem_u32(stage_ptr(s, 3));
#pragma unroll
                for (int j = 0; j < TBK / 8; ++j) {
                    const uint64_t dah = tc::make_smem_desc(a_hi + j * A_STEP, A_LBO, A_SBO);
                    const uint64_t dbh = tc::make_smem_desc(b_hi + j * B_STEP, B_LBO, B_SBO);
                    tc::mma_tf32_ss(tmem_d, dah, dbh, idesc, (it | j) != 0);
                    if (SPLIT) {
                        const uint64_t dal = tc::make_smem_desc(a_lo + j * A_STEP, A_LBO, A_SBO);
                        const uint64_t dbl = tc::make_smem_desc(b_lo + j * B_STEP, B_LBO, B_SBO);
                        tc::mma_tf32_ss(tmem_d, dah, dbl, idesc, 1u);
                        tc::mma_tf32_ss(tmem_d, dal, dbh, idesc, 1u);
                    }
                }
                tc::mma_commit(&empty_bar[s]);                       // frees the slot when these finish
                if (it == n_iter - 1) tc::mma_commit(&accum_bar);    // accumulator complete
            }
            __syncwarp();
        }
    }

    // ============================ epilogue (warps 0-7) ============================
    if (warp < 8) {
        if (n_iter > 0) {
            tc::mbar_wait(&accum_bar, 0);
            tc::fence_after_sync();
        }
        tc_epilogue_tile<BN>(p, tmem_d, m0, n0, n_mma, n_iter, warp, lane);
    }
    tc::fence_before_sync();
    __syncthreads();
    if (warp == 8) tc::tmem_dealloc<BN>(tmem_d);
}

__global__ void __launch_bounds__(256) tc_splitk_reduce_kernel(const TcGemmParams p) {
    const int64_t total = p.M * p.N;
    for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
         i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        float v = 0.0f;
        for (int z = 0; z < p.split_k; ++z) v += p.ws[static_cast<int64_t>(z) * total + i];
        const int64_t r = i / p.N, c = i % p.N;
        p.C[r * p.ldc + c] = tc_epilogue_one(p, r, c, v);
    }
}

template <int BN, bool AMN, bool BMN, bool VA, bool VB, bool SPLIT>
int launch_one(const TcGemmParams& p, dim3 grid, cudaStream_t st) {
    constexpr int bytes = Cfg<SPLIT>::STAGES * (SPLIT ? 2 : 1) * (slot_bytes(TBM) + slot_bytes(BN));
    static_assert(bytes <= 113 * 1024, "two CTAs per SM: epilogue of one overlaps the main loop of the other");
    auto kern = gemm_tcgen05_kernel<BN, AMN, BMN, VA, VB, SPLIT>;
    static bool configured = false;
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
        if (e != cudaSuccess) return static_cast<int>(e);
        configured = true;
    }
    kern<<<grid, NTHREADS, bytes, st>>>(p);
    return 0;
}

template <int BN, bool AMN, bool BMN>
int launch_vec(const TcGemmParams& p, bool va, bool vb, dim3 grid, cudaStream_t st) {
    // the unaligned (scalar-load) path is only instantiated for the exact 3-pass variant to bound
    // compile time; plain-TF32 requests with unaligned operands use it too
    const bool split = p.passes == 3;
    if (va && vb) {
        return split ? launch_one<BN, AMN, BMN, true, true, true>(p, grid, st)
                     : launch_one<BN, AMN, BMN, true, true, false>(p, grid, st);
    }
    if (va) return launch_one<BN, AMN, BMN, true, false, true>(p, grid, st);
    if (vb) return launch_one<BN, AMN, BMN, false, true, true>(p, grid, st);
    return launch_one<BN, AMN, BMN, false, false, true>(p, grid, st);
}

template <int BN>
int launch_major(const TcGemmParams& p, bool amn, bool bmn, bool va, bool vb, dim3 grid, cudaStream_t st) {
    if (!amn && !bmn) return launch_vec<BN, false, false>(p, va, vb, grid, st);
    if (!amn && bmn) return launch_vec<BN, false, true>(p, va, vb, grid, st);
    if (amn && !bmn) return launch_vec<BN, true, false>(p, va, vb, grid, st);
    return launch_vec<BN, true, true>(p, va, vb, grid, st);
}

}  // namespace

namespace tcgemm {
int tc_splitk_reduce(const TcGemmParams& p, cudaStream_t st) {
    const int64_t total = p.M * p.N;
    const unsigned blocks = static_cast<unsigned>(std::min<int64_t>(ceil_div(total, 256), 148 * 8));
    tc_splitk_reduce_kernel<<<blocks, 256, 0, st>>>(p);
    PLNLP_LAUNCH_CHECK();
    return 0;
}
}  // namespace tcgemm
}  // namespace plnlp

extern "C" int plnlp_gemm_tf32(int passes, int transa, int transb, int64_t M, int64_t N, int64_t K, const float* A,
                               int64_t lda, const float* B, int64_t ldb, float* C, int64_t ldc, float beta,
                               const float* bias, int act, const float* aux, int64_t ldaux, float drop_p,
                               uint64_t seed, float* workspace, int64_t workspace_bytes, int split_k,
                               void* stream) {
    using namespace plnlp;
    PLNLP_REQUIRE(passes == 1 || passes == 3, PLNLP_E_UNSUPPORTED);
    PLNLP_REQUIRE(M >= 0 && N >= 0 && K >= 0, PLNLP_E_SIZE);
    if (M == 0 || N == 0) return 0;
    PLNLP_REQUIRE(C && (K == 0 || (A && B)), PLNLP_E_NULL);     // K = 0 reads neither operand (empty tensors: NULL)
    PLNLP_REQUIRE(lda >= (transa ? M : K) && ldb >= (transb ? K : N) && ldc >= N, PLNLP_E_SIZE);
    PLNLP_REQUIRE(act >= 0 && act <= 2 && drop_p >= 0.0f && drop_p < 1.0f, PLNLP_E_SIZE);
    if (act == PLNLP_ACT_RELU_GRAD) PLNLP_REQUIRE(aux && ldaux >= N, PLNLP_E_NULL);
    if (split_k < 1 || K == 0) split_k = 1;
    TcGemmParams p{};
    p.M = M; p.N = N; p.K = K; p.A = A; p.lda = lda; p.B = B; p.ldb = ldb; p.C = C; p.ldc = ldc;
    p.beta = beta; p.bias = bias; p.act = act; p.aux = aux; p.ldaux = ldaux; p.drop_p = drop_p; p.seed = seed;
    p.passes = passes;
    int64_t kper = ceil_div(ceil_div(K, split_k), TBK) * TBK;
    if (kper == 0) kper = TBK;
    p.k_per_split = kper;
    p.split_k = split_k = static_cast<int>(K == 0 ? 1 : ceil_div(K, kper));
    p.ws = workspace;
    if (split_k > 1) {
        PLNLP_REQUIRE(workspace, PLNLP_E_NULL);
        PLNLP_REQUIRE(workspace_bytes >= static_cast<int64_t>(split_k) * M * N * 4, PLNLP_E_WORKSPACE);
        PLNLP_REQUIRE(aligned(workspace, 16), PLNLP_E_ALIGN);
    }
    const bool amn = transa != 0, bmn = transb == 0;
    const bool va = aligned(A, 16) && (lda % 4 == 0) && ((transa ? M : K) % 4 == 0);
    const bool vb = aligned(B, 16) && (ldb % 4 == 0) && ((transb ? K : N) % 4 == 0);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    int rc;
    if (N > 128) {
        const dim3 grid(static_cast<unsigned>(ceil_div(N, 256)), static_cast<unsigned>(ceil_div(M, TBM)),
                        static_cast<unsigned>(split_k));
        rc = launch_major<256>(p, amn, bmn, va, vb, grid, st);
    } else {
        const dim3 grid(static_cast<unsigned>(ceil_div(N, 128)), static_cast<unsigned>(ceil_div(M, TBM)),
                        static_cast<unsigned>(split_k));
        rc = launch_major<128>(p, amn, bmn, va, vb, grid, st);
    }
    if (rc != 0) return rc;
    PLNLP_LAUNCH_CHECK();
    if (split_k > 1) return tcgemm::tc_splitk_reduce(p, st);
    return 0;
}
