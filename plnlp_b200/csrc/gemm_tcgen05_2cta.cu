// Tensor-core GEMM for sm_100a with CTA PAIRS: tcgen05.mma.cta_group::2 kind::tf32.
//
// Same contract, operand layout, loader and epilogue as gemm_tcgen05.cu (see there); what changes is
// who multiplies what.  A cluster of two CTAs (the two SMs of one TPC) computes one 256 x 256 output
// tile: CTA r of the pair stages ITS 128 rows of A and ITS HALF (<= 128 rows) of the B tile; the leader
// CTA (cluster rank 0) issues one M = 256 MMA per k-step that reads both CTAs' shared memory and
// writes 128 accumulator rows into each CTA's TMEM.  Per unit of work every SM now reads / converts /
// stores half as much of B -- the kernel is bound by the L1 / shared-memory SRAM bandwidth
// (DESIGN.md), so this is where the time goes.
//
// Synchronisation per ring stage s (both CTAs run the same code):
//   loaders (256 threads / CTA): wait empty[s] (local) -> st.shared tiles -> fence.proxy.async ->
//                                arrive full[s] (local, count 256)
//   CTA 1, warp 8 (relay)      : wait full[s] -> ONE remote arrive (release.cluster) on the leader's peer[s]
//   CTA 0, warp 8 (MMA issuer) : wait full[s] and peer[s] (acquire.cluster) -> tcgen05.mma.cta_group::2 x
//                                k-steps x passes -> tcgen05.commit multicast to empty[s] of BOTH CTAs
//   last k-slab                : commit multicast to accum of both CTAs -> each CTA runs the epilogue for
//                                its own 128 rows.
#include <type_traits>

#include "gemm_tc_common.cuh"

namespace plnlp {

namespace {

using namespace tcgemm;

constexpr int BN2 = 256;     // pair tile columns (UMMA N, TMEM columns per CTA)
constexpr int BH2 = 128;     // B rows staged per CTA

template <bool SPLIT>
struct Cfg2 {
    static constexpr int STAGES = SPLIT ? 3 : 6;      // 2 CTAs per SM share the 227 KB
};

// AMODE: 0 = A read as stored; 1 = A gathered (GatherLoader): fused edge scoring forward, see plnlp_edge_mlp_fwd_tf32
// below; 2 = A = dZ1 formed from the stored activation (DzLoader): fused edge scoring backward, plnlp_edge_mlp_bwd_tf32.
// BHAD: the (MN-major) B operand is the re-gathered Hadamard product (HadamardLoaderMN).
template <bool AMN, bool BMN, bool VA, bool VB, bool SPLIT, int AMODE = 0, bool BHAD = false>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NTHREADS, 2)
    gemm_tcgen05_2cta_kernel(const TcGemmParams p) {
    constexpr bool AGATHER = AMODE == 1;
    static_assert(!BHAD || BMN, "the Hadamard B operand is MN-major");
    constexpr int STAGES = Cfg2<SPLIT>::STAGES;
    constexpr int A_SLOT = slot_bytes(TBM), B_SLOT = slot_bytes(BH2);
    constexpr int STAGE_BYTES = (SPLIT ? 2 : 1) * (A_SLOT + B_SLOT);
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ __align__(8) uint64_t full_bar[STAGES], peer_bar[STAGES], empty_bar[STAGES], accum_bar;
    __shared__ uint32_t tmem_holder;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t rank = tc::cluster_ctarank();
    const int64_t m0 = static_cast<int64_t>(blockIdx.x >> 1) * (2 * TBM) + rank * TBM;
    const int64_t n0 = static_cast<int64_t>(blockIdx.y) * BN2;
    const int64_t kbeg = static_cast<int64_t>(blockIdx.z) * p.k_per_split;
    const int64_t kend = min(p.K, kbeg + p.k_per_split);
    const int n_iter = static_cast<int>((kend - kbeg + TBK - 1) / TBK);
    const int64_t n_rem = ((p.N - n0 + 15) / 16) * 16;
    const int n_mma = n_rem < BN2 ? static_cast<int>(n_rem) : BN2;     // multiple of 16
    const int bhalf = n_mma / 2;                                       // B rows this CTA supplies

    if (tid == 0) {
        for (int s = 0; s < STAGES; ++s) {
            tc::mbar_init(&full_bar[s], LOADERS);
            tc::mbar_init(&peer_bar[s], 1);
            tc::mbar_init(&empty_bar[s], 1);
        }
        tc::mbar_init(&accum_bar, 1);
        tc::mbar_fence_init();
    }
    if (warp == 8) tc::tmem_alloc_2cta<BN2>(&tmem_holder);
    tc::fence_before_sync();
    tc::cluster_sync();              // barriers of BOTH CTAs are initialised before anyone signals them
    tc::fence_after_sync();
    const uint32_t tmem_d = tmem_holder;

    auto stage_ptr = [&](int s, int which) -> uint8_t* {  // which: 0 A.hi, 1 B.hi, 2 A.lo, 3 B.lo
        uint8_t* base = smem + s * STAGE_BYTES;
        return base + (which & 1 ? A_SLOT : 0) + (which & 2 ? (A_SLOT + B_SLOT) : 0);
    };

    if (warp < 8) {
        // ============================ loaders ============================
        float ra[2][nreg(TBM, AMN)][4], rb[2][nreg(BH2, BMN)][4];
        typename std::conditional<AGATHER, GatherLoader<TBM, VA>,
                                  typename std::conditional<AMODE == 2, DzLoader<TBM, AMN, VA>,
                                                            Loader<TBM, AMN, VA>>::type>::type la;
        typename std::conditional<BHAD, HadamardLoaderMN<BH2, VB>, Loader<BH2, BMN, VB>>::type lb;
        const int64_t b0 = n0 + static_cast<int64_t>(rank) * bhalf;
        const int64_t b_end = (b0 + bhalf) < p.N ? (b0 + bhalf) : p.N;   // rows past this CTA's half are zero
        const int ktot = static_cast<int>(kend - kbeg);
        if constexpr (AGATHER) la.init(p.A, p.lda, p.a_rows, p.a_edges, m0, p.M, kbeg, tid);
        else if constexpr (AMODE == 2) la.init(p.A, p.lda, m0, p.M, kbeg, p.dz_dscore, p.dz_w2, p.dz_scale, tid);
        else la.init(p.A, p.lda, m0, p.M, kbeg, tid);
        if constexpr (BHAD) lb.init(p.B, p.ldb, p.b_rows, p.b_edges, b0, b_end, kbeg, ktot, tid);
        else lb.init(p.B, p.ldb, b0, b_end, kbeg, tid);
        auto fetch = [&](int it, float (&a)[nreg(TBM, AMN)][4], float (&b)[nreg(BH2, BMN)][4]) {
            if (it < n_iter) {
                la.fetch(ktot - it * TBK, a);
                lb.fetch(ktot - it * TBK, b);
            }
        };
        auto publish = [&](int it, const float (&a)[nreg(TBM, AMN)][4], const float (&b)[nreg(BH2, BMN)][4]) {
            const int s = it % STAGES;
            const uint32_t ph = (it / STAGES) & 1;
            tc::mbar_wait(&empty_bar[s], ph ^ 1);
            la.template stash<SPLIT>(stage_ptr(s, 0), stage_ptr(s, 2), a);
            lb.template stash<SPLIT>(stage_ptr(s, 1), stage_ptr(s, 3), b);
#ifndef PLNLP_CONSUMER_SIDE_PROXY_FENCE
            tc::fence_proxy_async_smem();
#endif
            tc::mbar_arrive(&full_bar[s]);
        };
        fetch(0, ra[0], rb[0]);
        fetch(1, ra[1], rb[1]);
        for (int it = 0; it < n_iter; it += 2) {
            publish(it, ra[0], rb[0]);
            fetch(it + 2, ra[0], rb[0]);
            if (it + 1 < n_iter) {
                publish(it + 1, ra[1], rb[1]);
                fetch(it + 3, ra[1], rb[1]);
            }
        }
    } else if (rank == 0) {
        // ============================ MMA issuer (leader CTA) ============================
        const uint32_t idesc = tc::make_idesc_tf32(2 * TBM, n_mma, 0, 0);
        constexpr uint32_t A_LBO = tile_lbo(TBM), B_LBO = tile_lbo(BH2);
        constexpr uint32_t A_STEP = 2 * A_LBO, B_STEP = 2 * B_LBO;
        for (int it = 0; it < n_iter; ++it) {
            const int s = it % STAGES;
            const uint32_t ph = (it / STAGES) & 1;
            tc::mbar_wait(&full_bar[s], ph);
            tc::mbar_wait_cluster(&peer_bar[s], ph);
#ifdef PLNLP_CONSUMER_SIDE_PROXY_FENCE
            tc::fence_proxy_async_smem();     // EXPERIMENT: proxy fence on the consumer side only
#endif
            tc::fence_after_sync();
            if (lane == 0) {
                const uint32_t a_hi = tc::smem_u32(stage_ptr(s, 0)), b_hi = tc::smem_u32(stage_ptr(s, 1));
                const uint32_t a_lo = tc::smem_u32(stage_ptr(s, 2)), b_lo = tc::smem_u32(stage_ptr(s, 3));
#pragma unroll
                for (int j = 0; j < TBK / 8; ++j) {
                    const uint64_t dah = tc::make_smem_desc(a_hi + j * A_STEP, A_LBO, TILE_SBO);
                    const uint64_t dbh = tc::make_smem_desc(b_hi + j * B_STEP, B_LBO, TILE_SBO);
                    tc::mma_tf32_ss_2cta(tmem_d, dah, dbh, idesc, (it | j) != 0);
                    if (SPLIT) {
                        const uint64_t dal = tc::make_smem_desc(a_lo + j * A_STEP, A_LBO, TILE_SBO);
                        const uint64_t dbl = tc::make_smem_desc(b_lo + j * B_STEP, B_LBO, TILE_SBO);
                        tc::mma_tf32_ss_2cta(tmem_d, dah, dbl, idesc, 1u);
                        tc::mma_tf32_ss_2cta(tmem_d, dal, dbh, idesc, 1u);
                    }
                }
                tc::mma_commit_2cta(&empty_bar[s], 3);
                if (it == n_iter - 1) tc::mma_commit_2cta(&accum_bar, 3);
            }
            __syncwarp();
        }
    } else {
        // ============================ relay (peer CTA) ============================
        for (int it = 0; it < n_iter; ++it) {
            const int s = it % STAGES;
            const uint32_t ph = (it / STAGES) & 1;
            tc::mbar_wait(&full_bar[s], ph);
            if (lane == 0) tc::mbar_arrive_remote(&peer_bar[s], 0);
            __syncwarp();
        }
    }

    // ============================ epilogue (warps 0-7 of each CTA, its own 128 rows) ============
    if (warp < 8) {
        if (n_iter > 0) {
            tc::mbar_wait(&accum_bar, 0);
            tc::fence_after_sync();
        }
        tc_epilogue_tile<BN2>(p, tmem_d, m0, n0, n_mma, n_iter, warp, lane);
    }
    tc::fence_before_sync();
    tc::cluster_sync();              // the peer's shared memory / TMEM stay alive until both are done
    if (warp == 8) tc::tmem_dealloc_2cta<BN2>(tmem_d);
}

template <bool AMN, bool BMN, bool VA, bool VB, bool SPLIT, int AMODE = 0, bool BHAD = false>
int launch_one2(const TcGemmParams& p, dim3 grid, cudaStream_t st) {
    constexpr int bytes = Cfg2<SPLIT>::STAGES * (SPLIT ? 2 : 1) * (slot_bytes(TBM) + slot_bytes(BH2));
    static_assert(bytes <= 113 * 1024, "two CTAs per SM");
    auto kern = gemm_tcgen05_2cta_kernel<AMN, BMN, VA, VB, SPLIT, AMODE, BHAD>;
    static bool configured = false;
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
        if (e != cudaSuccess) return static_cast<int>(e);
        configured = true;
    }
    kern<<<grid, NTHREADS, bytes, st>>>(p);
    return 0;
}

template <bool AMN, bool BMN>
int launch_vec2(const TcGemmParams& p, bool va, bool vb, dim3 grid, cudaStream_t st) {
    const bool split = p.passes == 3;
    if (va && vb) {
        return split ? launch_one2<AMN, BMN, true, true, true>(p, grid, st)
                     : launch_one2<AMN, BMN, true, true, false>(p, grid, st);
    }
    if (va) return launch_one2<AMN, BMN, true, false, true>(p, grid, st);
    if (vb) return launch_one2<AMN, BMN, false, true, true>(p, grid, st);
    return launch_one2<AMN, BMN, false, false, true>(p, grid, st);
}

}  // namespace
}  // namespace plnlp

extern "C" int plnlp_gemm_tf32_2cta(int passes, int transa, int transb, int64_t M, int64_t N, int64_t K,
                                    const float* A, int64_t lda, const float* B, int64_t ldb, float* C,
                                    int64_t ldc, float beta, const float* bias, int act, const float* aux,
                                    int64_t ldaux, float drop_p, uint64_t seed, float* workspace,
                                    int64_t workspace_bytes, int split_k, void* stream) {
    using namespace plnlp;
    using namespace plnlp::tcgemm;
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
    // grid.x = 2 CTAs per 256-row pair tile (cluster dimension 2 along x)
    const dim3 grid(static_cast<unsigned>(2 * ceil_div(M, 2 * TBM)), static_cast<unsigned>(ceil_div(N, BN2)),
                    static_cast<unsigned>(split_k));
    int rc;
    if (!amn && !bmn) rc = launch_vec2<false, false>(p, va, vb, grid, st);
    else if (!amn && bmn) rc = launch_vec2<false, true>(p, va, vb, grid, st);
    else if (amn && !bmn) rc = launch_vec2<true, false>(p, va, vb, grid, st);
    else rc = launch_vec2<true, true>(p, va, vb, grid, st);
    if (rc != 0) return rc;
    PLNLP_LAUNCH_CHECK();
    if (split_k > 1) {
        // the split-k reduction (and its epilogue) is shared with the 1-CTA kernel
        return tc_splitk_reduce(p, st);
    }
    return 0;
}


// Fused edge scoring, MLP head forward (SURVEY.md a7/a9; model.py:152-156 + layer.py:80-87 for the usual
// 2-layer head): for every pair p
//     a0 = h[src_p] * h[dst_p]                       gathered by the loader, never written to HBM
//     a1 = dropout(relu(a0 @ W1^T + b1))             tensor cores; written to `a1` only if a1 != NULL
//     score_part[q][p] = a1[p, cols of partial q] . w2
// The caller adds the 2*ceil(N1/256) partials in index order and the output bias.
extern "C" int plnlp_edge_mlp_fwd_tf32(int passes, const float* h, int64_t ldh, int64_t n_rows, const int64_t* edges,
                                       int64_t P, int64_t H, const float* W1, int64_t ldw, const float* b1,
                                       int64_t N1, float drop_p, uint64_t seed, const float* w2, float* a1,
                                       int64_t lda1, float* score_part, int64_t score_ld, void* stream) {
    using namespace plnlp;
    using namespace plnlp::tcgemm;
    PLNLP_REQUIRE(passes == 1 || passes == 3, PLNLP_E_UNSUPPORTED);
    PLNLP_REQUIRE(P >= 0 && H > 0 && N1 > 0 && n_rows > 0, PLNLP_E_SIZE);
    if (P == 0) return 0;
    PLNLP_REQUIRE(h && edges && W1 && w2 && score_part, PLNLP_E_NULL);
    PLNLP_REQUIRE(ldh >= H && ldw >= H && score_ld >= P && (!a1 || lda1 >= N1), PLNLP_E_SIZE);
    PLNLP_REQUIRE(H <= 1024, PLNLP_E_UNSUPPORTED);     // one accumulator: keep K within the RZ error budget
    PLNLP_REQUIRE(drop_p >= 0.0f && drop_p < 1.0f, PLNLP_E_SIZE);
    TcGemmParams p{};
    p.M = P; p.N = N1; p.K = H; p.A = h; p.lda = ldh; p.B = W1; p.ldb = ldw; p.C = a1; p.ldc = lda1;
    p.beta = 0.0f; p.bias = b1; p.act = PLNLP_ACT_RELU; p.drop_p = drop_p; p.seed = seed; p.passes = passes;
    p.split_k = 1; p.k_per_split = ceil_div(H, TBK) * TBK;
    p.a_edges = edges; p.a_rows = n_rows; p.w_out = w2; p.score_part = score_part; p.score_ld = score_ld;
    const bool va = aligned(h, 16) && (ldh % 4 == 0) && (H % 4 == 0);
    const bool vb = aligned(W1, 16) && (ldw % 4 == 0) && (H % 4 == 0);
    const dim3 grid(static_cast<unsigned>(2 * ceil_div(P, 2 * TBM)), static_cast<unsigned>(ceil_div(N1, BN2)), 1);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    int rc;
    if (va && vb) {
        rc = passes == 3 ? launch_one2<false, false, true, true, true, 1>(p, grid, st)
                         : launch_one2<false, false, true, true, false, 1>(p, grid, st);
    } else {
        rc = launch_one2<false, false, false, false, true, 1>(p, grid, st);
    }
    if (rc != 0) return rc;
    PLNLP_LAUNCH_CHECK();
    return 0;
}


// Fused edge scoring, MLP head BACKWARD (model.py:161 through layer.py:80-87): with a1 = dropout(relu(a0 W1^T + b1))
// stored by the forward and dscore = d loss / d score from the pair loss,
//     dZ1 = (dscore (x) w2) . [a1 > 0] * drop_scale        formed in the loaders, never written to HBM
//     dA0 = dZ1 @ W1                    [P, H]             (the gradient of the Hadamard product, scattered next)
//     dW1 = dZ1^T @ (h[src] * h[dst])   [N1, H]            the Hadamard product re-gathered by the loader
// Two launches (+ the split-k reduction of dW1).  dw2 / db2 / db1 come from plnlp_mlp_out_bwd_f32 with dz = NULL.
extern "C" int64_t plnlp_edge_mlp_bwd_workspace_bytes(int64_t P, int64_t H, int64_t N1, int split_k) {
    if (P <= 0 || H <= 0 || N1 <= 0) return 0;
    if (split_k < 1) split_k = 1;
    return static_cast<int64_t>(split_k) * N1 * H * 4 + 16;
}

extern "C" int plnlp_edge_mlp_bwd_tf32(int passes, const float* h, int64_t ldh, int64_t n_rows, const int64_t* edges,
                                       int64_t P, int64_t H, const float* W1, int64_t ldw, int64_t N1,
                                       const float* a1, int64_t lda1, const float* dscore, const float* w2,
                                       float drop_scale, float* dA0, int64_t ldda0, float* dW1, int64_t lddw1,
                                       float* workspace, int64_t workspace_bytes, int split_k, void* stream) {
    using namespace plnlp;
    using namespace plnlp::tcgemm;
    PLNLP_REQUIRE(passes == 1 || passes == 3, PLNLP_E_UNSUPPORTED);
    PLNLP_REQUIRE(P >= 0 && H > 0 && N1 > 0 && n_rows > 0, PLNLP_E_SIZE);
    if (P == 0) return 0;
    PLNLP_REQUIRE(h && edges && W1 && a1 && dscore && w2 && dA0 && dW1, PLNLP_E_NULL);
    PLNLP_REQUIRE(ldh >= H && ldw >= H && lda1 >= N1 && ldda0 >= H && lddw1 >= H, PLNLP_E_SIZE);
    PLNLP_REQUIRE(N1 <= 1088, PLNLP_E_UNSUPPORTED);      // dA0 uses one accumulator over K = N1 (RZ error budget)
    // the loaders use whole 16-byte vectors
    PLNLP_REQUIRE((H % 4 == 0) && (N1 % 4 == 0) && (ldh % 4 == 0) && (ldw % 4 == 0) && (lda1 % 4 == 0), PLNLP_E_ALIGN);
    PLNLP_REQUIRE(aligned(h, 16) && aligned(W1, 16) && aligned(a1, 16), PLNLP_E_ALIGN);
    cudaStream_t st = static_cast<cudaStream_t>(stream);

    // ---- dA0 = dZ1 @ W1: M = P, N = H, K = N1; A = dZ1 (K-major, from a1), B[k = c, n = j] = W1[c*ldw + j] (MN-major)
    {
        TcGemmParams p{};
        p.M = P; p.N = H; p.K = N1; p.A = a1; p.lda = lda1; p.B = W1; p.ldb = ldw; p.C = dA0; p.ldc = ldda0;
        p.passes = passes; p.split_k = 1; p.k_per_split = ceil_div(N1, TBK) * TBK;
        p.dz_dscore = dscore; p.dz_w2 = w2; p.dz_scale = drop_scale;
        const dim3 grid(static_cast<unsigned>(2 * ceil_div(P, 2 * TBM)), static_cast<unsigned>(ceil_div(H, BN2)), 1);
        int rc = passes == 3 ? launch_one2<false, true, true, true, true, 2>(p, grid, st)
                             : launch_one2<false, true, true, true, false, 2>(p, grid, st);
        if (rc != 0) return rc;
        PLNLP_LAUNCH_CHECK();
    }
    // ---- dW1 = dZ1^T @ a0: M = N1, N = H, K = P; A[m = c, k = p] = dZ1[p, c] (MN-major, from a1),
    //      B[k = p, n = j] = h[src_p, j] * h[dst_p, j] (MN-major, gathered)
    {
        if (split_k < 1) split_k = 1;
        TcGemmParams p{};
        p.M = N1; p.N = H; p.K = P; p.A = a1; p.lda = lda1; p.B = h; p.ldb = ldh; p.C = dW1; p.ldc = lddw1;
        p.passes = passes;
        int64_t kper = ceil_div(ceil_div(P, split_k), TBK) * TBK;
        p.k_per_split = kper;
        p.split_k = split_k = static_cast<int>(ceil_div(P, kper));
        p.ws = workspace;
        if (split_k > 1) {
            PLNLP_REQUIRE(workspace, PLNLP_E_NULL);
            PLNLP_REQUIRE(workspace_bytes >= static_cast<int64_t>(split_k) * N1 * H * 4, PLNLP_E_WORKSPACE);
            PLNLP_REQUIRE(aligned(workspace, 16), PLNLP_E_ALIGN);
        }
        p.dz_dscore = dscore; p.dz_w2 = w2; p.dz_scale = drop_scale;
        p.b_edges = edges; p.b_rows = n_rows;
        PLNLP_REQUIRE(aligned(dscore, 16), PLNLP_E_ALIGN);
        const dim3 grid(static_cast<unsigned>(2 * ceil_div(N1, 2 * TBM)), static_cast<unsigned>(ceil_div(H, BN2)),
                        static_cast<unsigned>(split_k));
        int rc = passes == 3 ? launch_one2<true, true, true, true, true, 2, true>(p, grid, st)
                             : launch_one2<true, true, true, true, false, 2, true>(p, grid, st);
        if (rc != 0) return rc;
        PLNLP_LAUNCH_CHECK();
        if (split_k > 1) return tc_splitk_reduce(p, st);
    }
    return 0;
}
