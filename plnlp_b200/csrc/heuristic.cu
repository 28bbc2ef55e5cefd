// Common-neighbour link heuristics (plnlp_b200/heuristics.py): for every pair edges[p] = (u, v),
//
//   out[p] = sum over w in N(u) & N(v) of weight[w]     (weight == NULL: 1 per common neighbour -> CN)
//
// in fp64, over a cleaned CSR (rows sorted, distinct, diagonal-free int32 columns).  Adamic-Adar and Resource
// Allocation are the weight tables 1 / ln d(w) and 1 / d(w), built by the caller.
//
// One warp per pair; pairs are strided over the warps of the grid.  Hub rows of power-law graphs must not serialise a
// warp, so each pair takes the cheaper of two warp-parallel intersections, chosen from the two lengths alone:
//   * search: lane l walks entries l, l + 32, ... of the SHORTER list and binary-searches each in the longer one
//     (its keys ascend, so each search starts where the lane's previous one ended) -- for a short list against a hub;
//   * merge : the merge path of the two lists is cut into 32 equal diagonals; lane l finds its start by one binary
//     search and merges its 1/32 of the path, counting a common neighbour where it consumes it from the shorter list
//     (ties consume the shorter list first, so every common neighbour is counted exactly once) -- for hub-hub pairs.
// Every lane adds its terms in list order, then a fixed xor-butterfly sums the 32 lane totals: the result depends on
// the two lists only and is the same on every run.
#include "common.cuh"

namespace plnlp {
namespace {

constexpr int kHeurThreads = 256;

__device__ __forceinline__ int ilog2_ceil(int64_t x) {
    // ceil(log2(x + 1)): the steps of a binary search over x entries
    return 64 - __clzll(static_cast<unsigned long long>(x));
}

__global__ void __launch_bounds__(kHeurThreads) link_heuristic_kernel(const int64_t* __restrict__ rowptr,
                                                                     const int32_t* __restrict__ col,
                                                                     const double* __restrict__ weight,
                                                                     const int64_t* __restrict__ edges, int64_t P,
                                                                     double* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int64_t n_warps = (static_cast<int64_t>(gridDim.x) * blockDim.x) >> 5;
    for (int64_t p = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5; p < P; p += n_warps) {
        const int64_t u = __ldg(edges + 2 * p), v = __ldg(edges + 2 * p + 1);
        int64_t a0 = __ldg(rowptr + u), a1 = __ldg(rowptr + u + 1);
        int64_t b0 = __ldg(rowptr + v), b1 = __ldg(rowptr + v + 1);
        if (a1 - a0 > b1 - b0) {                    // a: the shorter list
            int64_t t = a0; a0 = b0; b0 = t;
            t = a1; a1 = b1; b1 = t;
        }
        const int64_t la = a1 - a0, lb = b1 - b0;
        const int32_t* A = col + a0;
        const int32_t* B = col + b0;
        double acc = 0.0;
        if (la > 0) {
            const int64_t steps_search = ((la + 31) >> 5) * ilog2_ceil(lb);
            const int64_t steps_merge = ((la + lb + 31) >> 5) + ilog2_ceil(la);
            if (steps_search <= steps_merge) {
                int64_t lo = 0;
                for (int64_t i = lane; i < la; i += 32) {
                    const int32_t w = __ldg(A + i);
                    int64_t hi = lb;
                    while (lo < hi) {                   // lower bound of w in B[lo, lb)
                        const int64_t m = (lo + hi) >> 1;
                        if (__ldg(B + m) < w) lo = m + 1; else hi = m;
                    }
                    if (lo < lb && __ldg(B + lo) == w) acc += weight ? __ldg(weight + w) : 1.0;
                }
            } else {
                const int64_t L = la + lb;
                const int64_t d0 = (L * lane) >> 5, d1 = (L * (lane + 1)) >> 5;
                // i = entries of A among the first d0 of the merge (A first on ties): the largest i with
                // A[i - 1] <= B[d0 - i]
                int64_t lo = d0 > lb ? d0 - lb : 0, hi = d0 < la ? d0 : la;
                while (lo < hi) {
                    const int64_t m = (lo + hi) >> 1;
                    if (__ldg(A + m) <= __ldg(B + d0 - m - 1)) lo = m + 1; else hi = m;
                }
                int64_t i = lo, j = d0 - lo;
                int32_t x = i < la ? __ldg(A + i) : INT32_MAX;
                int32_t y = j < lb ? __ldg(B + j) : INT32_MAX;
                for (int64_t d = d0; d < d1; ++d) {
                    if (i < la && (j >= lb || x <= y)) {
                        if (x == y) acc += weight ? __ldg(weight + x) : 1.0;
                        ++i;
                        x = i < la ? __ldg(A + i) : INT32_MAX;
                    } else {
                        ++j;
                        y = j < lb ? __ldg(B + j) : INT32_MAX;
                    }
                }
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (lane == 0) out[p] = acc;
    }
}

}  // namespace
}  // namespace plnlp

// out [P] fp64; rowptr int64 [n + 1] and col int32 [nnz] a cleaned CSR; edges int64 [P, 2] with ids in [0, n);
// weight fp64 [n] or NULL (CN)
extern "C" int plnlp_link_heuristic_f64(const int64_t* rowptr, const int32_t* col, int64_t n, int64_t nnz,
                                        const double* weight, const int64_t* edges, int64_t P, double* out,
                                        void* stream) {
    PLNLP_REQUIRE(n >= 0 && nnz >= 0 && P >= 0, PLNLP_E_SIZE);
    if (P == 0) return 0;
    PLNLP_REQUIRE(n > 0, PLNLP_E_SIZE);
    PLNLP_REQUIRE(rowptr && edges && out && (nnz == 0 || col), PLNLP_E_NULL);
    const int64_t blocks = std::min<int64_t>(plnlp::ceil_div(P, plnlp::kHeurThreads / 32), int64_t(plnlp::kNumSM) * 8);
    plnlp::link_heuristic_kernel<<<static_cast<unsigned>(blocks), plnlp::kHeurThreads, 0,
                                   static_cast<cudaStream_t>(stream)>>>(rowptr, col, weight, edges, P, out);
    PLNLP_LAUNCH_CHECK();
    return 0;
}
