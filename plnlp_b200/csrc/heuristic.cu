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

// The intersection skeleton shared by the sum and the list: N(u) & N(v) walked by the whole warp with the cheaper of
// the two modes above.  The argument order matters only for equal lengths (u's list is then the "shorter" one);
// callers pass (query, other).  The visitor sees the common neighbours:
//   * search: vis.search(hit, w) for each entry w of the shorter list a lane takes, in order.  With
//     Visitor::kWarpRounds every lane runs every 32-entry round (hit false past the end), so the visitor may ballot;
//   * merge : vis.merge(walk) once; walk(f) calls f(w) for the lane's common neighbours, in list order, and may be
//     called more than once.
template <class Visitor>
__device__ __forceinline__ void warp_intersect(const int64_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                                               int64_t u, int64_t v, int lane, Visitor& vis) {
    int64_t a0 = __ldg(rowptr + u), a1 = __ldg(rowptr + u + 1);
    int64_t b0 = __ldg(rowptr + v), b1 = __ldg(rowptr + v + 1);
    if (a1 - a0 > b1 - b0) {                    // a: the shorter list
        int64_t t = a0; a0 = b0; b0 = t;
        t = a1; a1 = b1; b1 = t;
    }
    const int64_t la = a1 - a0, lb = b1 - b0;
    const int32_t* A = col + a0;
    const int32_t* B = col + b0;
    if (la == 0) return;
    const int64_t steps_search = ((la + 31) >> 5) * ilog2_ceil(lb);
    const int64_t steps_merge = ((la + lb + 31) >> 5) + ilog2_ceil(la);
    if (steps_search <= steps_merge) {
        int64_t lo = 0;
        const int64_t end = Visitor::kWarpRounds ? ((la + 31) & ~int64_t(31)) : la;
        for (int64_t i = lane; i < end; i += 32) {
            int32_t w = 0;
            bool hit = false;
            if (i < la) {
                w = __ldg(A + i);
                int64_t hi = lb;
                while (lo < hi) {                   // lower bound of w in B[lo, lb)
                    const int64_t m = (lo + hi) >> 1;
                    if (__ldg(B + m) < w) lo = m + 1; else hi = m;
                }
                hit = lo < lb && __ldg(B + lo) == w;
            }
            vis.search(hit, w);
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
        const int64_t i_start = lo;
        vis.merge([&](auto&& f) {
            int64_t i = i_start, j = d0 - i_start;
            int32_t x = i < la ? __ldg(A + i) : INT32_MAX;
            int32_t y = j < lb ? __ldg(B + j) : INT32_MAX;
            for (int64_t d = d0; d < d1; ++d) {
                if (i < la && (j >= lb || x <= y)) {
                    if (x == y) f(x);
                    ++i;
                    x = i < la ? __ldg(A + i) : INT32_MAX;
                } else {
                    ++j;
                    y = j < lb ? __ldg(B + j) : INT32_MAX;
                }
            }
        });
    }
}

// the sum of weight[w] (1 when weight == NULL): lane terms in list order
struct SumVisitor {
    static constexpr bool kWarpRounds = false;
    const double* __restrict__ weight;
    double acc;
    __device__ __forceinline__ void add(int32_t w) { acc += weight ? __ldg(weight + w) : 1.0; }
    __device__ __forceinline__ void search(bool hit, int32_t w) {
        if (hit) add(w);
    }
    template <class Walk>
    __device__ __forceinline__ void merge(Walk&& walk) {
        walk([&](int32_t w) { add(w); });
    }
};

// the sum of weight[w] (1 when weight == NULL) over w in N(u) & N(v), computed by the whole warp and returned to
// every lane: the lane sums of warp_intersect, then the fixed butterfly
__device__ __forceinline__ double warp_common_neighbours(const int64_t* __restrict__ rowptr,
                                                         const int32_t* __restrict__ col,
                                                         const double* __restrict__ weight, int64_t u, int64_t v,
                                                         int lane) {
    SumVisitor vis{weight, 0.0};
    warp_intersect(rowptr, col, u, v, lane, vis);
    double acc = vis.acc;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    return acc;
}

// the list N(u) & N(v) in ascending id order, written to out[0 ..) by the whole warp
struct ListVisitor {
    static constexpr bool kWarpRounds = true;
    int32_t* __restrict__ out;
    int lane;
    int64_t base;       // entries written by the rounds before (search) -- warp-uniform
    __device__ __forceinline__ void search(bool hit, int32_t w) {
        // the rounds walk the shorter list in order and lane l holds entry l of the round: the hits of the lower
        // lanes come first
        const unsigned ballot = __ballot_sync(0xffffffffu, hit);
        if (hit) out[base + __popc(ballot & ((1u << lane) - 1u))] = w;
        base += __popc(ballot);
    }
    template <class Walk>
    __device__ __forceinline__ void merge(Walk&& walk) {
        // lane l's diagonal range follows lane l - 1's: count, exclusive warp scan, write
        int64_t cnt = 0;
        walk([&](int32_t) { ++cnt; });
        int64_t pos = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int64_t t = __shfl_up_sync(0xffffffffu, pos, o);
            if (lane >= o) pos += t;
        }
        pos = base + pos - cnt;
        walk([&](int32_t w) { out[pos++] = w; });
    }
};

__global__ void __launch_bounds__(kHeurThreads) link_heuristic_kernel(const int64_t* __restrict__ rowptr,
                                                                     const int32_t* __restrict__ col,
                                                                     const double* __restrict__ weight,
                                                                     const int64_t* __restrict__ edges, int64_t P,
                                                                     double* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int64_t n_warps = (static_cast<int64_t>(gridDim.x) * blockDim.x) >> 5;
    for (int64_t p = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5; p < P; p += n_warps) {
        const int64_t u = __ldg(edges + 2 * p), v = __ldg(edges + 2 * p + 1);
        // a negative id (the mean row of BaseModel.encode_for_test) has no neighbours
        const double acc = u < 0 || v < 0 ? 0.0 : warp_common_neighbours(rowptr, col, weight, u, v, lane);
        if (lane == 0) out[p] = acc;
    }
}

// one warp per pair: the common neighbours of edges[p] written to col_out[out_ptr[p] ..), ascending; a pair with a
// negative id has none
__global__ void __launch_bounds__(kHeurThreads) common_neighbour_list_kernel(const int64_t* __restrict__ rowptr,
                                                                            const int32_t* __restrict__ col,
                                                                            const int64_t* __restrict__ edges,
                                                                            int64_t P,
                                                                            const int64_t* __restrict__ out_ptr,
                                                                            int32_t* __restrict__ col_out) {
    const int lane = threadIdx.x & 31;
    const int64_t n_warps = (static_cast<int64_t>(gridDim.x) * blockDim.x) >> 5;
    for (int64_t p = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5; p < P; p += n_warps) {
        const int64_t u = __ldg(edges + 2 * p), v = __ldg(edges + 2 * p + 1);
        if (u < 0 || v < 0) continue;
        ListVisitor vis{col_out + __ldg(out_ptr + p), lane, 0};
        warp_intersect(rowptr, col, u, v, lane, vis);
    }
}

// the column of node j in a chunk: j - col0 when it lies in [col0, col0 + W), or, with cand (strictly ascending,
// W entries), its position there; -1 when the chunk has no such column
__device__ __forceinline__ int64_t chunk_column(const int64_t* __restrict__ cand, int64_t col0, int64_t W, int64_t j) {
    if (cand == nullptr) return j >= col0 && j - col0 < W ? j - col0 : -1;
    int64_t lo = 0, hi = W;
    while (lo < hi) {
        const int64_t m = (lo + hi) >> 1;
        if (__ldg(cand + m) < j) lo = m + 1; else hi = m;
    }
    return lo < W && __ldg(cand + lo) == j ? lo : -1;
}

// Mark: work item t in [0, item_ptr[Qc]) is (query qi, the (t - item_ptr[qi])-th w of N(nodes[qi])); one warp per
// item, items strided over the warps of the grid, lanes strided over R(w).  Every j of R(w) that has a column sets
// its bit; atomicOr makes the bitmap independent of the order.
__global__ void __launch_bounds__(kHeurThreads) two_hop_mark_kernel(
    const int64_t* __restrict__ rowptr, const int32_t* __restrict__ col, const int64_t* __restrict__ rrowptr,
    const int32_t* __restrict__ rcol, const int64_t* __restrict__ nodes, const int64_t* __restrict__ item_ptr,
    int64_t Qc, int64_t col0, int64_t W, const int64_t* __restrict__ cand, uint32_t* __restrict__ bitmap,
    int64_t words) {
    const int lane = threadIdx.x & 31;
    const int64_t n_warps = (static_cast<int64_t>(gridDim.x) * blockDim.x) >> 5;
    const int64_t total = __ldg(item_ptr + Qc);
    for (int64_t t = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5; t < total; t += n_warps) {
        int64_t lo = 0, hi = Qc;                    // the query: the last qi with item_ptr[qi] <= t
        while (hi - lo > 1) {
            const int64_t m = (lo + hi) >> 1;
            if (__ldg(item_ptr + m) <= t) lo = m; else hi = m;
        }
        const int64_t w = __ldg(col + __ldg(rowptr + __ldg(nodes + lo)) + (t - __ldg(item_ptr + lo)));
        uint32_t* row = bitmap + lo * words;
        const int64_t r1 = __ldg(rrowptr + w + 1);
        for (int64_t e = __ldg(rrowptr + w) + lane; e < r1; e += 32) {
            const int64_t c = chunk_column(cand, col0, W, __ldg(rcol + e));
            if (c >= 0) atomicOr(row + (c >> 5), 1u << (c & 31));
        }
    }
}

// Score: the bitmap [Qc, words] flattened; a warp takes runs of 32 words (one per lane, one coalesced load), skips
// the empty ones by ballot and, for every set bit of the others, intersects N(nodes[q]) with N(j) through
// warp_common_neighbours -- the routine of link_heuristic_kernel, so each entry equals that kernel's result for the
// pair (nodes[q], j) bit for bit.  Unmarked entries are left as they are (the caller zeroes s).
template <class T>
__global__ void __launch_bounds__(kHeurThreads) two_hop_score_kernel(
    const int64_t* __restrict__ rowptr, const int32_t* __restrict__ col, const double* __restrict__ weight,
    const int64_t* __restrict__ nodes, int64_t Qc, int64_t col0, const int64_t* __restrict__ cand,
    const uint32_t* __restrict__ bitmap, int64_t words, T* __restrict__ s, int64_t lds) {
    const int lane = threadIdx.x & 31;
    const int64_t n_warps = (static_cast<int64_t>(gridDim.x) * blockDim.x) >> 5;
    const int64_t total = Qc * words;
    for (int64_t g0 = ((static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5) * 32; g0 < total;
         g0 += n_warps * 32) {
        const int64_t g = g0 + lane;
        const uint32_t mine = g < total ? __ldg(bitmap + g) : 0u;
        unsigned live = __ballot_sync(0xffffffffu, mine != 0u);
        while (live) {
            const int src = __ffs(live) - 1;
            live &= live - 1;
            uint32_t bits = __shfl_sync(0xffffffffu, mine, src);
            const int64_t gw = g0 + src;
            const int64_t q = gw / words;
            const int64_t c_base = (gw - q * words) * 32;
            const int64_t u = __ldg(nodes + q);
            while (bits) {
                const int b = __ffs(static_cast<int>(bits)) - 1;
                bits &= bits - 1;
                const int64_t c = c_base + b;
                const int64_t j = cand != nullptr ? __ldg(cand + c) : col0 + c;
                const double acc = warp_common_neighbours(rowptr, col, weight, u, j, lane);
                if (lane == 0) s[q * lds + c] = static_cast<T>(acc);
            }
        }
    }
}

template <class T>
int two_hop_score(const int64_t* rowptr, const int32_t* col, int64_t n, int64_t nnz, const double* weight,
                  const int64_t* nodes, int64_t Qc, int64_t col0, int64_t W, const int64_t* cand,
                  const uint32_t* bitmap, T* s, int64_t lds, void* stream) {
    PLNLP_REQUIRE(n >= 0 && nnz >= 0 && Qc >= 0 && W >= 0 && col0 >= 0 && lds >= W, PLNLP_E_SIZE);
    if (Qc == 0 || W == 0) return 0;
    PLNLP_REQUIRE(n > 0, PLNLP_E_SIZE);
    PLNLP_REQUIRE(rowptr && nodes && bitmap && s && (nnz == 0 || col), PLNLP_E_NULL);
    const int64_t words = ceil_div(W, 32);
    const int64_t blocks = std::min<int64_t>(ceil_div(Qc * words, kHeurThreads), int64_t(kNumSM) * 8);
    two_hop_score_kernel<T><<<static_cast<unsigned>(blocks), kHeurThreads, 0, static_cast<cudaStream_t>(stream)>>>(
        rowptr, col, weight, nodes, Qc, col0, cand, bitmap, words, s, lds);
    PLNLP_LAUNCH_CHECK();
    return 0;
}

}  // namespace
}  // namespace plnlp

// out [P] fp64; rowptr int64 [n + 1] and col int32 [nnz] a cleaned CSR; edges int64 [P, 2] with ids in [-1, n) (a
// pair with a negative id scores 0); weight fp64 [n] or NULL (CN)
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

// col_out int32 [out_ptr[P]]: the common neighbours of every pair edges[p] (int64 [P, 2], ids in [-1, n)) at
// col_out[out_ptr[p] .. out_ptr[p + 1]), ascending.  out_ptr int64 [P + 1]: the running sum of the CN counts of
// plnlp_link_heuristic_f64 (weight NULL), out_ptr[0] = 0.  Same table as above.
extern "C" int plnlp_common_neighbour_list(const int64_t* rowptr, const int32_t* col, int64_t n, int64_t nnz,
                                           const int64_t* edges, int64_t P, const int64_t* out_ptr, int32_t* col_out,
                                           void* stream) {
    PLNLP_REQUIRE(n >= 0 && nnz >= 0 && P >= 0, PLNLP_E_SIZE);
    if (P == 0 || nnz == 0) return 0;       // no entries: every list is empty
    PLNLP_REQUIRE(n > 0, PLNLP_E_SIZE);
    PLNLP_REQUIRE(rowptr && col && edges && out_ptr && col_out, PLNLP_E_NULL);
    const int64_t blocks = std::min<int64_t>(plnlp::ceil_div(P, plnlp::kHeurThreads / 32), int64_t(plnlp::kNumSM) * 8);
    plnlp::common_neighbour_list_kernel<<<static_cast<unsigned>(blocks), plnlp::kHeurThreads, 0,
                                          static_cast<cudaStream_t>(stream)>>>(rowptr, col, edges, P, out_ptr,
                                                                               col_out);
    PLNLP_LAUNCH_CHECK();
    return 0;
}

// bitmap uint32 [Qc, ceil(W / 32)], zeroed by the caller: bit c of row qi is set when column c's node j is reachable
// from nodes[qi] in two steps, j in R(w) for some w in N(nodes[qi]).  rowptr / col: the cleaned table N; rrowptr /
// rcol: its transpose R; item_ptr int64 [Qc + 1]: the running sum of |N(nodes[qi])|, item_ptr[0] = 0.  Columns: the
// nodes [col0, col0 + W), or cand[0 .. W) (strictly ascending) when cand != NULL (then col0 = 0).
extern "C" int plnlp_two_hop_mark(const int64_t* rowptr, const int32_t* col, const int64_t* rrowptr,
                                  const int32_t* rcol, int64_t n, const int64_t* nodes, const int64_t* item_ptr,
                                  int64_t Qc, int64_t col0, int64_t W, const int64_t* cand, uint32_t* bitmap,
                                  void* stream) {
    PLNLP_REQUIRE(n >= 0 && Qc >= 0 && W >= 0 && col0 >= 0, PLNLP_E_SIZE);
    PLNLP_REQUIRE(cand == nullptr || col0 == 0, PLNLP_E_UNSUPPORTED);
    if (Qc == 0 || W == 0) return 0;
    PLNLP_REQUIRE(n > 0, PLNLP_E_SIZE);
    PLNLP_REQUIRE(rowptr && col && rrowptr && rcol && nodes && item_ptr && bitmap, PLNLP_E_NULL);
    const int64_t words = plnlp::ceil_div(W, 32);
    const int64_t blocks = int64_t(plnlp::kNumSM) * 8;      // the item count stays on the device
    plnlp::two_hop_mark_kernel<<<static_cast<unsigned>(blocks), plnlp::kHeurThreads, 0,
                                 static_cast<cudaStream_t>(stream)>>>(rowptr, col, rrowptr, rcol, nodes, item_ptr, Qc,
                                                                      col0, W, cand, bitmap, words);
    PLNLP_LAUNCH_CHECK();
    return 0;
}

// s [Qc, W] (row stride lds), zeroed by the caller: for every set bit c of row qi of the bitmap of
// plnlp_two_hop_mark, s[qi, c] = the sum of plnlp_link_heuristic_f64 for the pair (nodes[qi], column c's node),
// rounded to fp32 once (_f32) or kept in fp64 (_f64).  Same table, weight and column forms as above.
extern "C" int plnlp_two_hop_score_f32(const int64_t* rowptr, const int32_t* col, int64_t n, int64_t nnz,
                                       const double* weight, const int64_t* nodes, int64_t Qc, int64_t col0,
                                       int64_t W, const int64_t* cand, const uint32_t* bitmap, float* s, int64_t lds,
                                       void* stream) {
    PLNLP_REQUIRE(cand == nullptr || col0 == 0, PLNLP_E_UNSUPPORTED);
    return plnlp::two_hop_score<float>(rowptr, col, n, nnz, weight, nodes, Qc, col0, W, cand, bitmap, s, lds, stream);
}

extern "C" int plnlp_two_hop_score_f64(const int64_t* rowptr, const int32_t* col, int64_t n, int64_t nnz,
                                       const double* weight, const int64_t* nodes, int64_t Qc, int64_t col0,
                                       int64_t W, const int64_t* cand, const uint32_t* bitmap, double* s,
                                       int64_t lds, void* stream) {
    PLNLP_REQUIRE(cand == nullptr || col0 == 0, PLNLP_E_UNSUPPORTED);
    return plnlp::two_hop_score<double>(rowptr, col, n, nnz, weight, nodes, Qc, col0, W, cand, bitmap, s, lds,
                                        stream);
}
