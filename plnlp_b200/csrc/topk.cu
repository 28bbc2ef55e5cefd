// Link recommendation over all nodes: known-link masking, per-row top-k selection and filtered rank counts on
// dense score chunks S [Q, N] (one row per query node, one column per candidate node).
//
// Selection works on a 64-bit composite key per entry: the order-preserving float key (float_key, -0 folded
// into +0) in the high word and ~column in the low word.  Larger composite key = higher score, and among equal
// scores the lower column.  Every key of a row is distinct, so "the k largest keys" is exactly the top-k under
// the tie rule (score descending, then column ascending) and every selection below is order independent.
//
// A chunk may cover the candidate columns [col0, col0 + N) of a wider id space (one shard of a row-partitioned
// graph): keys, ids and the target comparison then use the global column col0 + j, so per-shard results merge
// into exactly the selection over the whole row (topk_cross_merge_kernel).
//
// A chunk may instead hold an arbitrary candidate set: column j is the node cand[j], cand strictly ascending.  Keys
// stay on the column, which orders exactly as the ids do; the mask and the target comparison find a node's column by
// binary search in cand, and the write tail reports cand[j].
//
// Two kernels, ONE pass over the score chunk:
//   topk_segment_kernel  one CTA per (row, segment of kSeg columns).  Streams its segment once, counts gt / ge
//                        against the target score, and keeps a candidate buffer in shared memory: an entry is
//                        admitted when its key beats the buffer's threshold; when the buffer runs full it is cut
//                        back to its k best (block radix select) and the threshold rises to the k-th key.  The
//                        segment's k best keys and its two counts go to the workspace.
//   topk_merge_kernel    one CTA per row: sums the counts, selects the k best of the segments' candidates (at most
//                        ceil(N / kSeg) * k keys, L2 resident), sorts them (bitonic, shared memory) and writes ids
//                        and scores.
// plus topk_cross_merge_kernel: one CTA per row, the k best of R per-shard sorted lists (ids, scores), with the
// select / sort / write tail of topk_merge_kernel.
// Integer outputs are exact; ids / scores do not depend on the launch configuration.
#include <cfloat>

#include "common.cuh"

namespace plnlp {
namespace {

constexpr int kThreads = 256;
constexpr int kUnroll = 8;                         // scores per thread per tile
constexpr int kTile = kThreads * kUnroll;          // 2048 scores per tile
constexpr int kMaxK = 1024;
constexpr int kCap = 4096;                         // candidate buffer: room for k + one full tile
constexpr int64_t kSeg = 65536;                    // columns per segment CTA
static_assert(kCap >= kMaxK + kTile, "a tile must fit behind k kept candidates");

__device__ __forceinline__ bool finite_score(float v) { return fabsf(v) <= FLT_MAX; }

// the column of node id among the strictly ascending cand[c0 .. c1), or -1
__device__ __forceinline__ int64_t cand_column(const int64_t* __restrict__ cand, int64_t c0, int64_t c1, int64_t id) {
    int64_t lo = c0, hi = c1;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (__ldg(cand + mid) < id) lo = mid + 1; else hi = mid;
    }
    return lo < c1 && __ldg(cand + lo) == id ? lo : -1;
}

__device__ __forceinline__ uint64_t cand_key(float v, uint32_t col) {
    const float c = v == 0.0f ? 0.0f : v;          // -0 ties with +0
    return (static_cast<uint64_t>(float_key(c)) << 32) | static_cast<uint32_t>(~col);
}

struct SelectShared {
    unsigned hist[256];
    uint64_t prefix;
    uint64_t min_key;
    int k_rem;
    int done;
};

// kk-th largest (1-based, kk <= n) of the distinct keys get(0..n), returned to every thread.  MSB-first 8-bit radix
// passes as csrc/rank.cu; once the chosen digit's bucket holds exactly the k_rem keys still wanted, the answer is the
// smallest key of that bucket and one min-sweep ends the search.  Needs kThreads threads; begins and ends in sync.
template <class Get>
__device__ uint64_t block_select(Get get, int n, int kk, SelectShared& sh) {
    const int tid = threadIdx.x;
    if (tid == 0) { sh.prefix = 0; sh.k_rem = kk; sh.done = 0; sh.min_key = ~0ull; }
    for (int pass = 0; pass < 8; ++pass) {
        const int shift = 56 - 8 * pass;
        const uint64_t himask = pass == 0 ? 0ull : (~0ull << (shift + 8));
        sh.hist[tid] = 0;
        __syncthreads();
        const uint64_t prefix = sh.prefix;
        for (int i = tid; i < n; i += kThreads) {
            const uint64_t key = get(i);
            if ((key & himask) == prefix) atomicAdd(&sh.hist[(key >> shift) & 255u], 1u);
        }
        __syncthreads();
        if (tid < 32) {
            // lane l owns bins 255 - 8l ... 248 - 8l (descending)
            unsigned c = 0;
#pragma unroll
            for (int j = 0; j < 8; ++j) c += sh.hist[255 - 8 * tid - j];
            unsigned incl = c;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned t = __shfl_up_sync(0xffffffffu, incl, o);
                if (tid >= o) incl += t;
            }
            const unsigned before = incl - c;
            const unsigned krem = static_cast<unsigned>(sh.k_rem);
            if (before < krem && krem <= incl) {
                unsigned cum = before;
                for (int j = 0; j < 8; ++j) {
                    const int b = 255 - 8 * tid - j;
                    const unsigned hb = sh.hist[b];
                    if (cum + hb >= krem) {
                        sh.prefix = prefix | (static_cast<uint64_t>(b) << shift);
                        sh.k_rem = static_cast<int>(krem - cum);
                        sh.done = (hb == krem - cum) ? 1 : 0;
                        break;
                    }
                    cum += hb;
                }
            }
        }
        __syncthreads();
        if (sh.done) {
            const uint64_t pmask = ~0ull << shift, p = sh.prefix;
            uint64_t m = ~0ull;
            for (int i = tid; i < n; i += kThreads) {
                const uint64_t key = get(i);
                if ((key & pmask) == p && key < m) m = key;
            }
            atomicMin(reinterpret_cast<unsigned long long*>(&sh.min_key), static_cast<unsigned long long>(m));
            __syncthreads();
            const uint64_t r = sh.min_key;
            __syncthreads();
            return r;
        }
    }
    const uint64_t r = sh.prefix;
    __syncthreads();
    return r;
}

struct SegShared {
    uint64_t buf[kCap];
    SelectShared sel;
    uint64_t thr;
    int cnt;
    int cnt2;
    int red[2][kThreads / 32];
};

// cut the buffer back to its k best keys (precondition: cnt > k); the threshold becomes the k-th key
__device__ void cut_to_k(SegShared& sh, int k) {
    const int n = sh.cnt;
    const uint64_t* buf = sh.buf;
    const uint64_t kth = block_select([buf](int i) { return buf[i]; }, n, k, sh.sel);
    constexpr int kPer = kCap / kThreads;
    uint64_t mine[kPer];
#pragma unroll
    for (int i = 0; i < kPer; ++i) {
        const int idx = i * kThreads + threadIdx.x;
        mine[i] = idx < n ? sh.buf[idx] : 0ull;
    }
    if (threadIdx.x == 0) sh.cnt2 = 0;
    __syncthreads();
#pragma unroll
    for (int i = 0; i < kPer; ++i)
        if (mine[i] >= kth && mine[i] != 0ull) sh.buf[atomicAdd(&sh.cnt2, 1)] = mine[i];
    __syncthreads();
    if (threadIdx.x == 0) { sh.cnt = k; sh.thr = kth; }
    __syncthreads();
}

// grid.x = Q * n_seg; CTA b handles row b / n_seg, global columns [col0 + seg * kSeg, min(col_end, ... + kSeg)).
// s_shifted = s - col0 (formed as an address by the host), so the loop runs on global columns: the column offset
// costs no register (the kernel stays at 62 registers, 4 CTAs per SM).  kIdCols (then col0 = 0): column j is the
// node col_id[j], and the target's column is looked up once, before the loop, within this CTA's segment -- a
// separate instantiation, so the lookup leaves the plain kernel's code and register allocation as they were.
template <bool kIdCols>
__global__ void __launch_bounds__(kThreads, 4) topk_segment_kernel(
    const float* __restrict__ s_shifted, int64_t lds, int64_t col0, int64_t col_end, int k, int n_seg,
    const int64_t* __restrict__ target, const float* __restrict__ target_score, const int64_t* __restrict__ col_id,
    uint64_t* __restrict__ cand, int* __restrict__ cand_n, int* __restrict__ part_gt, int* __restrict__ part_ge) {
    __shared__ SegShared sh;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t b = blockIdx.x;
    const int64_t q = b / n_seg;
    const int64_t c0 = col0 + (b % n_seg) * kSeg, c1 = min(col_end, c0 + kSeg);
    const float* row = s_shifted + q * lds;
    const bool rank = target != nullptr;
    int64_t tcol = rank ? target[q] : -1;
    if constexpr (kIdCols) tcol = rank ? cand_column(col_id, c0, c1, tcol) : -1;
    const float tval = rank ? target_score[q] : 0.0f;
    int cgt = 0, cge = 0;
    if (tid == 0) { sh.cnt = 0; sh.thr = 0ull; }   // every finite entry has a key > 0
    __syncthreads();
    for (int64_t base = c0; base < c1; base += kTile) {
        float v[kUnroll];
#pragma unroll
        for (int u = 0; u < kUnroll; ++u) {
            const int64_t j = base + u * kThreads + tid;
            v[u] = j < c1 ? __ldcs(row + j) : __int_as_float(0x7fc00000);
        }
        const uint64_t thr = sh.thr;
#pragma unroll
        for (int u = 0; u < kUnroll; ++u) {
            const int64_t j = base + u * kThreads + tid;
            const bool fin = finite_score(v[u]);
            if (rank && fin && j != tcol) {
                cgt += v[u] > tval;
                cge += v[u] >= tval;
            }
            if (k > 0) {
                const uint64_t key = fin ? cand_key(v[u], static_cast<uint32_t>(j)) : 0ull;
                const bool take = key > thr;
                const unsigned m = __ballot_sync(0xffffffffu, take);
                if (m) {
                    const int leader = __ffs(m) - 1;
                    int pos = 0;
                    if (lane == leader) pos = atomicAdd(&sh.cnt, __popc(m));
                    pos = __shfl_sync(0xffffffffu, pos, leader);
                    if (take) sh.buf[pos + __popc(m & ((1u << lane) - 1u))] = key;
                }
            }
        }
        __syncthreads();
        const int cnt = sh.cnt;
        __syncthreads();                   // every thread has read cnt before the next tile appends
        if (k > 0 && cnt > kCap - kTile) cut_to_k(sh, k);
    }
    if (k > 0) {
        if (sh.cnt > k) cut_to_k(sh, k);
        const int n = sh.cnt;
        for (int i = tid; i < n; i += kThreads) cand[b * k + i] = sh.buf[i];
        if (tid == 0) cand_n[b] = n;
    }
    if (rank) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            cgt += __shfl_xor_sync(0xffffffffu, cgt, o);
            cge += __shfl_xor_sync(0xffffffffu, cge, o);
        }
        if (lane == 0) { sh.red[0][warp] = cgt; sh.red[1][warp] = cge; }
        __syncthreads();
        if (tid == 0) {
            int a = 0, c = 0;
            for (int w = 0; w < kThreads / 32; ++w) { a += sh.red[0][w]; c += sh.red[1][w]; }
            part_gt[b] = a;
            part_ge[b] = c;
        }
    }
}

struct MergeShared {
    uint64_t buf[kMaxK];
    SelectShared sel;
    int total;
    int cnt;
};

// the tail of both merges, run by one CTA for one row: the k best of the keys get(0 .. slots) -- ``total`` of them
// live, dead slots read as key 0, below every live key -- sorted descending (bitonic, shared memory) and written as
// (id, score), the tail (-1, -inf); id = col_id[column] when col_id != NULL.  Begins in sync.
template <class Get>
__device__ void select_sort_write(Get get, int slots, int total, int k, const int64_t* __restrict__ col_id,
                                  int64_t* __restrict__ ids, float* __restrict__ scores, MergeShared& sh) {
    const int tid = threadIdx.x;
    const int m = min(total, k);
    const uint64_t kth = total > k ? block_select(get, slots, k, sh.sel) : 1ull;
    for (int i = tid; i < slots; i += kThreads) {
        const uint64_t key = get(i);
        if (key >= kth && key != 0ull) sh.buf[atomicAdd(&sh.cnt, 1)] = key;
    }
    int len = 1;
    while (len < m) len <<= 1;
    for (int i = m + tid; i < len; i += kThreads) sh.buf[i] = 0ull;
    __syncthreads();
    // bitonic sort, descending
    for (int size = 2; size <= len; size <<= 1) {
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int i = tid; i < len / 2; i += kThreads) {
                const int lo = 2 * i - (i & (stride - 1));
                const int hi = lo + stride;
                const bool desc = (lo & size) == 0;
                const uint64_t a = sh.buf[lo], c = sh.buf[hi];
                if ((a < c) == desc) { sh.buf[lo] = c; sh.buf[hi] = a; }
            }
            __syncthreads();
        }
    }
    for (int i = tid; i < k; i += kThreads) {
        if (i < m) {
            const uint64_t key = sh.buf[i];
            const uint32_t c = ~static_cast<uint32_t>(key);
            ids[i] = col_id != nullptr ? __ldg(col_id + c) : static_cast<int64_t>(c);
            scores[i] = key_float(static_cast<uint32_t>(key >> 32));
        } else {
            ids[i] = -1;
            scores[i] = -INFINITY;
        }
    }
}

// one CTA per row: gt / ge sums, then the k best of the n_seg * k candidate slots (slot i of segment g is live when
// i < cand_n[g]), sorted, written as (id, score); the id of column j is col_id[j] when col_id != NULL
__global__ void __launch_bounds__(kThreads) topk_merge_kernel(
    const uint64_t* __restrict__ cand, const int* __restrict__ cand_n, const int* __restrict__ part_gt,
    const int* __restrict__ part_ge, int n_seg, int k, const int64_t* __restrict__ col_id, int64_t* __restrict__ ids,
    float* __restrict__ scores, int32_t* __restrict__ gt, int32_t* __restrict__ ge) {
    __shared__ MergeShared sh;
    const int tid = threadIdx.x;
    const int64_t q = blockIdx.x;
    const int64_t g0 = q * n_seg;
    if (gt != nullptr && tid == 0) {
        int a = 0, c = 0;
        for (int g = 0; g < n_seg; ++g) { a += part_gt[g0 + g]; c += part_ge[g0 + g]; }
        gt[q] = a;
        ge[q] = c;
    }
    if (k == 0) return;
    if (tid == 0) {
        int t = 0;
        for (int g = 0; g < n_seg; ++g) t += cand_n[g0 + g];
        sh.total = t;
        sh.cnt = 0;
    }
    __syncthreads();
    const uint64_t* rc = cand + g0 * k;
    const int* rn = cand_n + g0;
    auto get = [rc, rn, k](int i) -> uint64_t { return (i % k) < __ldg(rn + i / k) ? __ldg(rc + i) : 0ull; };
    select_sort_write(get, n_seg * k, sh.total, k, col_id, ids + q * k, scores + q * k, sh);
}

// one CTA per row q: the k best of the R sorted lists ids_in / scores_in [R, Q, k_in] (rank-major, as an all-gather
// of the per-shard [Q, k_in] results lays them out).  The keys are rebuilt from (score, global id), so the result is
// the selection over the union of the lists whatever the split; an entry with id < 0 or a non-finite score is dead.
__global__ void __launch_bounds__(kThreads) topk_cross_merge_kernel(
    const int64_t* __restrict__ ids_in, const float* __restrict__ scores_in, int R, int64_t Q, int k_in, int k,
    int64_t* __restrict__ ids, float* __restrict__ scores) {
    __shared__ MergeShared sh;
    const int tid = threadIdx.x;
    const int64_t q = blockIdx.x;
    auto get = [ids_in, scores_in, Q, k_in, q](int i) -> uint64_t {
        const int64_t at = (static_cast<int64_t>(i / k_in) * Q + q) * k_in + i % k_in;
        const int64_t id = __ldg(ids_in + at);
        const float v = __ldg(scores_in + at);
        return id >= 0 && finite_score(v) ? cand_key(v, static_cast<uint32_t>(id)) : 0ull;
    };
    const int slots = R * k_in;
    if (tid == 0) { sh.total = 0; sh.cnt = 0; }
    __syncthreads();
    int live = 0;
    for (int i = tid; i < slots; i += kThreads) live += get(i) != 0ull;
    if (live) atomicAdd(&sh.total, live);
    __syncthreads();
    select_sort_write(get, slots, sh.total, k, nullptr, ids + q * k, scores + q * k, sh);
}

// row q covers the global columns [col0, col0 + N): a known link c sits at column c - col0; or, with cand (col0 = 0),
// the nodes cand[0 .. N): c sits at its position in cand, if any
__global__ void __launch_bounds__(128) score_mask_kernel(float* __restrict__ s, int64_t lds, int64_t N, int64_t col0,
                                                         const int64_t* __restrict__ cand,
                                                         const int64_t* __restrict__ node,
                                                         const int64_t* __restrict__ rowptr,
                                                         const int32_t* __restrict__ col, int exclude_self) {
    const int64_t q = blockIdx.x;
    const int64_t n = node[q];
    float* row = s + q * lds;
    if (rowptr != nullptr) {
        const int64_t e1 = rowptr[n + 1];
        for (int64_t e = rowptr[n] + threadIdx.x; e < e1; e += blockDim.x) {
            const int64_t c = cand != nullptr ? cand_column(cand, 0, N, col[e]) : col[e] - col0;
            if (c >= 0 && c < N) row[c] = -INFINITY;
        }
    }
    const int64_t self = cand != nullptr ? (exclude_self ? cand_column(cand, 0, N, n) : -1) : n - col0;
    if (exclude_self && threadIdx.x == 0 && self >= 0 && self < N) row[self] = -INFINITY;
}

int64_t n_segments(int64_t N) { return ceil_div(N, kSeg); }

int64_t align16(int64_t b) { return (b + 15) / 16 * 16; }

}  // namespace
}  // namespace plnlp

using namespace plnlp;

namespace {

int score_mask(float* s, int64_t lds, int64_t Q, int64_t N, int64_t col0, const int64_t* cand, const int64_t* node,
               const int64_t* rowptr, const int32_t* col, int exclude_self, void* stream) {
    PLNLP_REQUIRE(Q >= 0 && N >= 1 && lds >= N && col0 >= 0 && col0 + N < (int64_t{1} << 31), PLNLP_E_SIZE);
    if (Q == 0) return 0;
    PLNLP_REQUIRE(s && node && (rowptr == nullptr) == (col == nullptr), PLNLP_E_NULL);
    score_mask_kernel<<<static_cast<unsigned>(Q), 128, 0, static_cast<cudaStream_t>(stream)>>>(
        s, lds, N, col0, cand, node, rowptr, col, exclude_self);
    PLNLP_LAUNCH_CHECK();
    return 0;
}

}  // namespace

extern "C" int plnlp_score_mask_cols_f32(float* s, int64_t lds, int64_t Q, int64_t N, int64_t col0,
                                         const int64_t* node, const int64_t* rowptr, const int32_t* col,
                                         int exclude_self, void* stream) {
    return score_mask(s, lds, Q, N, col0, nullptr, node, rowptr, col, exclude_self, stream);
}

extern "C" int plnlp_score_mask_cand_f32(float* s, int64_t lds, int64_t Q, int64_t C, const int64_t* cand,
                                         const int64_t* node, const int64_t* rowptr, const int32_t* col,
                                         int exclude_self, void* stream) {
    PLNLP_REQUIRE(Q == 0 || cand, PLNLP_E_NULL);
    return score_mask(s, lds, Q, C, 0, cand, node, rowptr, col, exclude_self, stream);
}

extern "C" int plnlp_score_mask_f32(float* s, int64_t lds, int64_t Q, int64_t N, const int64_t* node,
                                    const int64_t* rowptr, const int32_t* col, int exclude_self, void* stream) {
    return plnlp_score_mask_cols_f32(s, lds, Q, N, 0, node, rowptr, col, exclude_self, stream);
}

extern "C" int64_t plnlp_topk_rows_workspace_bytes(int64_t Q, int64_t N, int64_t k) {
    if (Q < 0 || N < 1 || k < 0) return 0;
    const int64_t slots = Q * n_segments(N);
    return align16(slots * k * 8) + 3 * align16(slots * 4);
}

extern "C" int plnlp_topk_rows_cand_f32(const float* s, int64_t lds, int64_t Q, int64_t N, int64_t col0, int64_t k,
                                        const int64_t* target, const float* target_score, int64_t* ids,
                                        float* scores, int32_t* gt, int32_t* ge, void* workspace,
                                        int64_t workspace_bytes, const int64_t* cand, void* stream) {
    PLNLP_REQUIRE(Q >= 0 && N >= 1 && lds >= N && k >= 0 && col0 >= 0 && col0 + N < (int64_t{1} << 31),
                  PLNLP_E_SIZE);
    PLNLP_REQUIRE(k <= kMaxK && (cand == nullptr || col0 == 0), PLNLP_E_UNSUPPORTED);
    PLNLP_REQUIRE(k > 0 || target != nullptr, PLNLP_E_SIZE);             // nothing to compute
    if (Q == 0) return 0;
    PLNLP_REQUIRE(s && workspace, PLNLP_E_NULL);
    if (k > 0) PLNLP_REQUIRE(ids && scores, PLNLP_E_NULL);
    if (target != nullptr) PLNLP_REQUIRE(target_score && gt && ge, PLNLP_E_NULL);
    PLNLP_REQUIRE(workspace_bytes >= plnlp_topk_rows_workspace_bytes(Q, N, k), PLNLP_E_WORKSPACE);
    PLNLP_REQUIRE(aligned(workspace, 16), PLNLP_E_ALIGN);
    const int64_t n_seg = n_segments(N);
    const int64_t slots = Q * n_seg;
    PLNLP_REQUIRE(slots < (int64_t{1} << 31), PLNLP_E_SIZE);
    char* w = static_cast<char*>(workspace);
    uint64_t* keys = reinterpret_cast<uint64_t*>(w);
    int* cand_n = reinterpret_cast<int*>(w + align16(slots * k * 8));
    int* part_gt = cand_n + align16(slots * 4) / 4;
    int* part_ge = part_gt + align16(slots * 4) / 4;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const float* s_shifted = reinterpret_cast<const float*>(reinterpret_cast<uintptr_t>(s) - 4 * col0);
    auto segment = cand != nullptr ? topk_segment_kernel<true> : topk_segment_kernel<false>;
    segment<<<static_cast<unsigned>(slots), kThreads, 0, st>>>(
        s_shifted, lds, col0, col0 + N, static_cast<int>(k), static_cast<int>(n_seg), target, target_score, cand,
        keys, cand_n, part_gt, part_ge);
    PLNLP_LAUNCH_CHECK();
    topk_merge_kernel<<<static_cast<unsigned>(Q), kThreads, 0, st>>>(
        keys, cand_n, part_gt, part_ge, static_cast<int>(n_seg), static_cast<int>(k), cand, ids, scores, gt, ge);
    PLNLP_LAUNCH_CHECK();
    return 0;
}

extern "C" int plnlp_topk_rows_cols_f32(const float* s, int64_t lds, int64_t Q, int64_t N, int64_t col0, int64_t k,
                                        const int64_t* target, const float* target_score, int64_t* ids,
                                        float* scores, int32_t* gt, int32_t* ge, void* workspace,
                                        int64_t workspace_bytes, void* stream) {
    return plnlp_topk_rows_cand_f32(s, lds, Q, N, col0, k, target, target_score, ids, scores, gt, ge, workspace,
                                    workspace_bytes, nullptr, stream);
}

extern "C" int plnlp_topk_rows_f32(const float* s, int64_t lds, int64_t Q, int64_t N, int64_t k,
                                   const int64_t* target, const float* target_score, int64_t* ids, float* scores,
                                   int32_t* gt, int32_t* ge, void* workspace, int64_t workspace_bytes,
                                   void* stream) {
    return plnlp_topk_rows_cols_f32(s, lds, Q, N, 0, k, target, target_score, ids, scores, gt, ge, workspace,
                                    workspace_bytes, stream);
}

extern "C" int plnlp_topk_merge_f32(const int64_t* ids_in, const float* scores_in, int64_t R, int64_t Q,
                                    int64_t k_in, int64_t k, int64_t* ids, float* scores, void* stream) {
    PLNLP_REQUIRE(R >= 1 && Q >= 0 && k_in >= 1 && k >= 1 && R * k_in < (int64_t{1} << 31), PLNLP_E_SIZE);
    PLNLP_REQUIRE(k <= kMaxK, PLNLP_E_UNSUPPORTED);
    if (Q == 0) return 0;
    PLNLP_REQUIRE(ids_in && scores_in && ids && scores, PLNLP_E_NULL);
    topk_cross_merge_kernel<<<static_cast<unsigned>(Q), kThreads, 0, static_cast<cudaStream_t>(stream)>>>(
        ids_in, scores_in, static_cast<int>(R), Q, static_cast<int>(k_in), static_cast<int>(k), ids, scores);
    PLNLP_LAUNCH_CHECK();
    return 0;
}
