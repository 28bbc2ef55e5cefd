// One hop of the path-based link scores (plnlp_b200/paths.py: Katz and Personalized PageRank) for a block of B
// source columns.  The state x [n, B] is fp32 and node-major (row stride ldx); for every output row j of
// [r0, r0 + rows)
//
//   y[j - r0, c] = fp32( cm * s + (src[c] == j ? ba : 0) ),   s = sum over w in R(j) of wt(w) * x[w, c]
//
// with wt(w) = weight[w] (fp64), or 1 when weight == NULL.  Products, sums, the multiply and the add are fp64, rounded
// to nearest with no contraction (__dmul_rn / __dadd_rn), and each output is rounded to fp32 once.
//
// Order: the entries of R(j) (ascending w) are cut into the work items of an SpMM plan (graph.build_plan with the
// fixed chunk paths.PROP_CHUNK).  One warp sums an item's entries in order, starting from +0; a one-item row is
// finished by that warp, and the partials of a split (hub) row are added in item order by a second, fixed-order pass.
// Every sum depends on the plan and the inputs only: the same on every run and for every B.
//
// Columns: B = 32 V, V in {1, 2, 4, 8}; lane l owns the columns [l V, l V + V) and keeps their fp64 sums in registers.
//
// Live map: live_in[w] == 0 promises x[w, :] == 0.  Every x and every wt is >= 0, so such a row would add +0 to a sum
// that is >= +0 and change no bit: it is not gathered.  The lanes test 32 entries at once and the warp walks only the
// live ones, up to four rows in flight.  live_out[j - r0] = 1 when any output of row j is non-zero, else 0.
#include <cstring>

#include "common.cuh"

namespace plnlp {
namespace {

constexpr int kPropThreads = 256;
constexpr int kPropInFlight = 4;

struct PropParams {
    const int32_t* item_ptr;    // [n_items + 1]: item t covers entries [item_ptr[t], item_ptr[t + 1])
    const int32_t* item_row;    // local output row of item t
    const int32_t* item_slot;   // partial slot of item t, -1 for a one-item row
    int64_t n_items;
    const int32_t* col;         // node ids w of the entries
    const int32_t* fix_ptr;     // split row f: slots [fix_ptr[f], fix_ptr[f + 1])
    const int32_t* fix_row;
    int64_t n_fix;
    double* partial;            // [n_partial, B]
    const double* weight;       // [n] or NULL
    const float* x;
    int64_t ldx;
    const int64_t* src;         // [B], -1 for a padding column
    int64_t B;
    double cm, ba;
    const uint8_t* live_in;     // [n] or NULL
    uint8_t* live_out;          // [rows] or NULL
    int64_t r0;
    float* y;
    int64_t ldy;
};

template <int V>
__device__ __forceinline__ void finish_row(const PropParams& p, int64_t row, const double (&s)[V], int lane) {
    const int64_t j = p.r0 + row;
    float out[V];
    bool nz = false;
#pragma unroll
    for (int i = 0; i < V; ++i) {
        const double add = __ldg(p.src + lane * V + i) == j ? p.ba : 0.0;
        out[i] = __double2float_rn(__dadd_rn(__dmul_rn(p.cm, s[i]), add));
        nz |= out[i] != 0.0f;
    }
    store_vec<V>(p.y + row * p.ldy + lane * V, out);
    const unsigned any = __ballot_sync(0xffffffffu, nz);
    if (lane == 0 && p.live_out) p.live_out[row] = any ? 1 : 0;
}

template <int V>
__global__ void __launch_bounds__(kPropThreads, V >= 8 ? 2 : 3) propagate_kernel(const PropParams p) {
    const int lane = threadIdx.x & 31;
    const int64_t item = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    if (item >= p.n_items) return;                  // whole warps
    const int32_t beg = __ldg(p.item_ptr + item), end = __ldg(p.item_ptr + item + 1);
    const float* xl = p.x + lane * V;
    double acc[V];
#pragma unroll
    for (int i = 0; i < V; ++i) acc[i] = 0.0;
    for (int32_t base = beg; base < end; base += 32) {
        const int32_t e = base + lane;
        int32_t w = 0;
        bool live = false;
        double wt = 1.0;
        if (e < end) {
            w = __ldg(p.col + e);
            live = p.live_in == nullptr || __ldg(p.live_in + w) != 0;
            if (p.weight) wt = __ldg(p.weight + w);
        }
        unsigned m = __ballot_sync(0xffffffffu, live);
        while (m) {                                 // the live entries in ascending order, kPropInFlight at a time
            int from[kPropInFlight];
            bool ok[kPropInFlight];
#pragma unroll
            for (int k = 0; k < kPropInFlight; ++k) {
                ok[k] = m != 0u;
                from[k] = ok[k] ? __ffs(static_cast<int>(m)) - 1 : 0;
                m &= m - 1u;
            }
            float xv[kPropInFlight][V];
            double wk[kPropInFlight];
#pragma unroll
            for (int k = 0; k < kPropInFlight; ++k) {
                const int32_t wr = __shfl_sync(0xffffffffu, w, from[k]);
                wk[k] = __shfl_sync(0xffffffffu, wt, from[k]);
                if (ok[k]) {
                    load_vec<V>(xv[k], xl + static_cast<int64_t>(wr) * p.ldx);
                } else {
#pragma unroll
                    for (int i = 0; i < V; ++i) xv[k][i] = 0.0f;
                }
            }
#pragma unroll
            for (int k = 0; k < kPropInFlight; ++k) {
                if (!ok[k]) continue;
#pragma unroll
                for (int i = 0; i < V; ++i) {
                    const double t = static_cast<double>(xv[k][i]);
                    acc[i] = __dadd_rn(acc[i], p.weight ? __dmul_rn(wk[k], t) : t);
                }
            }
        }
    }
    const int32_t slot = __ldg(p.item_slot + item);
    if (slot >= 0) {
        double* dst = p.partial + static_cast<int64_t>(slot) * p.B + lane * V;
#pragma unroll
        for (int i = 0; i < V; ++i) dst[i] = acc[i];
        return;
    }
    finish_row<V>(p, __ldg(p.item_row + item), acc, lane);
}

// split rows: one warp adds the row's partial slots in slot (= item) order, then the epilogue
template <int V>
__global__ void __launch_bounds__(kPropThreads) propagate_fix_kernel(const PropParams p) {
    const int lane = threadIdx.x & 31;
    const int64_t f = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    if (f >= p.n_fix) return;
    const int32_t s0 = __ldg(p.fix_ptr + f), s1 = __ldg(p.fix_ptr + f + 1);
    double s[V];
#pragma unroll
    for (int i = 0; i < V; ++i) s[i] = 0.0;
    for (int32_t t = s0; t < s1; ++t) {
        const double* src = p.partial + static_cast<int64_t>(t) * p.B + lane * V;
#pragma unroll
        for (int i = 0; i < V; ++i) s[i] = __dadd_rn(s[i], src[i]);
    }
    finish_row<V>(p, __ldg(p.fix_row + f), s, lane);
}

template <int V>
int launch(const PropParams& p, cudaStream_t st) {
    const int64_t warps = kPropThreads / 32;
    propagate_kernel<V><<<static_cast<unsigned>(ceil_div(p.n_items, warps)), kPropThreads, 0, st>>>(p);
    PLNLP_LAUNCH_CHECK();
    if (p.n_fix > 0) {
        propagate_fix_kernel<V><<<static_cast<unsigned>(ceil_div(p.n_fix, warps)), kPropThreads, 0, st>>>(p);
        PLNLP_LAUNCH_CHECK();
    }
    return 0;
}

}  // namespace
}  // namespace plnlp

extern "C" int plnlp_propagate_f32(const int32_t* item_ptr, const int32_t* item_row, const int32_t* item_slot,
                                   int64_t n_items, const int32_t* col, const int32_t* fix_ptr,
                                   const int32_t* fix_row, int64_t n_fix, double* partial, const double* weight,
                                   const float* x, int64_t ldx, const int64_t* src, int64_t B, uint64_t c_bits,
                                   uint64_t b_bits, const uint8_t* live_in, uint8_t* live_out, int64_t r0,
                                   int64_t rows, float* y, int64_t ldy, void* stream) {
    PLNLP_REQUIRE(n_items >= 0 && n_fix >= 0 && r0 >= 0 && rows >= 0, PLNLP_E_SIZE);
    PLNLP_REQUIRE(B == 32 || B == 64 || B == 128 || B == 256, PLNLP_E_SIZE);
    PLNLP_REQUIRE(ldx >= B && ldy >= B && n_items >= rows && n_items < (int64_t(1) << 36), PLNLP_E_SIZE);
    if (n_items == 0) return 0;
    PLNLP_REQUIRE(item_ptr && item_row && item_slot && col && x && src && y, PLNLP_E_NULL);
    if (n_fix > 0) PLNLP_REQUIRE(fix_ptr && fix_row && partial, PLNLP_E_NULL);
    const int V = static_cast<int>(B / 32);
    const int vec = V < 4 ? V : 4;                 // float elements per vector access
    PLNLP_REQUIRE(ldx % vec == 0 && ldy % vec == 0 && plnlp::aligned(x, 4 * vec) && plnlp::aligned(y, 4 * vec) &&
                      (partial == nullptr || plnlp::aligned(partial, 8)),
                  PLNLP_E_ALIGN);
    plnlp::PropParams p{item_ptr, item_row, item_slot, n_items, col, fix_ptr, fix_row, n_fix, partial, weight, x, ldx,
                        src, B, 0.0, 0.0, live_in, live_out, r0, y, ldy};
    std::memcpy(&p.cm, &c_bits, sizeof(double));   // the ABI passes the fp64 coefficients as their bit patterns
    std::memcpy(&p.ba, &b_bits, sizeof(double));
    auto st = static_cast<cudaStream_t>(stream);
    switch (V) {
        case 1: return plnlp::launch<1>(p, st);
        case 2: return plnlp::launch<2>(p, st);
        case 4: return plnlp::launch<4>(p, st);
        default: return plnlp::launch<8>(p, st);
    }
}
