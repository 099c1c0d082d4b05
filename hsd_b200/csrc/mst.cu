// Minimum spanning tree of the complete graph under the structural distance, by Borůvka rounds over row
// panels (engine.degree_mst), so the N x N matrix never has to exist.  Edges are ordered by
// E(u, v) = (float(D[u][v]), min(u, v), max(u, v)), a total order: the MST is unique.  For a fixed node i
// that order on its edges is the order of (D[i][j], j), so node i's best edge leaving its component is the
// minimum of the int64 key K(d, j) = float_bits(d) << 32 | j.  Distances are finite and >= 0: the bits are
// below 2^31 and the signed compare orders the keys; INT64_MAX means "no edge".  A minimum does not depend
// on the order of its updates, so the 64-bit atomicMin below gives the same keys whatever the schedule.
//
//   mst_panel_min        a panel of the k-NN sweep (block row r is node node0 + r, column c is node node0 + c;
//                        the upper part c > r holds every pair the panel owns once).  A CTA owns 32 rows x 256
//                        columns: thread t holds column c0 + t, reads the tile's rows in order (each row read is
//                        1 KB of consecutive floats) and keeps the column's minimum in registers; a row's
//                        minimum is two warp reductions (distance bits, then the smallest column among the
//                        matches) staged in shared memory across the 8 warps.  One atomicMin per (row, tile)
//                        and per (column, tile).  The lower part and the ld padding are never read.
//   mst_list_candidates  one warp per node: the first entry of its k-NN list outside its component is its exact
//                        best edge (the lists are ordered by (distance, id), the order of K); a node whose full
//                        list lies inside its component is exhausted, and every edge it has outside is at least
//                        as long as its k-th entry, which becomes its bound.
//
// Mutual reachability (engine.degree_mreach_mst, HDBSCAN): the distance is d_mr(a, b) = max(core[a], core[b],
// D[a][b]) with core[i] >= 0 finite, so d_mr is one of its three float32 operands and, all of them being >= 0,
// their maximum is the maximum of their bits.  The order is E on d_mr and the keys are K(d_mr, j).
//
//   mst_panel_min<true>  the panel kernel above with the compared value max(blk[r][c], core[a], core[b]): the
//                        32 row cores sit in shared memory beside row_comp, the column's core in a register;
//                        the panel is still read once.
//   mst_list_candidates_mreach  one warp per node.  The lists are ordered by D, not by d_mr, so the first entry
//                        outside the component is no longer the best: the key is the minimum of
//                        K(max(core_i, core_j, val), j) over all the list's entries j outside i's component.
//                        It is exact when the list is short (it holds every other node) or when its distance is
//                        strictly below val[i][k-1]: an unlisted j has D[i][j] >= val[i][k-1], hence
//                        d_mr(i, j) >= val[i][k-1], longer than the key.  Exact keys get bound +inf.  Otherwise
//                        the key (INT64_MAX when there is none) is kept and the bound is val[i][k-1], a lower
//                        bound of every unlisted edge.  A component whose chosen edge (the minimum of its
//                        members' keys, every key a real edge) is strictly below its members' smallest bound is
//                        then certified (engine._mst_contract): an inexact member's better edge, if any, is
//                        unlisted and at least its bound long.
#include <climits>
#include <cmath>

#include "hsd_common.cuh"

namespace hsd {

constexpr int PM_COLS = 256;                       // panel min: columns (threads) per CTA
constexpr int PM_ROWS = 32;                        // panel min: rows per CTA
constexpr int PM_UNROLL = 8;                       // rows whose loads are in flight together
constexpr int PM_WARPS = PM_COLS / 32;
constexpr int LC_WARPS = 8;                        // list candidates: nodes per CTA
constexpr long long KEY_NONE = LLONG_MAX;

template <bool MREACH>
__global__ void __launch_bounds__(PM_COLS)
mst_panel_min_kernel(const float* __restrict__ blk, int64_t ld, int n_rows, int n_cols, int node0,
                     const int32_t* __restrict__ comp, const float* __restrict__ core,
                     long long* __restrict__ key_io) {
    __shared__ int32_t row_comp[PM_ROWS];
    __shared__ uint32_t row_core[MREACH ? PM_ROWS : 1];
    __shared__ long long row_min[PM_ROWS][PM_WARPS];
    const int r0 = blockIdx.y * PM_ROWS, c0 = blockIdx.x * PM_COLS;
    if (c0 + PM_COLS - 1 <= r0) return;                               // tile at or below the diagonal: uniform
    const int rows = min(PM_ROWS, n_rows - r0);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x < rows) {
        row_comp[threadIdx.x] = __ldg(comp + node0 + r0 + threadIdx.x);
        if (MREACH) row_core[threadIdx.x] = __float_as_uint(__ldg(core + node0 + r0 + threadIdx.x));
    }
    __syncthreads();
    const int c = c0 + threadIdx.x;
    const bool col_in = c < n_cols;
    const int comp_c = col_in ? __ldg(comp + node0 + c) : 0;
    const uint32_t core_c = MREACH && col_in ? __float_as_uint(__ldg(core + node0 + c)) : 0u;
    uint32_t col_bits = UINT_MAX;                                     // column minimum: (bits, first row)
    int col_row = 0;
    for (int rb = 0; rb < rows; rb += PM_UNROLL) {
        float v[PM_UNROLL];
        bool ok[PM_UNROLL];
#pragma unroll
        for (int q = 0; q < PM_UNROLL; ++q) {                         // PM_UNROLL row loads in flight
            const int rr = rb + q, r = r0 + rr;
            const bool in = rr < rows && col_in && c > r;             // upper part only
            ok[q] = in && row_comp[rr < rows ? rr : 0] != comp_c;
            v[q] = in ? blk[(int64_t)r * ld + c] : 0.f;
        }
#pragma unroll
        for (int q = 0; q < PM_UNROLL; ++q) {
            const int rr = rb + q;
            if (rr >= rows) break;                                    // uniform over the CTA
            uint32_t bits = ok[q] ? __float_as_uint(v[q]) : UINT_MAX;
            if (MREACH && ok[q]) bits = max(bits, max(row_core[rr], core_c));   // values >= 0: max on the bits
            if (bits < col_bits) {                                    // rows ascend: the first row keeps a tie
                col_bits = bits;
                col_row = r0 + rr;
            }
            const uint32_t wb = __reduce_min_sync(0xffffffffu, bits);
            const uint32_t wc = __reduce_min_sync(0xffffffffu, bits == wb ? (uint32_t)c : UINT_MAX);
            if (lane == 0)
                row_min[rr][warp] = wb == UINT_MAX ? KEY_NONE : (long long)wb << 32 | (uint32_t)(node0 + (int)wc);
        }
    }
    if (col_bits != UINT_MAX) atomicMin(key_io + node0 + c, (long long)col_bits << 32 | (uint32_t)(node0 + col_row));
    __syncthreads();
    if (threadIdx.x < rows) {
        long long m = row_min[threadIdx.x][0];
#pragma unroll
        for (int w = 1; w < PM_WARPS; ++w) m = min(m, row_min[threadIdx.x][w]);
        if (m != KEY_NONE) atomicMin(key_io + node0 + r0 + threadIdx.x, m);
    }
}

__global__ void __launch_bounds__(LC_WARPS * 32)
mst_list_candidates_kernel(const int32_t* __restrict__ idx, const float* __restrict__ val, int n, int k,
                           const int32_t* __restrict__ comp, long long* __restrict__ key_out,
                           float* __restrict__ bound_out) {
    const int i = blockIdx.x * LC_WARPS + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (i >= n) return;                                               // warps are independent
    const int32_t* li = idx + (int64_t)i * k;
    const float* lv = val + (int64_t)i * k;
    const int ci = __ldg(comp + i);
    for (int t0 = 0; t0 < k; t0 += 32) {
        const int t = t0 + lane;
        const int j = t < k ? __ldg(li + t) : -1;
        const uint32_t out = __ballot_sync(0xffffffffu, j >= 0 && __ldg(comp + j) != ci);
        if (out) {                                                    // the first entry outside: the exact best
            const int f = __ffs(out) - 1;
            if (lane == f) {
                key_out[i] = (long long)__float_as_uint(__ldg(lv + t)) << 32 | (uint32_t)j;
                bound_out[i] = INFINITY;
            }
            return;
        }
    }
    if (lane == 0) {                                                  // every entry inside the component
        key_out[i] = KEY_NONE;
        const bool full = __ldg(li + k - 1) >= 0;                     // a short list holds every other node
        bound_out[i] = full ? __ldg(lv + k - 1) : INFINITY;
    }
}

__global__ void __launch_bounds__(LC_WARPS * 32)
mst_list_candidates_mreach_kernel(const int32_t* __restrict__ idx, const float* __restrict__ val, int n, int k,
                                  const int32_t* __restrict__ comp, const float* __restrict__ core,
                                  long long* __restrict__ key_out, float* __restrict__ bound_out) {
    const int i = blockIdx.x * LC_WARPS + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (i >= n) return;                                               // warps are independent
    const int32_t* li = idx + (int64_t)i * k;
    const float* lv = val + (int64_t)i * k;
    const int ci = __ldg(comp + i);
    const uint32_t core_i = __float_as_uint(__ldg(core + i));
    uint32_t best_bits = UINT_MAX, best_j = UINT_MAX;                 // this lane's minimum of (d_mr bits, j)
    for (int t0 = 0; t0 < k; t0 += 32) {
        const int t = t0 + lane;
        const int j = t < k ? __ldg(li + t) : -1;
        if (j >= 0 && __ldg(comp + j) != ci) {
            const uint32_t bits = max(core_i, max(__float_as_uint(__ldg(core + j)), __float_as_uint(__ldg(lv + t))));
            if (bits < best_bits || (bits == best_bits && (uint32_t)j < best_j)) {
                best_bits = bits;
                best_j = (uint32_t)j;
            }
        }
    }
    const uint32_t wb = __reduce_min_sync(0xffffffffu, best_bits);
    const uint32_t wj = __reduce_min_sync(0xffffffffu, best_bits == wb ? best_j : UINT_MAX);
    if (lane == 0) {
        const bool full = __ldg(li + k - 1) >= 0;                     // a short list holds every other node
        const float last = __ldg(lv + k - 1);
        const bool exact = !full || wb < __float_as_uint(last);       // none (UINT_MAX) is never below
        key_out[i] = wb == UINT_MAX ? KEY_NONE : (long long)wb << 32 | wj;
        bound_out[i] = exact ? INFINITY : last;
    }
}

}  // namespace hsd

extern "C" int hsd_mst_panel_min(const float* blk, int64_t ld, int32_t n_rows, int32_t n_cols, int32_t node0,
                                 const int32_t* comp, int64_t* key_io, void* stream) {
    using namespace hsd;
    HSD_REQUIRE(blk && comp && key_io, "null pointer");
    HSD_REQUIRE(n_rows >= 0 && n_cols >= 0 && ld >= n_cols, "bad sizes (ld must be >= n_cols)");
    HSD_REQUIRE(n_rows <= n_cols, "n_rows must be <= n_cols (block row r is block column r)");
    HSD_REQUIRE(node0 >= 0 && (int64_t)node0 + n_cols <= INT32_MAX, "node ids must be non-negative int32");
    HSD_REQUIRE(n_rows <= (int64_t)PM_ROWS * 65535, "n_rows too large");
    if (n_rows == 0) return HSD_OK;
    const dim3 grid((unsigned)((n_cols + PM_COLS - 1) / PM_COLS), (unsigned)((n_rows + PM_ROWS - 1) / PM_ROWS));
    mst_panel_min_kernel<false><<<grid, PM_COLS, 0, (cudaStream_t)stream>>>(blk, ld, n_rows, n_cols, node0, comp,
                                                                             nullptr, (long long*)key_io);
    HSD_CUDA_TRY(cudaGetLastError());
    return HSD_OK;
}

extern "C" int hsd_mst_list_candidates(const int32_t* idx, const float* val, int32_t n, int32_t k,
                                       const int32_t* comp, int64_t* key_out, float* bound_out, void* stream) {
    using namespace hsd;
    HSD_REQUIRE(idx && val && comp && key_out && bound_out, "null pointer");
    HSD_REQUIRE(k >= 1 && k <= 64, "k must be in 1..64");
    HSD_REQUIRE(n >= 0, "bad sizes (n must be >= 0)");
    if (n == 0) return HSD_OK;
    const unsigned grid = (unsigned)((n + LC_WARPS - 1) / LC_WARPS);
    mst_list_candidates_kernel<<<grid, LC_WARPS * 32, 0, (cudaStream_t)stream>>>(idx, val, n, k, comp,
                                                                                  (long long*)key_out, bound_out);
    HSD_CUDA_TRY(cudaGetLastError());
    return HSD_OK;
}

extern "C" int hsd_mst_panel_min_mreach(const float* blk, int64_t ld, int32_t n_rows, int32_t n_cols, int32_t node0,
                                        const int32_t* comp, const float* core, int64_t* key_io, void* stream) {
    using namespace hsd;
    HSD_REQUIRE(blk && comp && core && key_io, "null pointer");
    HSD_REQUIRE(n_rows >= 0 && n_cols >= 0 && ld >= n_cols, "bad sizes (ld must be >= n_cols)");
    HSD_REQUIRE(n_rows <= n_cols, "n_rows must be <= n_cols (block row r is block column r)");
    HSD_REQUIRE(node0 >= 0 && (int64_t)node0 + n_cols <= INT32_MAX, "node ids must be non-negative int32");
    HSD_REQUIRE(n_rows <= (int64_t)PM_ROWS * 65535, "n_rows too large");
    if (n_rows == 0) return HSD_OK;
    const dim3 grid((unsigned)((n_cols + PM_COLS - 1) / PM_COLS), (unsigned)((n_rows + PM_ROWS - 1) / PM_ROWS));
    mst_panel_min_kernel<true><<<grid, PM_COLS, 0, (cudaStream_t)stream>>>(blk, ld, n_rows, n_cols, node0, comp,
                                                                            core, (long long*)key_io);
    HSD_CUDA_TRY(cudaGetLastError());
    return HSD_OK;
}

extern "C" int hsd_mst_list_candidates_mreach(const int32_t* idx, const float* val, int32_t n, int32_t k,
                                              const int32_t* comp, const float* core, int64_t* key_out,
                                              float* bound_out, void* stream) {
    using namespace hsd;
    HSD_REQUIRE(idx && val && comp && core && key_out && bound_out, "null pointer");
    HSD_REQUIRE(k >= 1 && k <= 64, "k must be in 1..64");
    HSD_REQUIRE(n >= 0, "bad sizes (n must be >= 0)");
    if (n == 0) return HSD_OK;
    const unsigned grid = (unsigned)((n + LC_WARPS - 1) / LC_WARPS);
    mst_list_candidates_mreach_kernel<<<grid, LC_WARPS * 32, 0, (cudaStream_t)stream>>>(
        idx, val, n, k, comp, core, (long long*)key_out, bound_out);
    HSD_CUDA_TRY(cudaGetLastError());
    return HSD_OK;
}
