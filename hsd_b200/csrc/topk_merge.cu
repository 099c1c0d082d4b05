// K7 over row panels — merging k-nearest-neighbour lists, so that the k-NN of every node can be
// found without the N x N matrix ever existing (engine.degree_knn).  The panel sweep computes a
// block B = rows [r0, r1) x columns [r0, N) at a time; hsd_topk_rows selects along its rows, and the
// two kernels here fold the results into running per-node lists:
//
//   topk_merge       list-of-lists merge (the row pass, n_lists = 1; the reduction over the ranks of
//                    a multi-GPU sweep, n_lists = world).  One warp per row stages the running list and
//                    the candidate lists in shared memory; every element finds its output position as
//                    its index in its own list plus, for every other list, the number of elements that
//                    sort before it there (binary search; equal keys are ordered by list number, so the
//                    -1 / +inf padding lands last and each output slot has exactly one writer);
//   topk_merge_cols  the column pass: block column c (node col_node0 + c) receives the candidates
//                    (B[r][c], row_node0 + r) of every block row.  One thread per column streams its
//                    column top to bottom (a warp reads 32 consecutive floats of a row: coalesced), keeps
//                    its running list sorted in shared memory (entry t of the CTA's column q at
//                    [t][q]: conflict-free) and the list's current k-th entry in registers; a candidate
//                    that sorts before that entry is inserted by shifting the tail.  Once the list has
//                    warmed up almost every candidate fails the one register compare.
//
// Order everywhere: (distance, node id) with the id compared unsigned, so the -1 padding sorts after
// every real id; distances are >= 0 and finite.  No atomics: results do not depend on the schedule.
#include "hsd_common.cuh"

namespace hsd {

constexpr int TM_MAX_K = 64;        // the k limit of hsd_topk_rows (TK_MAX in topk.cu)
constexpr int TM_MAX_LISTS = 64;
constexpr int TM_WARPS = 4;         // rows per CTA of the list merge
constexpr int TC_THREADS = 128;     // columns per CTA of the column pass
constexpr int TC_UNROLL = 16;       // loads in flight per thread of the column pass

// (val a, id ia) sorts before (val b, id ib)
__device__ __forceinline__ bool tm_before(float a, int ia, float b, int ib) {
    return a < b || (a == b && (uint32_t)ia < (uint32_t)ib);
}

__global__ void __launch_bounds__(TM_WARPS * 32)
topk_merge_kernel(const int32_t* __restrict__ idx_in, const float* __restrict__ val_in, int n_lists,
                  int64_t list_stride, int idx_offset, int n_rows, int k, int warps,
                  int32_t* __restrict__ idx_io, float* __restrict__ val_io) {
    extern __shared__ __align__(16) unsigned char tm_smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int L = n_lists + 1;                       // list 0: the running list
    const int row = blockIdx.x * warps + warp;
    if (warp >= warps || row >= n_rows) return;      // warps work independently: no block barrier below
    float* sv = reinterpret_cast<float*>(tm_smem) + (int64_t)warp * L * k * 2;
    int* si = reinterpret_cast<int*>(sv + L * k);
    const int64_t base = (int64_t)row * k;
    for (int e = lane; e < L * k; e += 32) {
        const int l = e / k, t = e - l * k;
        if (l == 0) {
            sv[e] = val_io[base + t];
            si[e] = idx_io[base + t];
        } else {
            const int64_t o = (int64_t)(l - 1) * list_stride + base + t;
            const int id = __ldg(idx_in + o);
            sv[e] = __ldg(val_in + o);
            si[e] = (id == -1) ? -1 : id + idx_offset;
        }
    }
    __syncwarp();
    for (int e = lane; e < L * k; e += 32) {
        const int l = e / k, t = e - l * k;
        const float v = sv[e];
        const int id = si[e];
        int pos = t;
        for (int m = 0; m < L && pos < k; ++m) {
            if (m == l) continue;
            const float* mv = sv + m * k;
            const int* mi = si + m * k;
            // elements of list m placed before this one: those sorting before it, and equal ones of lower lists
            int lo = 0, hi = k;
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                const bool before = (m < l) ? !tm_before(v, id, mv[mid], mi[mid]) : tm_before(mv[mid], mi[mid], v, id);
                if (before) lo = mid + 1; else hi = mid;
            }
            pos += lo;
        }
        if (pos < k) {
            val_io[base + pos] = v;
            idx_io[base + pos] = id;
        }
    }
}

__global__ void __launch_bounds__(TC_THREADS)
topk_merge_cols_kernel(const float* __restrict__ blk, int64_t ld, int n_rows, int c_begin, int n_cols,
                       int row_node0, int col_node0, int k, int32_t* __restrict__ idx_io,
                       float* __restrict__ val_io) {
    extern __shared__ __align__(16) unsigned char tc_smem[];
    float* lv = reinterpret_cast<float*>(tc_smem);                 // [k][TC_THREADS]
    int* li = reinterpret_cast<int*>(lv + k * TC_THREADS);         // [k][TC_THREADS]
    const int tid = threadIdx.x;
    const int c = c_begin + blockIdx.x * TC_THREADS + tid;
    if (c >= n_cols) return;                                       // columns are independent: no barrier below
    const int64_t base = ((int64_t)col_node0 + c) * k;
    for (int t = 0; t < k; ++t) {
        lv[t * TC_THREADS + tid] = val_io[base + t];
        li[t * TC_THREADS + tid] = idx_io[base + t];
    }
    float tv = lv[(k - 1) * TC_THREADS + tid];                     // the current k-th entry
    int ti = li[(k - 1) * TC_THREADS + tid];
    auto offer = [&](float v, int id) {
        if (!tm_before(v, id, tv, ti)) return;
        int p = k - 1;                                             // the old k-th entry drops out
        while (p > 0 && tm_before(v, id, lv[(p - 1) * TC_THREADS + tid], li[(p - 1) * TC_THREADS + tid])) {
            lv[p * TC_THREADS + tid] = lv[(p - 1) * TC_THREADS + tid];
            li[p * TC_THREADS + tid] = li[(p - 1) * TC_THREADS + tid];
            --p;
        }
        lv[p * TC_THREADS + tid] = v;
        li[p * TC_THREADS + tid] = id;
        tv = lv[(k - 1) * TC_THREADS + tid];
        ti = li[(k - 1) * TC_THREADS + tid];
    };
    const float* col = blk + c;
    int r = 0;
    for (; r + TC_UNROLL <= n_rows; r += TC_UNROLL) {
        float v[TC_UNROLL];
#pragma unroll
        for (int q = 0; q < TC_UNROLL; ++q) v[q] = __ldg(col + (int64_t)(r + q) * ld);
#pragma unroll
        for (int q = 0; q < TC_UNROLL; ++q) offer(v[q], row_node0 + r + q);
    }
    for (; r < n_rows; ++r) offer(__ldg(col + (int64_t)r * ld), row_node0 + r);
    for (int t = 0; t < k; ++t) {
        val_io[base + t] = lv[t * TC_THREADS + tid];
        idx_io[base + t] = li[t * TC_THREADS + tid];
    }
}

}  // namespace hsd

extern "C" int hsd_topk_merge(const int32_t* idx_in, const float* val_in, int32_t n_lists, int64_t list_stride,
                              int32_t idx_offset, int32_t n_rows, int32_t k, int32_t* idx_io, float* val_io,
                              void* stream) {
    using namespace hsd;
    HSD_REQUIRE(idx_in && val_in && idx_io && val_io, "null pointer");
    HSD_REQUIRE(k >= 1 && k <= TM_MAX_K, "k must be in 1..64");
    HSD_REQUIRE(n_lists >= 1 && n_lists <= TM_MAX_LISTS, "n_lists must be in 1..64");
    HSD_REQUIRE(n_rows >= 0, "bad sizes");
    HSD_REQUIRE(n_lists == 1 || list_stride >= (int64_t)n_rows * k, "list_stride must be >= n_rows * k");
    HSD_REQUIRE(idx_offset >= 0, "idx_offset must be >= 0");
    if (n_rows == 0) return HSD_OK;
    const int per_warp = (n_lists + 1) * k * 8;                    // <= 33 KB
    const int warps = per_warp * TM_WARPS <= 48 * 1024 ? TM_WARPS : (48 * 1024) / per_warp;
    const unsigned grid = (unsigned)((n_rows + warps - 1) / warps);
    topk_merge_kernel<<<grid, TM_WARPS * 32, per_warp * warps, (cudaStream_t)stream>>>(
        idx_in, val_in, n_lists, list_stride, idx_offset, n_rows, k, warps, idx_io, val_io);
    HSD_CUDA_TRY(cudaGetLastError());
    return HSD_OK;
}

extern "C" int hsd_topk_merge_cols(const float* blk, int64_t ld, int32_t n_rows, int32_t c_begin, int32_t n_cols,
                                   int32_t row_node0, int32_t col_node0, int32_t k, int32_t* idx_io, float* val_io,
                                   void* stream) {
    using namespace hsd;
    HSD_REQUIRE(blk && idx_io && val_io, "null pointer");
    HSD_REQUIRE(k >= 1 && k <= TM_MAX_K, "k must be in 1..64");
    HSD_REQUIRE(n_rows >= 0 && n_cols >= 0 && ld >= n_cols, "bad sizes (ld must be >= n_cols)");
    HSD_REQUIRE(c_begin >= 0 && c_begin <= n_cols, "c_begin must be in 0..n_cols");
    HSD_REQUIRE(row_node0 >= 0 && col_node0 >= 0 && (int64_t)row_node0 + n_rows <= INT32_MAX,
                "node ids must be non-negative int32");
    if (n_rows == 0 || c_begin == n_cols) return HSD_OK;
    const int smem = k * TC_THREADS * 8;                           // <= 64 KB
    HSD_CUDA_TRY(cudaFuncSetAttribute(topk_merge_cols_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    const unsigned grid = (unsigned)((n_cols - c_begin + TC_THREADS - 1) / TC_THREADS);
    topk_merge_cols_kernel<<<grid, TC_THREADS, smem, (cudaStream_t)stream>>>(
        blk, ld, n_rows, c_begin, n_cols, row_node0, col_node0, k, idx_io, val_io);
    HSD_CUDA_TRY(cudaGetLastError());
    return HSD_OK;
}
