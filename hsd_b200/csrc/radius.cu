// K7 radius graph over row panels — every node pair within a distance r, as a symmetric CSR graph,
// without the N x N matrix ever existing (engine.degree_radius).  A panel is the block B[R][ld] the
// k-NN sweep builds: block row r is node r0 + r, block column c is node r0 + c (c < n_cols), and its
// upper part (c > r) holds every unordered pair the panel owns, each exactly once.
//
//   radius_count      reads the upper part once (a warp reads 32 consecutive values of a row: coalesced)
//                     and writes the hit bitmap H[r][c / 32] (one __ballot_sync per word), per-row hit counts
//                     and per-column hit counts of every chunk of HSD_RADIUS_CHUNK_ROWS rows.  Integer atomics
//                     on the counts: their totals do not depend on the schedule.  Lanes never read the ld
//                     padding or the part c <= r.
//   radius_emit_rows  one warp per row walks the row's bitmap words and gathers its hits in ascending c:
//                     (col_node0 + c, B[r][c]) at row_off[r]: the panel's upper rows;
//   radius_emit_cols  one thread per (column, row chunk) walks the bitmap down the chunk's rows r < c (a CTA
//                     spans 256 consecutive columns, so a bitmap row read is one 32-byte sector) and writes
//                     (row_node0 + r, B[r][c]) in ascending r at col_off[c][chunk]: the lower entries the
//                     panel's columns receive.  The row chunks give a tall panel enough CTAs to hide latency;
//   radius_merge_parts  the ranks' partial CSRs of a sharded sweep (engine.degree_radius with world > 1) into
//                     one: each entry's slot is its rank among its row's entries of every part, from binary
//                     searches (no atomics), so hub rows of N - 1 entries balance like short ones;
//   radius_scatter    assembly: 8 lanes per segment (a node's piece of one panel) copy the piece to
//                     idx_out / val_out at indptr[node] + cursor[node] and advances the cursor.  Called
//                     once per piece in panel order, column piece before row piece, so every output row
//                     is ascending by construction.
//
// Positions come from exclusive scans of the counts, never from atomics: the output is deterministic.
// Every kernel is instantiated for float (degree mode panels) and double (wavelet mode matrices).
#include <cmath>

#include "hsd_common.cuh"

namespace hsd {

constexpr int RC_THREADS = 256;                    // count pass: RC_ROWS rows x RC_SEG_WORDS words per CTA
constexpr int RC_ROWS = RC_THREADS / 32;           // one warp per row
constexpr int RC_SEG_WORDS = 32;                   // words (x 32 columns) of a row per warp
constexpr int RC_UNROLL = 8;                       // loads in flight per lane of the count pass
constexpr int RE_WARPS = 8;                        // row emit: rows per CTA
constexpr int CE_THREADS = 256;                    // column emit: columns per CTA (8 bitmap words: one sector)
constexpr int CE_UNROLL = 8;                       // bitmap loads in flight per thread of the column emit
constexpr int CHUNK = HSD_RADIUS_CHUNK_ROWS;        // rows per column-count chunk
constexpr int RS_THREADS = 256;                    // scatter: threads per CTA
constexpr int RS_GROUP = 8;                        // scatter: lanes per segment (~20 neighbours per node: short)
constexpr int RM_THREADS = 256;                    // merge of the ranks' parts: threads per CTA
constexpr int RM_MAX_PARTS = 64;                   // parts a merge takes (their starts live in shared memory)
constexpr int RM_CTAS_PER_SM = 8;                  // merge grid: CTAs per SM of the grid-stride loop

template <typename T>
__global__ void __launch_bounds__(RC_THREADS)
radius_count_kernel(const T* __restrict__ blk, int64_t ld, int n_rows, int n_cols, int n_chunks, T thr,
                    uint32_t* __restrict__ hits, int64_t hits_ld, int32_t* __restrict__ row_cnt,
                    int32_t* __restrict__ col_cnt) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int r = blockIdx.x * RC_ROWS + warp;                        // one warp per row of the CTA's row group
    if (r >= n_rows) return;                                          // warps are independent: no block barrier
    const int64_t n_words = (n_cols + 31) >> 5;
    const int64_t w_first = ((int64_t)r + 1) >> 5;                    // first word holding a column c > r
    const int64_t w_end = min((int64_t)(blockIdx.y + 1) * RC_SEG_WORDS, n_words);
    const T* row = blk + (int64_t)r * ld;
    uint32_t* h = hits + (int64_t)r * hits_ld;
    int total = 0;
    for (int64_t w0 = max((int64_t)blockIdx.y * RC_SEG_WORDS, w_first); w0 < w_end; w0 += RC_UNROLL) {
        T v[RC_UNROLL];
        bool ok[RC_UNROLL];
#pragma unroll
        for (int q = 0; q < RC_UNROLL; ++q) {                         // RC_UNROLL coalesced loads in flight
            const int64_t c = (w0 + q) * 32 + lane;
            ok[q] = w0 + q < w_end && c > r && c < n_cols;
            v[q] = ok[q] ? row[c] : T(0);
        }
#pragma unroll
        for (int q = 0; q < RC_UNROLL; ++q) {
            if (w0 + q >= w_end) break;                               // warp-uniform
            const bool hit = ok[q] && v[q] <= thr;
            const uint32_t word = __ballot_sync(0xffffffffu, hit);
            if (lane == 0) h[w0 + q] = word;
            if (hit) atomicAdd(col_cnt + ((w0 + q) * 32 + lane) * n_chunks + r / CHUNK, 1);
            total += __popc(word);
        }
    }
    if (lane == 0 && total) atomicAdd(row_cnt + r, total);
}

template <typename T>
__global__ void __launch_bounds__(RE_WARPS * 32)
radius_emit_rows_kernel(const T* __restrict__ blk, int64_t ld, int n_rows, int n_cols,
                        const uint32_t* __restrict__ hits, int64_t hits_ld, const int64_t* __restrict__ row_off,
                        int col_node0, int32_t* __restrict__ idx_out, T* __restrict__ val_out) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int r = blockIdx.x * RE_WARPS + warp;
    if (r >= n_rows) return;
    const int64_t n_words = (n_cols + 31) >> 5;
    const T* row = blk + (int64_t)r * ld;
    const uint32_t* h = hits + (int64_t)r * hits_ld;
    int64_t base = row_off[r];
    for (int64_t w0 = ((int64_t)r + 1) >> 5; w0 < n_words; w0 += 32) {
        const uint32_t word = (w0 + lane < n_words) ? h[w0 + lane] : 0u;
        int inc = __popc(word);                                       // inclusive scan of the words' hits
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += t;
        }
        const int exc = inc - __popc(word);
        uint32_t nz = __ballot_sync(0xffffffffu, word != 0u);
        while (nz) {
            const int j = __ffs(nz) - 1;
            nz &= nz - 1;
            const uint32_t wj = __shfl_sync(0xffffffffu, word, j);
            const int bj = __shfl_sync(0xffffffffu, exc, j);
            if ((wj >> lane) & 1u) {
                const int64_t pos = base + bj + __popc(wj & ((1u << lane) - 1u));
                const int64_t c = (w0 + j) * 32 + lane;
                idx_out[pos] = col_node0 + (int)c;
                val_out[pos] = row[c];
            }
        }
        base += __shfl_sync(0xffffffffu, inc, 31);
    }
}

template <typename T>
__global__ void __launch_bounds__(CE_THREADS)
radius_emit_cols_kernel(const T* __restrict__ blk, int64_t ld, int n_rows, int n_cols,
                        const uint32_t* __restrict__ hits, int64_t hits_ld, const int64_t* __restrict__ col_off,
                        int row_node0, int32_t* __restrict__ idx_out, T* __restrict__ val_out) {
    const int c = blockIdx.x * CE_THREADS + threadIdx.x;
    const int chunk = blockIdx.y, n_chunks = gridDim.y;
    if (c >= n_cols) return;                                          // columns are independent: no barrier
    const int rows = min(min(c, n_rows), (chunk + 1) * CHUNK);        // rows r < c of this chunk reach column c
    const uint32_t bit = 1u << (c & 31);
    const uint32_t* h = hits + (c >> 5);
    int64_t pos = col_off[(int64_t)c * n_chunks + chunk];
    int r = chunk * CHUNK;
    for (; r + CE_UNROLL <= rows; r += CE_UNROLL) {
        uint32_t w[CE_UNROLL];
#pragma unroll
        for (int q = 0; q < CE_UNROLL; ++q) w[q] = __ldg(h + (int64_t)(r + q) * hits_ld);
#pragma unroll
        for (int q = 0; q < CE_UNROLL; ++q) {
            if (w[q] & bit) {
                idx_out[pos] = row_node0 + r + q;
                val_out[pos] = blk[(int64_t)(r + q) * ld + c];
                ++pos;
            }
        }
    }
    for (; r < rows; ++r) {
        if (__ldg(h + (int64_t)r * hits_ld) & bit) {
            idx_out[pos] = row_node0 + r;
            val_out[pos] = blk[(int64_t)r * ld + c];
            ++pos;
        }
    }
}

template <typename T>
__global__ void __launch_bounds__(RS_THREADS)
radius_scatter_kernel(const int32_t* __restrict__ idx, const T* __restrict__ val, const int64_t* __restrict__ off,
                      int n_seg, int node0, const int64_t* __restrict__ indptr, int64_t* __restrict__ cursor,
                      int32_t* __restrict__ idx_out, T* __restrict__ val_out) {
    const int g = threadIdx.x % RS_GROUP;                             // lane within the segment's group
    const int64_t s = ((int64_t)blockIdx.x * RS_THREADS + threadIdx.x) / RS_GROUP;
    if (s >= n_seg) return;                                           // returns are uniform over a group
    const int64_t src = off[s], len = off[s + 1] - src;
    if (len == 0) return;
    const int node = node0 + (int)s;
    const int64_t dst = indptr[node] + cursor[node];
    for (int64_t t = g; t < len; t += RS_GROUP) {
        idx_out[dst + t] = idx[src + t];
        val_out[dst + t] = val[src + t];
    }
    const unsigned group_mask = ((1u << RS_GROUP) - 1u) << ((threadIdx.x & 31) & ~(RS_GROUP - 1));
    __syncwarp(group_mask);                                           // every lane of the group has read cursor[node]
    if (g == 0) cursor[node] += len;
}

// first index t in [lo, hi) with key < a[t] (upper) or key <= a[t] (lower); hi when there is none
template <bool UPPER, typename K>
__device__ __forceinline__ int64_t bound_in(const K* __restrict__ a, int64_t lo, int64_t hi, K key) {
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (UPPER ? a[mid] <= key : a[mid] < key) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

// One thread per input entry (grid-stride).  Part starts in the flat entry space are a block-wide scan of the
// parts' sizes in shared memory; entry e of part p, row i, at position k of its row goes to
// indptr[i] + k + sum_{q<p} upper_bound(row i of q, id) + sum_{q>p} lower_bound(row i of q, id): the rank of
// (id, p, k) among the row's entries of all parts, so the slots form a permutation whatever the schedule.
template <typename V>
__global__ void __launch_bounds__(RM_THREADS)
radius_merge_parts_kernel(int n_parts, int n_rows, const int64_t* __restrict__ part_indptr,
                          const int64_t* __restrict__ part_base, const int32_t* __restrict__ idx,
                          const V* __restrict__ val, const int64_t* __restrict__ indptr,
                          int32_t* __restrict__ idx_out, V* __restrict__ val_out) {
    __shared__ int64_t start[RM_MAX_PARTS + 1];                       // start[p]: part p's first flat entry
    const int64_t ld = (int64_t)n_rows + 1;
    if (threadIdx.x == 0) {
        int64_t s = 0;
        for (int p = 0; p < n_parts; ++p) {
            start[p] = s;
            s += part_indptr[p * ld + n_rows] - part_indptr[p * ld];
        }
        start[n_parts] = s;
    }
    __syncthreads();
    const int64_t total = start[n_parts];
    for (int64_t e = (int64_t)blockIdx.x * RM_THREADS + threadIdx.x; e < total; e += (int64_t)gridDim.x * RM_THREADS) {
        const int p = (int)bound_in<true>(start, 0, n_parts, e) - 1;   // the last part starting at or before e
        const int64_t* ip = part_indptr + p * ld;
        const int64_t k = ip[0] + (e - start[p]);                     // offset in part p's own indptr
        const int i = (int)bound_in<true>(ip, 0, n_rows + 1, k) - 1;   // row of k (empty rows skipped)
        const int32_t id = idx[part_base[p] + k];
        int64_t slot = indptr[i] + (k - ip[i]);
        for (int q = 0; q < n_parts; ++q) {
            if (q == p) continue;
            const int64_t* iq = part_indptr + q * ld;
            const int32_t* row = idx + part_base[q];
            const int64_t lo = iq[i], hi = iq[i + 1];
            slot += (q < p ? bound_in<true>(row, lo, hi, id) : bound_in<false>(row, lo, hi, id)) - lo;
        }
        idx_out[slot] = id;
        val_out[slot] = val[part_base[p] + k];
    }
}

// the largest T that does not exceed radius (radius >= 0, not NaN): `D <= it` equals `(double)D <= radius`
template <typename T>
static T threshold_of(double radius) {
    T t = (T)radius;
    if ((double)t > radius) t = std::nextafter(t, (T)0);
    return t;
}

template <typename T>
static int launch_count(const void* blk, int64_t ld, int32_t n_rows, int32_t n_cols, double radius, uint32_t* hits,
                        int64_t hits_ld, int32_t* row_cnt, int32_t* col_cnt, cudaStream_t st) {
    HSD_CUDA_TRY(cudaMemsetAsync(row_cnt, 0, sizeof(int32_t) * n_rows, st));
    const int n_chunks = (n_rows + CHUNK - 1) / CHUNK;
    HSD_CUDA_TRY(cudaMemsetAsync(col_cnt, 0, sizeof(int32_t) * n_cols * n_chunks, st));
    const int64_t n_words = (n_cols + 31) / 32;
    const dim3 grid((unsigned)((n_rows + RC_ROWS - 1) / RC_ROWS), (unsigned)((n_words + RC_SEG_WORDS - 1) / RC_SEG_WORDS));
    radius_count_kernel<T><<<grid, RC_THREADS, 0, st>>>((const T*)blk, ld, n_rows, n_cols, n_chunks, threshold_of<T>(radius), hits,
                                                        hits_ld, row_cnt, col_cnt);
    HSD_CUDA_TRY(cudaGetLastError());
    return HSD_OK;
}

}  // namespace hsd

#define HSD_RADIUS_BLOCK_ARGS_OK(blk, elem_bytes, ld, n_rows, n_cols, hits, hits_ld)                          \
    HSD_REQUIRE(blk && hits, "null pointer");                                                                 \
    HSD_REQUIRE(elem_bytes == 4 || elem_bytes == 8, "elem_bytes must be 4 (float) or 8 (double)");           \
    HSD_REQUIRE(n_rows >= 0 && n_cols >= 0 && ld >= n_cols, "bad sizes (ld must be >= n_cols)");              \
    HSD_REQUIRE(hits_ld >= ((int64_t)n_cols + 31) / 32, "hits_ld must be >= ceil(n_cols / 32)")

extern "C" int hsd_radius_count(const void* blk, int32_t elem_bytes, int64_t ld, int32_t n_rows, int32_t n_cols,
                                double radius, uint32_t* hits, int64_t hits_ld, int32_t* row_cnt, int32_t* col_cnt,
                                void* stream) {
    using namespace hsd;
    HSD_RADIUS_BLOCK_ARGS_OK(blk, elem_bytes, ld, n_rows, n_cols, hits, hits_ld);
    HSD_REQUIRE(row_cnt && col_cnt, "null pointer");
    HSD_REQUIRE(!std::isnan(radius) && radius >= 0.0, "radius must be >= 0 and not NaN");
    HSD_REQUIRE(((int64_t)n_cols + 31) / 32 <= (int64_t)RC_SEG_WORDS * 65535, "n_cols too large");
    HSD_REQUIRE(n_rows <= (int64_t)CHUNK * 65535, "n_rows too large");
    if (n_rows == 0 || n_cols == 0) {
        if (n_rows) HSD_CUDA_TRY(cudaMemsetAsync(row_cnt, 0, sizeof(int32_t) * n_rows, (cudaStream_t)stream));
        return HSD_OK;
    }
    return elem_bytes == 4
        ? launch_count<float>(blk, ld, n_rows, n_cols, radius, hits, hits_ld, row_cnt, col_cnt, (cudaStream_t)stream)
        : launch_count<double>(blk, ld, n_rows, n_cols, radius, hits, hits_ld, row_cnt, col_cnt, (cudaStream_t)stream);
}

extern "C" int hsd_radius_emit_rows(const void* blk, int32_t elem_bytes, int64_t ld, int32_t n_rows, int32_t n_cols,
                                    const uint32_t* hits, int64_t hits_ld, const int64_t* row_off, int32_t col_node0,
                                    int32_t* idx_out, void* val_out, void* stream) {
    using namespace hsd;
    HSD_RADIUS_BLOCK_ARGS_OK(blk, elem_bytes, ld, n_rows, n_cols, hits, hits_ld);
    HSD_REQUIRE(row_off && idx_out && val_out, "null pointer");
    HSD_REQUIRE(col_node0 >= 0 && (int64_t)col_node0 + n_cols <= INT32_MAX, "node ids must be non-negative int32");
    if (n_rows == 0 || n_cols == 0) return HSD_OK;
    const unsigned grid = (unsigned)((n_rows + RE_WARPS - 1) / RE_WARPS);
    const cudaStream_t st = (cudaStream_t)stream;
    if (elem_bytes == 4)
        radius_emit_rows_kernel<float><<<grid, RE_WARPS * 32, 0, st>>>((const float*)blk, ld, n_rows, n_cols, hits,
                                                                        hits_ld, row_off, col_node0, idx_out,
                                                                        (float*)val_out);
    else
        radius_emit_rows_kernel<double><<<grid, RE_WARPS * 32, 0, st>>>((const double*)blk, ld, n_rows, n_cols, hits,
                                                                         hits_ld, row_off, col_node0, idx_out,
                                                                         (double*)val_out);
    HSD_CUDA_TRY(cudaGetLastError());
    return HSD_OK;
}

extern "C" int hsd_radius_emit_cols(const void* blk, int32_t elem_bytes, int64_t ld, int32_t n_rows, int32_t n_cols,
                                    const uint32_t* hits, int64_t hits_ld, const int64_t* col_off, int32_t row_node0,
                                    int32_t* idx_out, void* val_out, void* stream) {
    using namespace hsd;
    HSD_RADIUS_BLOCK_ARGS_OK(blk, elem_bytes, ld, n_rows, n_cols, hits, hits_ld);
    HSD_REQUIRE(col_off && idx_out && val_out, "null pointer");
    HSD_REQUIRE(row_node0 >= 0 && (int64_t)row_node0 + n_rows <= INT32_MAX, "node ids must be non-negative int32");
    HSD_REQUIRE(n_rows <= (int64_t)CHUNK * 65535, "n_rows too large");
    if (n_rows == 0 || n_cols == 0) return HSD_OK;
    const dim3 grid((unsigned)((n_cols + CE_THREADS - 1) / CE_THREADS), (unsigned)((n_rows + CHUNK - 1) / CHUNK));
    const cudaStream_t st = (cudaStream_t)stream;
    if (elem_bytes == 4)
        radius_emit_cols_kernel<float><<<grid, CE_THREADS, 0, st>>>((const float*)blk, ld, n_rows, n_cols, hits,
                                                                     hits_ld, col_off, row_node0, idx_out,
                                                                     (float*)val_out);
    else
        radius_emit_cols_kernel<double><<<grid, CE_THREADS, 0, st>>>((const double*)blk, ld, n_rows, n_cols, hits,
                                                                      hits_ld, col_off, row_node0, idx_out,
                                                                      (double*)val_out);
    HSD_CUDA_TRY(cudaGetLastError());
    return HSD_OK;
}

extern "C" int hsd_radius_scatter(const int32_t* idx, const void* val, int32_t elem_bytes, const int64_t* off,
                                  int32_t n_seg, int32_t node0, const int64_t* indptr, int64_t* cursor,
                                  int32_t* idx_out, void* val_out, void* stream) {
    using namespace hsd;
    HSD_REQUIRE(off && indptr && cursor && idx_out && val_out, "null pointer");
    HSD_REQUIRE(elem_bytes == 4 || elem_bytes == 8, "elem_bytes must be 4 (float) or 8 (double)");
    HSD_REQUIRE(n_seg >= 0 && node0 >= 0 && (int64_t)node0 + n_seg <= INT32_MAX, "bad sizes");
    if (n_seg == 0) return HSD_OK;
    HSD_REQUIRE(idx && val, "null pointer");                          // an empty piece may have no storage
    const unsigned grid = (unsigned)(((int64_t)n_seg * RS_GROUP + RS_THREADS - 1) / RS_THREADS);
    const cudaStream_t st = (cudaStream_t)stream;
    if (elem_bytes == 4)
        radius_scatter_kernel<float><<<grid, RS_THREADS, 0, st>>>(idx, (const float*)val, off, n_seg, node0, indptr,
                                                                      cursor, idx_out, (float*)val_out);
    else
        radius_scatter_kernel<double><<<grid, RS_THREADS, 0, st>>>(idx, (const double*)val, off, n_seg, node0,
                                                                       indptr, cursor, idx_out, (double*)val_out);
    HSD_CUDA_TRY(cudaGetLastError());
    return HSD_OK;
}

extern "C" int hsd_radius_merge_parts(int32_t n_parts, int32_t n_rows, const int64_t* part_indptr,
                                      const int64_t* part_base, const int32_t* idx, const void* val,
                                      int32_t elem_bytes, const int64_t* indptr, int32_t* idx_out, void* val_out,
                                      void* stream) {
    using namespace hsd;
    HSD_REQUIRE(part_indptr && part_base && idx && val && indptr && idx_out && val_out, "null pointer");
    HSD_REQUIRE(elem_bytes == 4 || elem_bytes == 8, "elem_bytes must be 4 (float) or 8 (double)");
    HSD_REQUIRE(n_parts >= 1 && n_parts <= RM_MAX_PARTS, "n_parts must be in 1..64");
    HSD_REQUIRE(n_rows >= 0, "bad sizes (n_rows must be >= 0)");
    if (n_rows == 0) return HSD_OK;
    int dev = 0, sms = 0;
    HSD_CUDA_TRY(cudaGetDevice(&dev));
    HSD_CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const unsigned grid = (unsigned)(sms * RM_CTAS_PER_SM);
    const cudaStream_t st = (cudaStream_t)stream;
    if (elem_bytes == 4)     // the distances are copied as bit patterns
        radius_merge_parts_kernel<uint32_t><<<grid, RM_THREADS, 0, st>>>(n_parts, n_rows, part_indptr, part_base, idx,
                                                                         (const uint32_t*)val, indptr, idx_out,
                                                                         (uint32_t*)val_out);
    else
        radius_merge_parts_kernel<uint64_t><<<grid, RM_THREADS, 0, st>>>(n_parts, n_rows, part_indptr, part_base, idx,
                                                                         (const uint64_t*)val, indptr, idx_out,
                                                                         (uint64_t*)val_out);
    HSD_CUDA_TRY(cudaGetLastError());
    return HSD_OK;
}
