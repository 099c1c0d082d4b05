/*
 * hsd_b200.h — C-ABI of the B200-native HSD structural-distance hot path.
 *
 * The reference (Sngunfei/HSD) is pure Python and has no FFI of its own; the
 * boundary it exposes is the Python class API of model/HSD.py,
 * model/multiscale_HSD.py, model/dynamic_HSD.py and tools/hierarchy.py.  The
 * entry points below are what a ctypes binding behind those classes calls
 * (see INTEGRATION.md for the binding stub).  Each one cites the reference
 * loop (file:line under the reference tree) it replaces.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller unless the name
 *     ends in `_host`; no hidden allocation, no hidden synchronisation;
 *   - `stream` is a cudaStream_t passed as void*; work is enqueued on it and
 *     the call returns immediately;
 *   - return value: 0 = HSD_OK, negative = error (hsd_last_error_string());
 *   - node ids are int32; the CSR handed to the BFS entry points must be in
 *     *degree-ascending node order* (ties by original id).  That order is what
 *     lets the per-ring degree CDF be a prefix-popcount over the ring bitmap
 *     instead of a histogram with atomics (DESIGN.md §3).
 */
#ifndef HSD_B200_H
#define HSD_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HSD_OK                 0
#define HSD_ERR_INVALID       -1   /* bad argument */
#define HSD_ERR_CUDA          -2   /* a CUDA runtime/driver call failed */
#define HSD_ERR_UNSUPPORTED   -3   /* size outside what the kernels handle */
#define HSD_ERR_NO_DEVICE     -4   /* no sm_100 device / driver entry point */

#define HSD_PAIR_TILE        128   /* pairwise kernel tile edge (nodes) */
#define HSD_PAIR_KCHUNK       16   /* pairwise kernel K chunk (signature rows) */

int         hsd_version(void);
const char* hsd_last_error_string(void);

/* ---- K1/K2: k-hop rings + per-ring degree CDF ------------------------------
 * Replaces tools/hierarchy.py:16-38 (get_hierarchical_representation /
 * get_node_hierarchical_structure: level-synchronous BFS, rings kept as sets)
 * and, in degree mode, the per-ring sort inside
 * scipy.stats.wasserstein_distance as called from model/HSD.py:103-112.
 *
 * One CTA per source.  The seen set, the ring bitmaps and the ring's prefix
 * popcount are N-bit / N/32-word arrays in shared memory; the frontier ring is
 * compacted and expanded edge-balanced (every thread walks an equal share of the
 * concatenated adjacency lists with 16-byte loads).  For hop h = 1..hops the ring
 * bitmap is turned into
 *   sig[row][1 + (h-1)*(n_bins-1) + b] = CDF_h(support[b]) * (support[b+1]-support[b])
 * for b = 0..n_bins-2, and sig[row][0] = degree(source) (the hop-0 ring is the
 * source alone, so its W1 term is |deg_i - deg_j|).  L1 distance between two
 * such rows == sum over hops of the 1-D Wasserstein-1 distance between the
 * degree multisets of the rings.
 *
 *   rowptr[n_nodes+1], col[nnz]   CSR, degree-ascending node order; col must be 16-byte aligned and
 *                                 readable up to the next multiple of 4 entries (it is read with LDG.128)
 *   src_nodes[n_src]              sources (ids in that order)
 *   out_rows[n_src]               row of sig / ring_sizes / ring_bitmaps each source writes
 *   bin_end[n_bins]               # nodes with degree <= support[b]  (== first id of bin b+1)
 *   delta[n_bins-1]               support[b+1]-support[b]
 *   sig (nullable)                float[rows][sig_ld], sig_ld >= 1 + hops*(n_bins-1)
 *   ring_sizes (nullable)         int32[rows][hops+1]
 *   ring_bitmaps (nullable)       uint32[rows][hops+1][ceil(n_nodes/32)]
 *   empty_as_zero                 0: an empty ring sets *status |= 1 (caller raises, like scipy);
 *                                 1: an empty ring is the point mass at 0 (tools/metrics.py:18-36 padding)
 *   status                        int32[1], OR-ed flags, caller zeroes it
 *   cta_threads                   0 = pick from the graph size; 128/256/512/1024 to override (one hub
 *                                 source is latency-bound inside its CTA: hubs finish ~2x sooner with 1024
 *                                 threads, low-degree sources run best with 256)
 */
int hsd_ring_signature_degree(const int32_t* rowptr, const int32_t* col, int32_t n_nodes,
                              const int32_t* src_nodes, const int32_t* out_rows, int32_t n_src,
                              int32_t hops,
                              const int32_t* bin_end, const float* delta, int32_t n_bins,
                              float* sig, int64_t sig_ld,
                              int32_t* ring_sizes, uint32_t* ring_bitmaps,
                              int32_t empty_as_zero, int32_t* status, int32_t cta_threads, void* stream);

/* Same kernel with the all-gather of the signature table fused in: every signature row is
 * stored into the local table AND into n_peers peer-mapped copies of it (sig_peers: DEVICE
 * array of n_peers base pointers, same layout; NVLink peer memory) as it is produced, so the
 * ranks of a sharded run need no collective afterwards — only a barrier.  The reference's
 * counterpart is pickling the whole model into every Pool task (model/HSD.py:122-124). */
int hsd_ring_signature_degree_allgather(const int32_t* rowptr, const int32_t* col, int32_t n_nodes,
                                        const int32_t* src_nodes, const int32_t* out_rows, int32_t n_src,
                                        int32_t hops, const int32_t* bin_end, const float* delta,
                                        int32_t n_bins, float* sig, int64_t sig_ld,
                                        float* const* sig_peers, int32_t n_peers,
                                        int32_t* ring_sizes, int32_t empty_as_zero, int32_t* status,
                                        int32_t cta_threads, void* stream);

/* Dense variant of the two entry points above, for when (almost) every node is a source: the balls obey
 * ball_h(s) = {s} U OR_{u in N(s)} ball_{h-1}(u), so a level of ALL nodes is 2E coalesced ORs of N-bit rows
 * of the previous level's table (no per-edge bitmap lookups, no atomics after level 1, no level barriers);
 * ring_h = ball_h & ~ball_{h-1}, then the same prefix-popcount CDF.  Outputs are bit-identical to
 * hsd_ring_signature_degree (sig / ring_sizes / ring_bitmaps / status, sig_peers as in the _allgather entry,
 * nullable).  Intermediate levels are computed for all n_nodes nodes whatever n_src is, and the cost is
 * O(E N / 32) per level whatever the ball sizes: the host picks this variant when most nodes are sources
 * and the workspace fits.  workspace: hsd_ring_dense_workspace_words(n_nodes) uint32 words (two N x N-bit
 * tables + a node -> output-row map), 16-byte aligned, caller-owned; nnz = rowptr[n_nodes]; hops >= 1;
 * src_nodes must be DISTINCT (the fused level kernel emits one output row per node). */
int64_t hsd_ring_dense_workspace_words(int32_t n_nodes);
int hsd_ring_signature_degree_dense(const int32_t* rowptr, const int32_t* col, int32_t n_nodes,
                                    const int32_t* src_nodes, const int32_t* out_rows, int32_t n_src,
                                    int32_t hops, const int32_t* bin_end, const float* delta, int32_t n_bins,
                                    float* sig, int64_t sig_ld, float* const* sig_peers, int32_t n_peers,
                                    int32_t* ring_sizes, uint32_t* ring_bitmaps, int32_t empty_as_zero,
                                    int32_t* status, uint32_t* workspace, int64_t workspace_words, int64_t nnz,
                                    void* stream);

/* Dense variant across several GPUs, split by bitmap COLUMNS: the OR recursion is independent per bitmap word,
 * so rank r runs every level for ALL nodes on its own range of 16-byte bitmap pieces [word4_begin, word4_end)
 * with no exchange (1/W of the work and of the table memory) and emits the PARTIAL integer prefix counts of
 * that range: counts[s][(h-1)(n_bins-1) + b] = members of ring_h(s) in the range with id < bin_end[b],
 * counts[s][hops (n_bins-1) + h-1] = members of ring_h(s) in the range (s = degree-order id; ld_c >=
 * hops (n_bins-1) + hops).  The caller sums `counts` over the ranks (one integer all-reduce: exact and
 * order-free) and hsd_ring_signature_from_counts turns the sums into the same signature rows / ring sizes /
 * status as the other variants, bit for bit.  workspace: hsd_ring_cols_workspace_words(...) uint32 words. */
int64_t hsd_ring_cols_workspace_words(int32_t n_nodes, int32_t word4_begin, int32_t word4_end);
int hsd_ring_counts_dense_cols(const int32_t* rowptr, const int32_t* col, int32_t n_nodes, int64_t nnz,
                               int32_t hops, const int32_t* bin_end, int32_t n_bins,
                               int32_t word4_begin, int32_t word4_end, int32_t* counts, int64_t ld_c,
                               uint32_t* workspace, int64_t workspace_words, void* stream);
int hsd_ring_signature_from_counts(const int32_t* rowptr, const int32_t* counts, int64_t ld_c,
                                   const int32_t* src_nodes, const int32_t* out_rows, int32_t n_src,
                                   int32_t hops, const float* delta, int32_t n_bins, float* sig, int64_t sig_ld,
                                   int32_t* ring_sizes, int32_t empty_as_zero, int32_t* status, void* stream);

/* Graphs above ~400k nodes: the four N-bit bitmaps of a source no longer fit shared memory.  The
 * BFS entry points then use a caller-owned DEVICE workspace of hsd_bfs_workspace_words(n_nodes)
 * uint32 words (0 = not needed), registered per host thread with hsd_bfs_set_workspace (NULL
 * unregisters); CTAs become persistent and keep their bitmaps in an L2-resident slice of it. */
int64_t hsd_bfs_workspace_words(int32_t n_nodes);
int hsd_bfs_set_workspace(uint32_t* workspace, int64_t words);

/* Rings only (tools/hierarchy.py:25-38, model/HSD.py:87-94 ring sizes). */
int hsd_bfs_rings(const int32_t* rowptr, const int32_t* col, int32_t n_nodes,
                  const int32_t* src_nodes, const int32_t* out_rows, int32_t n_src,
                  int32_t hops,
                  int32_t* ring_sizes, uint32_t* ring_bitmaps, void* stream);

/* ---- layout: row-major signatures -> K-major table for the pairwise kernel --
 * sig[.][sig_ld] (first k_used columns) -> sigT[k_pad][n_pad]: output column
 * col0 + r (r < n_rows) is table row r, or table row src_rows[r] when src_rows is
 * given (the multi-GPU plan deals BFS sources round-robin to ranks for balance, so
 * the gathered table is in dealt order).  Rows k_used..k_pad-1 and columns beyond
 * the data must be zero (caller memsets sigT once). */
int hsd_signature_transpose(const float* sig, int64_t sig_ld, int32_t n_rows, int32_t k_used,
                            float* sigT, int64_t n_pad, int32_t col0, const int32_t* src_rows,
                            void* stream);

/* ---- incremental update: scatter recomputed rows into the symmetric matrix ----
 * DynamicHSD (model/dynamic_HSD.py:23-24 is a stub; BASELINE config 5): blk[a][c], a < m, c < n, holds
 * the recomputed distances of row idx[a] (int64 node ids, ascending) to every column.  Stores
 * D[idx[a]][c] = blk[a][c] and, when mirror != 0, D[c][idx[a]] = blk[a][c] (D row-major, leading
 * dimension d_ld; needs n rows when mirrored).  Replaces two torch index_put passes over the block. */
int hsd_scatter_symmetric(const float* blk, int64_t blk_ld, int32_t m, int32_t n, const int64_t* idx,
                          float* D, int64_t d_ld, int32_t mirror, void* stream);

/* ---- K3: pairwise L1 over the K-major signature table ----------------------
 * Replaces the O(N^2 (H+1)) scipy loop model/HSD.py:103-112 (and :144-159).
 *   out[(i-row0)*ld_out + (j-col0)] = sum_k |sigT[k][i] - sigT[k][j]|
 * for i in [row0,row0+n_rows), j in [col0,col0+n_cols).
 * symmetric != 0 requires row0 == col0 and n_cols >= n_rows (a square, or the
 * trapezoid "rows of a panel x every column from the panel's first row on"); only
 * tiles on or above the diagonal are computed and each is also stored mirrored at
 * out[(j-row0)*ld_out + (i-col0)] (so `out` must have n_cols rows), the way the
 * reference fills dist_mat[i,j] = dist_mat[j,i] (model/HSD.py:112).  Panels of
 * rows processed in order therefore complete the matrix top to bottom, which is
 * what lets the host pipeline stream finished rows out while later panels compute.
 * sigT: float[k_pad][n_pad] with k_pad = k_used rounded up to HSD_PAIR_KCHUNK (rows
 * k_used..k_pad-1 must be zero),
 * n_pad % 4 == 0, base 16-byte aligned; row0 % 4 == 0 and col0 % 4 == 0 (TMA tile origins must be
 * 16-byte aligned). Tiles are staged by TMA (cp.async.bulk.tensor.2d). */
int hsd_pairwise_l1(const float* sigT, int32_t k_used, int64_t n_pad,
                    int32_t row0, int32_t n_rows, int32_t col0, int32_t n_cols,
                    int32_t symmetric, float* out, int64_t ld_out, void* stream);

/* ---- K3 over several GPUs: symmetric tiles, mirrored through peer memory ------
 * The logical N x N matrix is row-block sharded: block r = float[rows_per_rank][ld_out]
 * in GPU r's memory, shard_ptrs[r] (a DEVICE array of `world` pointers) its base as
 * mapped into THIS process (own allocation for r == rank, NVLink peer mapping
 * otherwise).  Rank `rank` computes upper-triangle tiles rank, rank+world, ... of the
 * whole matrix and stores each tile to the owner of its rows AND, mirrored, to the
 * owner of its columns with plain st.global on the peer pointers — so no tile is
 * computed twice anywhere in the job and the N(N-1)/2 pairs cost the same FADDs on
 * G GPUs as on one.  Block r is complete once every rank's launch has finished
 * (the caller issues one barrier).  The reference mirrors dist_mat[i,j] = dist_mat[j,i]
 * the same way (model/HSD.py:112). */
int hsd_pairwise_l1_sharded(const float* sigT, int32_t k_used, int64_t n_pad, int32_t n_nodes,
                            int32_t rank, int32_t world, int32_t rows_per_rank,
                            float* const* shard_ptrs, int64_t ld_out, void* stream);

/* The same kernels driven by an explicit tile list (round 2): tile_list int32[n_tiles][3] = {first row, first
 * column, mirror flag} of 128 x tile_n tiles (tile_n = 128 or 64; rows / columns are node ids, multiples of
 * 128 / tile_n).  A listed tile is stored to the owner of its rows and, when the flag is set, mirrored to the
 * owner of its columns.  The host deals the upper-triangle tiles so that every tile is computed by the owner
 * of its ROW block or of its COLUMN block, oriented so that the mirrored (short-run) store is the local one
 * and only the direct (long-run) store crosses NVLink: half the peer traffic of hsd_pairwise_l1_sharded's
 * round-robin dealing, none of it in 32-byte pieces (hsd_b200/sharded.py::symmetric_tile_list). */
int hsd_pairwise_l1_tile_list(const float* sigT, int32_t k_used, int64_t n_pad, int32_t n_nodes,
                              const int32_t* tile_list, int32_t n_tiles, int32_t tile_n,
                              int32_t rows_per_rank, float* const* shard_ptrs, int64_t ld_out, void* stream);

/* ---- K2 (value mode): ring gather + sort ----------------------------------
 * Replaces model/HSD.py:71-83 (get_hierarchical_coeffcients) plus the argsort
 * inside scipy's _cdf_distance.  For each (row r, hop h) gathers
 * psi[r*psi_ld + orig_of[j]] for every j set in ring_bitmaps[r][h] and writes
 * them ascending at vals[offsets[r*(hops+1)+h] ...].  offsets = exclusive scan
 * of ring_sizes (int64).  psi row r must be the wavelet row of the source that
 * wrote out_row r.  orig_of may be NULL (bitmaps already in psi's column order).
 * max_ring_size (host-known, from ring_sizes) sizes the in-shared-memory bitonic
 * sort; rings above 16384 members return HSD_ERR_UNSUPPORTED. */
int hsd_ring_signature_values(const double* psi, int64_t psi_ld,
                              const uint32_t* ring_bitmaps, const int32_t* ring_sizes,
                              const int64_t* offsets, const int32_t* orig_of,
                              int32_t n_rows, int32_t hops, int32_t n_nodes,
                              int32_t max_ring_size, double* vals, void* stream);

/* ---- K3 (value mode): exact ragged W1 by two-pointer merge, FP64 ------------
 * Replaces scipy.stats.wasserstein_distance as called at model/HSD.py:111 on
 * ragged multisets:  out[i*ld+j] = out[j*ld+i] = sum_h W1(vals_i_h, vals_j_h),
 * h in [hop_begin, hop_end).  Rows i in [row0,row0+n_rows) against all j > i
 * (j < n_total); diagonal written as 0. An empty ring sets *status |= 1. */
int hsd_pairwise_w1_merge(const double* vals, const int64_t* offsets, const int32_t* ring_sizes,
                          int32_t n_total, int32_t hops, int32_t hop_begin, int32_t hop_end,
                          int32_t row0, int32_t n_rows,
                          double* out, int64_t ld_out, int32_t* status, void* stream);

/* ---- K3 (aligned mode, tools/metrics.py:18-36,151-192) ----------------------
 * The reference's second distance path pads the shorter multiset with zeros,
 * sorts, and calls scipy on equal-length arrays, i.e.
 *   d = (1/L) * sum_k |p_desc[k] - q_desc[k]|,  L = max(n_p, n_q), 0 when both empty.
 * Same ragged ascending `vals` as above. metric: 0 = 'wasserstein', 1 = 'hellinger'
 * (tools/metrics.py:117-138 on the same aligned ascending arrays), 2 = 'wasserstein_guass'
 * (tools/metrics.py:54-71: (u1-u2)^2 + s1 + s2 - 2 sqrt(s1 s2) of the padded arrays). */
int hsd_pairwise_aligned(const double* vals, const int64_t* offsets, const int32_t* ring_sizes,
                         int32_t n_total, int32_t hops, int32_t hop_begin, int32_t hop_end,
                         int32_t metric, int32_t row0, int32_t n_rows,
                         double* out, int64_t ld_out, void* stream);

/* ---- K3 (row worker exactly as written, model/HSD.py:140-161) ---------------
 * out[i*ld + j] = sum_{h < hop_end} aligned(Psi[i, ring_h(i)], Psi[i, ring_h(j)]) for
 * j > i, 0 for j <= i; BOTH signals come from wavelet row i (the reference indexes q
 * with startIndex, :155) and hops run 0..hop-1 (:148).  Inputs per row i:
 *   sorted_vals[i][t]  t-th smallest value of Psi[i, :]   (double[n][n])
 *   order[i][t]        the node holding it                 (int32[n][n])
 * ring bitmaps/sizes rows are original indices; bit_of maps original index -> bit id
 * (NULL: identity). metric as in hsd_pairwise_aligned. */
int hsd_pairwise_worker(const double* sorted_vals, const int32_t* order,
                        const uint32_t* ring_bitmaps, const int32_t* ring_sizes,
                        const int32_t* bit_of, int32_t n_nodes, int32_t hops, int32_t hop_end,
                        int32_t metric, int32_t row0, int32_t n_rows,
                        double* out, int64_t ld_out, void* stream);

/* ---- K4: Chebyshev heat-kernel wavelets as CSR SpMM -------------------------
 * Replaces pygsp cheby_op as driven one impulse at a time by model/HSD.py:50-59
 * (and model/GraphWave.py:31-39).  Computes, for a block of n_cols impulse
 * columns [col0, col0+n_cols) and n_scales coefficient sets,
 *   R_s = 1/2 c_{s,0} T_0 + sum_{k=1..order} c_{s,k} T_k,
 *   T_0 = E, T_1 = (L E - a E)/a, T_k = (2/a)(L - a I) T_{k-1} - T_{k-2},  a = lmax/2,
 * with L = D - A taken from the CSR (original node order, unit weights), then
 * the reference threshold x > thr ? x : 0 (model/HSD.py:65).
 *   coeff_host  HOST double[n_scales][order+1] (copied into the launch arguments)
 *   n_cols   even (columns are processed in 16-byte pairs); col0 + n_cols may exceed n_nodes by one
 *            (an all-zero impulse column) so an odd node count can be padded
 *   work     double[3][n_nodes][n_cols]   (T ring buffer)
 *   out      double[n_scales][n_nodes][n_cols]; out[s][v][c] = Psi_s[col0+c][v] (= Psi_s[v][col0+c], symmetric)
 */
int hsd_cheb_spmm(const int32_t* rowptr, const int32_t* col, int32_t n_nodes,
                  double lmax, const double* coeff_host, int32_t n_scales, int32_t order,
                  int32_t col0, int32_t n_cols, double threshold,
                  double* work, double* out, void* stream);

/* ---- exact heat-kernel wavelets from an eigendecomposition, threshold fused ------
 * Replaces model/HSD.py:61-66 / model/GraphWave.py:42-49 (two dense np.dot + np.vectorize):
 *   out[i][j] = sum_k U[i][k] exp(-scale lam[k]) U[j][k], then (apply_threshold != 0)
 *   out = out > threshold ? out : 0.  U double[n][ldu] holds the eigenvectors as COLUMNS (what
 * numpy / torch eigh return), lam double[n].  One FP64 kernel; only tiles on or above the diagonal
 * are computed and each is stored mirrored, so out is exactly symmetric and the un-thresholded
 * product is never materialised.  (The eigendecomposition stays on the vendor solver.) */
int hsd_exact_wavelets(const double* U, int64_t ldu, const double* lam, int32_t n_nodes,
                       double scale, double threshold, int32_t apply_threshold, double* out,
                       int64_t ld_out, void* stream);

/* y = L x, L = D - A from the CSR (unit weights, self-loops cancel), one FP64 vector.  The
 * building block of the lmax estimate that replaces pygsp's Graph.estimate_lmax (ARPACK;
 * call sites model/HSD.py:51, model/multiscale_HSD.py:28) with a power iteration on the device. */
int hsd_laplacian_spmv(const int32_t* rowptr, const int32_t* col, int32_t n_nodes,
                       const double* x, double* y, void* stream);

/* ---- K5: ring gather-reduce for MultiHSD embeddings -------------------------
 * Replaces model/multiscale_HSD.py:45-61 (get_triple) / :64-73 (get_layer_sum):
 * emb[col0+c][s][h][0..1] = [sum, mean] of psiT[s][v][c] over v in ring_h(col0+c);
 * empty ring -> [0, 0].  psiT is the output layout of hsd_cheb_spmm
 * (double[n_scales][n_nodes][n_cols]).  ring_bitmaps / ring_sizes rows are
 * indexed by the source's ORIGINAL index; bitmap bits are original ids when
 * orig_of == NULL, degree-order ids (mapped through orig_of) otherwise.
 *   emb      double[n_nodes][n_scales][hops+1][2]; rows col0..col0+n_cols-1 are overwritten
 *   scratch  double[scratch_elems] workspace, >= n_cols*n_scales*(hops+1); more lets the node
 *            range be split over more CTAs (partial sums are combined in a fixed order, so
 *            the result is deterministic).  hops <= 7. */
int hsd_ring_reduce(const double* psiT, int32_t n_scales, int32_t n_nodes, int32_t n_cols,
                    const uint32_t* ring_bitmaps, const int32_t* ring_sizes,
                    const int32_t* orig_of, int32_t hops, int32_t col0, double* emb,
                    double* scratch, int64_t scratch_elems, void* stream);

/* ---- K6: GraphWave characteristic-function embedding --------------------------
 * Replaces model/GraphWave.py:53-69: out[i][2k], out[i][2k+1] = Re, Im of
 * mean_j exp(i * sample_points[k] * psi[i][j]), j < n_cols.  FP64, deterministic.
 *   psi double[n_rows][psi_ld], sample_points double[n_points] (device), out double[n_rows][2*n_points] */
int hsd_characteristic_function(const double* psi, int64_t psi_ld, int32_t n_rows, int32_t n_cols,
                                const double* sample_points, int32_t n_points, double* out, void* stream);

/* ---- K7: k nearest neighbours per row of the distance matrix -------------------
 * The consumer right after the path: the reference passes the N x N ndarray to sklearn's
 * precomputed-metric KNN (tools/evaluate.py:61-69, called from main.py:29).  Here the
 * selection runs on the device-resident (possibly row-sharded) matrix: for row r the k
 * smallest D[r][j], j != self_col0 + r, j allowed by col_mask (nullable bitmap over columns;
 * lets a caller restrict neighbours to a training fold), ordered by (distance, column).
 *   idx_out int32[n_rows][k] (-1 where fewer than k candidates), val_out float[n_rows][k]; 1 <= k <= 64.
 * Distances must be >= 0 (rows with a huge class of exactly tied candidates are resolved by a radix
 * select on the float bit pattern, whose unsigned order equals the numeric order only for >= 0). */
int hsd_topk_rows(const float* D, int64_t ld, int32_t n_rows, int32_t n_cols, int32_t k,
                  int32_t self_col0, const uint32_t* col_mask, int32_t* idx_out, float* val_out,
                  void* stream);

/* K7 without the matrix: the k-NN lists of all N nodes are built from row panels of the distance
 * matrix, one panel at a time (hsd_b200/engine.py::degree_knn), so only N x k results and one panel
 * ever occupy the device.  Running lists idx_io int32[..][k] / val_io float[..][k] start as -1 / +inf;
 * every list is sorted by (distance, node id) and padded with -1 / +inf, like hsd_topk_rows writes
 * them.  Because that order is total, merging the top-k lists of disjoint candidate sets gives exactly
 * the top-k of their union: the result equals hsd_topk_rows on the whole matrix bit for bit.
 * 1 <= k <= 64, distances >= 0; no atomics, so results do not depend on the schedule.
 *
 * hsd_topk_merge: for rows r < n_rows, merges n_lists (1..64) candidate lists
 *   idx_in / val_in [l * list_stride + r * k + t]   (l < n_lists; list_stride >= n_rows * k when n_lists > 1)
 * into the running lists idx_io / val_io [r * k + t] in place; idx_offset is added to every candidate
 * id that is not -1 (a panel's hsd_topk_rows ids are block columns).  Each candidate must be absent
 * from the running list and from the other candidate lists (disjoint column sets).
 *
 * hsd_topk_merge_cols: the column pass of a panel.  blk float[n_rows][ld] (ld >= n_cols) is a block
 * whose row r is node row_node0 + r and whose column c is node col_node0 + c; for every column
 * c in [c_begin, n_cols) the candidates (blk[r][c], row_node0 + r), r < n_rows, are merged into the
 * running list of node col_node0 + c, stored at idx_io / val_io [(col_node0 + c) * k + t].  The
 * caller keeps the self pair out (c_begin past the block's diagonal). */
int hsd_topk_merge(const int32_t* idx_in, const float* val_in, int32_t n_lists, int64_t list_stride,
                   int32_t idx_offset, int32_t n_rows, int32_t k, int32_t* idx_io, float* val_io,
                   void* stream);
int hsd_topk_merge_cols(const float* blk, int64_t ld, int32_t n_rows, int32_t c_begin, int32_t n_cols,
                        int32_t row_node0, int32_t col_node0, int32_t k, int32_t* idx_io, float* val_io,
                        void* stream);

/* K7 radius graph: every pair (i, j), i != j, with D[i][j] <= radius, as a symmetric CSR graph built from
 * the same row panels (hsd_b200/engine.py::degree_radius), so the N x N matrix never has to exist.
 * blk is a panel of float (elem_bytes 4) or double (elem_bytes 8) values [n_rows][ld], ld >= n_cols:
 * block row r is node r0 + r, block column c is node r0 + c, and only its upper part (c > r) is read —
 * it holds every pair the panel owns once.  hits uint32[n_rows][hits_ld], hits_ld >= ceil(n_cols / 32),
 * is the hit bitmap (bit c % 32 of word [r][c / 32]: blk[r][c] <= radius, c > r); radius >= 0, not NaN,
 * +inf allowed.  The compare is (double)blk[r][c] <= radius; for float blocks it is done as
 * blk[r][c] <= the largest float not above radius.  No atomics decide a position: results do not depend
 * on the schedule.
 *
 * hsd_radius_count: writes hits (words holding a column c > r), row_cnt int32[n_rows] (hits of row r) and
 *   col_cnt int32[n_cols][n_chunks] (hits of column c over the rows r < c of chunk q, rows
 *   [q * HSD_RADIUS_CHUNK_ROWS, (q + 1) * HSD_RADIUS_CHUNK_ROWS), n_chunks = ceil(n_rows / HSD_RADIUS_CHUNK_ROWS));
 *   both counts are zeroed first.
 * hsd_radius_emit_rows: row r's hits in ascending c, (col_node0 + c, blk[r][c]), at idx_out / val_out
 *   [row_off[r] ..], row_off int64 the exclusive scan of row_cnt.
 * hsd_radius_emit_cols: column c's hits in ascending r, (row_node0 + r, blk[r][c]), at idx_out / val_out
 *   [col_off[c][0] ..], col_off int64[n_cols][n_chunks] the exclusive scan of col_cnt in that (row-major) order.
 * hsd_radius_scatter: assembly of the CSR.  Segment s < n_seg is node node0 + s's piece
 *   idx / val [off[s], off[s + 1]) (off int64[n_seg + 1], e.g. a row_off or col_off with its total
 *   appended); it is copied to idx_out / val_out at indptr[node] + cursor[node], and cursor[node] grows by
 *   its length.  Called per piece in panel order, column piece before row piece, every output row comes
 *   out ascending.
 * hsd_radius_merge_parts: the partial CSRs of a sweep split over ranks (each rank's panels give every row
 *   some of its entries) merged into one CSR.  Part p < n_parts (1..64) has its own offsets
 *   part_indptr[p * (n_rows + 1) + i] and its entries at idx / val [part_base[p] + part_indptr[p][i] ..
 *   part_base[p] + part_indptr[p][i + 1]), ascending by id within a row.  indptr int64[n_rows + 1] is the
 *   caller's scan of the summed row lengths.  Row i of idx_out / val_out [indptr[i] .. indptr[i + 1]) is the
 *   stable merge by id of row i of every part; equal ids (absent when the parts are disjoint) are ordered by
 *   part index, so the result never depends on the schedule.  Nothing outside [indptr[0], indptr[n_rows])
 *   is written; the values (elem_bytes 4 or 8) are copied bit for bit. */
#define HSD_RADIUS_CHUNK_ROWS 512
int hsd_radius_count(const void* blk, int32_t elem_bytes, int64_t ld, int32_t n_rows, int32_t n_cols,
                     double radius, uint32_t* hits, int64_t hits_ld, int32_t* row_cnt, int32_t* col_cnt,
                     void* stream);
int hsd_radius_emit_rows(const void* blk, int32_t elem_bytes, int64_t ld, int32_t n_rows, int32_t n_cols,
                         const uint32_t* hits, int64_t hits_ld, const int64_t* row_off, int32_t col_node0,
                         int32_t* idx_out, void* val_out, void* stream);
int hsd_radius_emit_cols(const void* blk, int32_t elem_bytes, int64_t ld, int32_t n_rows, int32_t n_cols,
                         const uint32_t* hits, int64_t hits_ld, const int64_t* col_off, int32_t row_node0,
                         int32_t* idx_out, void* val_out, void* stream);
int hsd_radius_scatter(const int32_t* idx, const void* val, int32_t elem_bytes, const int64_t* off,
                       int32_t n_seg, int32_t node0, const int64_t* indptr, int64_t* cursor,
                       int32_t* idx_out, void* val_out, void* stream);
int hsd_radius_merge_parts(int32_t n_parts, int32_t n_rows, const int64_t* part_indptr, const int64_t* part_base,
                           const int32_t* idx, const void* val, int32_t elem_bytes, const int64_t* indptr,
                           int32_t* idx_out, void* val_out, void* stream);

/* K7 minimum spanning tree: the MST of the complete graph under the distance, by Borůvka rounds over the
 * same row panels (hsd_b200/engine.py::degree_mst), so the N x N matrix never has to exist.  Edges are
 * ordered by E(u, v) = (D[u][v], min(u, v), max(u, v)); for a fixed node i that is the order of (D[i][j], j),
 * so node i's best edge leaving its component is the minimum of the int64 key
 * K(d, j) = float_bits(d) << 32 | j (distances finite and >= 0); INT64_MAX stands for "no edge".  comp
 * int32[N] labels the components.  Keys are minima: results do not depend on the schedule.
 *
 * hsd_mst_panel_min: blk float[n_rows][ld] (n_rows <= n_cols <= ld) is a panel whose row r is node
 *   node0 + r and whose column c is node node0 + c; only its upper part (c > r) is read.  For every element
 *   with comp[a] != comp[b] (a = node0 + r, b = node0 + c) key_io[a] is lowered to K(blk[r][c], b) and
 *   key_io[b] to K(blk[r][c], a); smaller keys already there are kept.
 * hsd_mst_list_candidates: idx / val [n][k] (1 <= k <= 64) are k-NN lists ordered by (distance, id) and
 *   padded with -1 / +inf (degree_knn's).  key_out[i] = K of the first entry of node i's list outside its
 *   component, and bound_out[i] = +inf; when there is none, key_out[i] = INT64_MAX and bound_out[i] is the
 *   distance of the k-th entry (every edge of i leaving its component is at least that long), or +inf when
 *   the list is short (it holds every other node).
 * hsd_single_linkage_host (HOST pointers, no CUDA): the n - 1 MST edges (u[t], v[t], dist[t]) in
 *   non-decreasing dist -> Z double[n - 1][4] in scipy's linkage format: row t merges the clusters holding
 *   u[t] and v[t], ids Z[t][0] < Z[t][1] (ids below n are nodes, n + s is the cluster row s formed), at height
 *   dist[t], into a cluster of Z[t][3] nodes.  Edges that are not distinct nodes in 0..n-1, heights that are
 *   not finite, negative or decreasing, and an edge that closes a cycle are rejected. */
int hsd_mst_panel_min(const float* blk, int64_t ld, int32_t n_rows, int32_t n_cols, int32_t node0,
                      const int32_t* comp, int64_t* key_io, void* stream);
int hsd_mst_list_candidates(const int32_t* idx, const float* val, int32_t n, int32_t k, const int32_t* comp,
                            int64_t* key_out, float* bound_out, void* stream);
int hsd_single_linkage_host(const int32_t* u, const int32_t* v, const float* dist, int32_t n, double* Z);

/* K7b mutual-reachability minimum spanning tree (HDBSCAN; hsd_b200/engine.py::degree_mreach_mst): the MST above
 * under d_mr(a, b) = max(core[a], core[b], D[a][b]), core float[N] finite and >= 0 (node i's core distance), so
 * d_mr is one of its operands and keys are K(d_mr, j).
 *
 * hsd_mst_panel_min_mreach: hsd_mst_panel_min with the compared value max(blk[r][c], core[a], core[b]).
 * hsd_mst_list_candidates_mreach: the lists are ordered by D, not by d_mr.  key_out[i] = the minimum of
 *   K(max(core[i], core[j], val[i][t]), j) over the entries j of node i's list outside its component
 *   (INT64_MAX when there is none).  bound_out[i] = +inf when that key is exact: the list is short (it holds
 *   every other node) or the key's distance is strictly below val[i][k-1] (an unlisted j has
 *   d_mr(i, j) >= D[i][j] >= val[i][k-1]); else bound_out[i] = val[i][k-1], a lower bound of every unlisted
 *   edge of i.
 * hsd_hdbscan_host (HOST pointers, no CUDA): Z double[n - 1][4], hsd_single_linkage_host's linkage of the
 *   mutual-reachability MST -> labels int64[n] (-1: noise) and probabilities double[n], what scikit-learn's
 *   HDBSCAN tree_to_labels(Z, min_cluster_size, method, allow_single_cluster, 0.0, None) returns, with the
 *   same float64 operations in the same order.  method 0 = "eom", 1 = "leaf"; n >= 2, min_cluster_size >= 2. */
int hsd_mst_panel_min_mreach(const float* blk, int64_t ld, int32_t n_rows, int32_t n_cols, int32_t node0,
                             const int32_t* comp, const float* core, int64_t* key_io, void* stream);
int hsd_mst_list_candidates_mreach(const int32_t* idx, const float* val, int32_t n, int32_t k, const int32_t* comp,
                                   const float* core, int64_t* key_out, float* bound_out, void* stream);
int hsd_hdbscan_host(const double* Z, int32_t n, int32_t min_cluster_size, int32_t method,
                     int32_t allow_single_cluster, int64_t* labels, double* probabilities);

/* ---- e2e path: ship each unordered pair once, mirror on the host --------------------
 * The reference returns the dense symmetric ndarray (model/HSD.py:100-114, dist_mat[i,j] =
 * dist_mat[j,i]).  Over PCIe the matrix is the e2e bottleneck, so the host pipeline copies only
 * the upper trapezoid of every finished row panel (hsd_copy2d_to_host: one cudaMemcpy2DAsync,
 * rows x width_bytes window, both pitches in bytes; dst_host should be pinned) and the host cores
 * fill the rows below it: hsd_mirror_upper_to_lower_host sets D[j][i] = D[i][j] for
 * row_begin <= i < row_end, i < j < n (HOST pointers; row_begin a multiple of 64; blocked
 * transposes on n_threads threads, AVX2 + streaming stores when the CPU has them). */
int hsd_copy2d_to_host(void* dst_host, int64_t dst_pitch_bytes, const void* src_dev, int64_t src_pitch_bytes,
                       int64_t width_bytes, int64_t rows, void* stream);
int hsd_mirror_upper_to_lower_host(float* D_host, int64_t ld, int32_t n, int32_t row_begin,
                                   int32_t row_end, int32_t n_threads);

/* ---- measurement helper: FP32 CUDA-core issue peak ---------------------------
 * Runs a register-only FADD kernel (same sub + |.|-accumulate instruction mix as
 * the pairwise inner loop, no memory) and returns lane-ops in *lane_ops; the
 * caller times it with events on `stream`.  Used by bench.py for the live
 * roofline denominator. */
int hsd_fp32_peak_probe(float* sink, int32_t iters, int64_t* lane_ops_host, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* HSD_B200_H */
