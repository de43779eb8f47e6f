/* nabo_b200 - C ABI of the B200-native nabo cell-projection hot path.
 *
 * Drop-in boundary (SURVEY.md 8b).  The reference (parashardhapola/nabo 0.4.1) has
 * no FFI: its hot path is five module-level Python operators called by
 * Dataset / Mapping / Graph.  Each entry point below replaces one of them and is
 * what a ctypes binding inside the reference would call (see INTEGRATION.md).
 * File:line citations are relative to the reference checkout.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless its name ends in _host;
 *   - the caller owns every buffer, including workspace (query the size first);
 *   - every call is asynchronous on `stream` (a cudaStream_t, passed as void*);
 *   - return value: 0 = OK, <0 = invalid argument (NABO_E*), >0 = cudaError_t;
 *     nabo_last_error() returns a thread-local message.  No exceptions, no global
 *     state, no host fallback: without a CUDA device every compute call fails.
 *   - matrices are row-major; `ld*` is the row stride in elements.
 *   - neighbour order everywhere: ascending distance, ties by ascending index,
 *     NaN distances and masked reference cells last (numpy.ma.argsort semantics of
 *     nabo/_mapping.py:135-146; the reference's own tie order is unspecified).
 */
#ifndef NABO_B200_H
#define NABO_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NABO_ABI_VERSION 1

#define NABO_EINVAL (-1)      /* bad argument                                  */
#define NABO_EWORKSPACE (-2)  /* workspace missing or too small                */
#define NABO_EUNSUPPORTED (-3)/* shape outside what the kernels are built for  */

/* metric ids.  Reference dispatch: euclidean when the query set IS the reference
 * (intra_ref), modified Canberra otherwise (nabo/_mapping.py:119-124, 433-440).
 * Cosine and query!=reference Euclidean are extensions (BASELINE.json). */
#define NABO_EUCLIDEAN 0
#define NABO_MOD_CANBERRA 1
#define NABO_COSINE 2

/* kNN engines */
#define NABO_MODE_EXACT 0 /* FP64 brute force in the reference's arithmetic order */
#define NABO_MODE_FAST 1  /* tensor-core / FP32 candidate pass + exact FP64 re-rank
                             + certificate, exact fallback for uncertified rows   */

int nabo_abi_version(void);
const char* nabo_last_error(void);
/* 0 when a compute-capability 10.x device is current; fills sm count if non-NULL. */
int nabo_device_check(int* sm_count);

/* ---- (1) full distance tiles: replace the two numba kernels -------------------
 * _euclidean_dist(x, y, d)            nabo/_mapping.py:16-26
 * _mod_canberra_dist(x, y, d, f)      nabo/_mapping.py:29-45
 * Caller allocates d (m x n, row stride ldd); filled in place; bit-identical to
 * the numba kernels (sequential ascending-k FP64, no FMA contraction). */
int nabo_euclidean_dist(const double* x, int ldx, const double* y, int ldy, double* d, int ldd,
                        int m, int n, int g, void* stream);
int nabo_mod_canberra_dist(const double* x, int ldx, const double* y, int ldy, double* d, int ldd,
                           int m, int n, int g, double f, void* stream);
int nabo_cosine_dist(const double* x, int ldx, const double* y, int ldy, double* d, int ldd,
                     int m, int n, int g, void* stream);

/* ---- (2) fused distance + per-query top-k: replaces _calc_dist ------------------
 * nabo/_mapping.py:48-148, restricted to what _calc_snn consumes ([:k] of every
 * sorted row, :190/:193): the N x M matrix is never written.
 *   q (n_query x g), r (n_ref x g)  FP64 PCA coordinates (first use_comps columns)
 *   ref_mask   n_ref bytes, non-zero = ignore_ref_cells member (sorts last) or NULL
 *   drop_first non-zero = reference<->reference rows: drop the first sorted
 *              element ("self", :141-142) and return the next k
 *   idx_offset added to every output index (reference-sharded mode)
 *   out_idx (n_query x k) int32, out_dist (n_query x k) FP64 (NaN for masked /
 *   missing entries, idx -1 when fewer than k references exist)
 *   stats_host optional int64[8], filled only if non-NULL (forces a stream sync at the
 *              end of the call): [0] rows re-ranked, [1] rows sent to the exact
 *              brute-force engine, [2] candidates kept per row, [3] kernels launched,
 *              [4] ns spent in the dominant distance/top-k kernel (CUDA events on
 *              `stream`), [5] ns in the exact re-rank, [6] ns in the exact fallback,
 *              [7] ns in operand preparation.
 *   mode = NABO_MODE_FAST runs the candidate pass + re-rank where a fast plan exists, and
 *   the exact engine (same results) elsewhere; ksel = k + drop_first:
 *     Euclidean / cosine  1 <= g <= 128, ksel <= 128 (tensor-core pass: 128-key buffers for
 *                         ksel + 8 <= 96, 256-key buffers for 89 <= ksel <= 128)
 *     modified Canberra   ksel + 8 <= 64; g <= 128 with dist_factor >= 1e-6 (bit-sliced
 *                         pass), g <= 77 otherwise (FP16 two-phase pass)
 */
size_t nabo_knn_workspace_bytes(int n_query, int n_ref, int g, int k, int metric, int mode);
int nabo_knn(const double* q, int ldq, const double* r, int ldr, int n_query, int n_ref, int g,
             int k, int metric, double dist_factor, const uint8_t* ref_mask, int drop_first,
             int idx_offset, int mode, int32_t* out_idx, double* out_dist, void* workspace,
             size_t workspace_bytes, int64_t* stats_host, void* stream);

/* Candidate pass alone (Euclidean / cosine): TMA-fed tcgen05 GEMM with a fused
 * per-query top-K' filter.  out_cand (n_query x K') LOCAL reference indices sorted by
 * candidate score (-1 = empty), K' = nabo_knn_candidates_width(k, drop_first);
 * out_tau (n_query) = score threshold every non-candidate is at or above (+inf = no
 * reference was rejected); optional out_qn2 (n_query) and out_scal (4 doubles: scale,
 * 1/scale, max scaled reference norm, cosine flag) are what the certificate uses.
 * Takes 1 <= g <= 128 and k + drop_first + 8 <= 96; NABO_EUNSUPPORTED otherwise.
 * nabo_knn(mode = NABO_MODE_FAST) = this + nabo_rerank_exact + certificate + fallback. */
int nabo_knn_candidates_width(int k, int drop_first);
size_t nabo_knn_candidates_workspace_bytes(int n_query, int n_ref, int g, int k, int drop_first);
int nabo_knn_candidates(const double* q, int ldq, const double* r, int ldr, int n_query, int n_ref,
                        int g, int k, int metric, const uint8_t* ref_mask, int drop_first,
                        int32_t* out_cand, float* out_tau, double* out_qn2, double* out_scal,
                        void* workspace, size_t workspace_bytes, void* stream);

/* Exact re-rank of caller-supplied candidates (cand: n_query x n_cand int32 LOCAL
 * reference indices, -1 = empty) in the reference's arithmetic; writes the best k. */
int nabo_rerank_exact(const double* q, int ldq, const double* r, int ldr, int n_query, int n_ref,
                      int g, int k, int metric, double dist_factor, const uint8_t* ref_mask,
                      int drop_first, int idx_offset, const int32_t* cand, int n_cand,
                      int32_t* out_idx, double* out_dist, void* stream);

/* ---- (3) candidate merge for the reference-sharded mode -------------------------
 * idx/dist: n_shards blocks of (n_query x k), shard-major (the layout an NCCL
 * all-gather produces); result = the k best per query by (dist, idx). */
int nabo_merge_topk(const int32_t* idx, const double* dist, int n_shards, int n_query, int k,
                    int32_t* out_idx, double* out_dist, void* stream);

/* The same merge with one (n_query x k) idx / dist block per shard at arbitrary device addresses
 * (host tables of n_shards <= 16 pointers): the per-source blocks of an all-to-all or peer-written
 * receive buffer are merged in place.  drop_first != 0 drops the first merged entry (the global
 * "self" of a reference-sharded self-kNN) and writes k - 1 columns. */
int nabo_merge_topk_parts(int n_shards, const int32_t* const* shard_idx_host,
                          const double* const* shard_dist_host, int n_query, int k, int drop_first,
                          int32_t* out_idx, double* out_dist, void* stream);

/* nabo_knn with ROUTED result rows (reference-sharded mode): row t goes to part p with
 * part_bounds_host[p] <= t < part_bounds_host[p+1] (n_parts + 1 ascending ints from 0 to n_query),
 * at row t - bounds[p] of part_idx_host[p] / part_dist_host[p] ((rows_p x k) blocks, n_parts <= 16).
 * The blocks may be slices of a local all-to-all send buffer or peer-GPU memory mapped over NVLink:
 * the re-rank kernel that produces a row delivers it. */
int nabo_knn_routed(const double* q, int ldq, const double* r, int ldr, int n_query, int n_ref, int g,
                    int k, int metric, double dist_factor, const uint8_t* ref_mask, int drop_first,
                    int idx_offset, int mode, int n_parts, const int* part_bounds_host,
                    int32_t* const* part_idx_host, double* const* part_dist_host, void* workspace,
                    size_t workspace_bytes, int64_t* stats_host, void* stream);

/* ---- (3b) prepared reference: pack a reference once, map any number of query batches ------
 * The reference-side operands of the fast engine - the packed FP16 tensor-core tiles and their scale
 * (Euclidean / cosine), or the FP32 copy, bin edges and bit planes of the sliced pass (modified Canberra) -
 * depend on (reference rows, g, metric, ref_mask) alone.  nabo_ref_prepare builds them once into a caller-owned
 * device buffer and fills a host descriptor; nabo_knn_prepared then maps query batches against it.  Every result
 * is bit-identical to nabo_knn / nabo_knn_routed on the same inputs (the exact re-rank, the certificate and the
 * exact fallback decide every row).  The descriptor keeps the caller's FP64 rows and mask by address (the re-rank
 * and the fallback read them): both, and the buffer, must stay allocated and unchanged while it is in use.
 *
 * The tensor-core scale of a prepared reference comes from the reference's largest norm alone (cosine: 32), not
 * from the queries: a query whose scaled coordinates would overflow FP16 (about 500x the largest reference norm)
 * is sent to the exact fallback and counted in stats_host[1].
 * Calls the prepared operands do not serve run the existing path on the stored rows: mode = NABO_MODE_EXACT, k
 * beyond the fast plans (the exact engine), and modified Canberra with dist_factor < 1e-6 (the FP16 two-phase pass);
 * nabo_knn_prepared_workspace_bytes then returns the one-shot size.
 * Status: a descriptor that was not filled by nabo_ref_prepare or does not match its buffer -> NABO_EINVAL; another
 * ABI version, a metric / g without a fast plan (1 <= g <= 128) or k + drop_first > 128 -> NABO_EUNSUPPORTED. */
#define NABO_PREPARED_MAGIC 0x5250424eu   /* "NBPR" */
#define NABO_PLAN_TC 1                     /* tensor-core operands (Euclidean, cosine)   */
#define NABO_PLAN_SLICED 2                 /* bit-sliced operands (modified Canberra)    */
typedef struct nabo_prepared_ref {
    uint32_t magic;            /* NABO_PREPARED_MAGIC                                        */
    int abi_version;           /* NABO_ABI_VERSION of the library that prepared it           */
    int n_ref, g, metric, plan;
    const double* r;           /* the caller's FP64 rows (n_ref x g, row stride ldr)         */
    int ldr;
    const uint8_t* ref_mask;   /* the caller's mask or NULL                                  */
    void* buffer;              /* the caller's buffer (nabo_ref_prepared_bytes)              */
    size_t buffer_bytes;
    const void* ops[3];        /* operand addresses inside buffer (tiles, scale / FP32 copy, planes, edges) */
} nabo_prepared_ref;

/* device bytes of the prepared operands; 0 when metric / g have no fast plan.  Tensor-core plan: 128-row tiles of
 * 2 * ceil16(3g + 3) bytes per row (320 B per row at g = 50) + 8 B per row. */
size_t nabo_ref_prepared_bytes(int n_ref, int g, int metric);
int nabo_ref_prepare(const double* r, int ldr, int n_ref, int g, int metric, const uint8_t* ref_mask, void* buffer,
                     size_t buffer_bytes, nabo_prepared_ref* prepared_host, void* stream);
/* per-call (query-side) workspace; smaller than nabo_knn_workspace_bytes by the reference's share.  0 for an
 * invalid descriptor. */
size_t nabo_knn_prepared_workspace_bytes(int n_query, const nabo_prepared_ref* prepared_host, int k,
                                         double dist_factor, int mode);
int nabo_knn_prepared(const double* q, int ldq, int n_query, const nabo_prepared_ref* prepared_host, int k,
                      double dist_factor, int drop_first, int idx_offset, int mode, int32_t* out_idx,
                      double* out_dist, void* workspace, size_t workspace_bytes, int64_t* stats_host, void* stream);
int nabo_knn_prepared_routed(const double* q, int ldq, int n_query, const nabo_prepared_ref* prepared_host, int k,
                             double dist_factor, int drop_first, int idx_offset, int mode, int n_parts,
                             const int* part_bounds_host, int32_t* const* part_idx_host,
                             double* const* part_dist_host, void* workspace, size_t workspace_bytes,
                             int64_t* stats_host, void* stream);

/* ---- (4) SNN neighbour weights: replaces _calc_snn ------------------------------
 * nabo/_mapping.py:151-200.  counts[t][j] = |set(tgt_knn[t]) & set(ref_knn[tgt_knn[t][j]])|
 * weights[t][j] = lut[counts] with lut[s] = round(s / (2(k-1) - s), 2) built on
 * the host with Python's round() (so weights are bit-exact); an edge exists iff
 * counts > 0 (:195).  Negative indices (missing neighbours) give count 0. */
int nabo_snn_weights(const int32_t* tgt_knn, int n_query, int k, const int32_t* ref_knn, int n_ref,
                     int k_ref, const double* lut, uint8_t* out_counts, double* out_weights,
                     void* stream);

/* ---- (5) per-reference mapping scores: replaces Graph.get_mapping_score core ----
 * nabo/_graph.py:643-653, 690-693.  Edges (t -> tgt_knn[t][j], weight) with
 * counts > 0 are sorted by (reference, target) with a stable LSD radix sort and
 * summed per reference cell IN TARGET ORDER (the reference's adjacency order), so
 * the result is deterministic and independent of scheduling.  include (n_query
 * bytes or NULL) selects the target subset; n_include is its size (the divisor). */
size_t nabo_scores_workspace_bytes(int n_query, int k, int n_ref);
int nabo_mapping_scores(const int32_t* tgt_knn, const uint8_t* counts, const double* lut,
                        int n_query, int k, int n_ref, const uint8_t* include, int n_include,
                        double min_weight, int weighted, double score_multiplier,
                        double min_score, double* out_scores, void* workspace,
                        size_t workspace_bytes, void* stream);

/* GPU-count-independent form of the same score (sharded modes; SURVEY.md section 7): the weight
 * table in INTEGER units (int_weights[c], 0 = no edge / filtered; for the reference's table
 * round(w, 2) * 100, exact) is accumulated per reference cell with integer atomics
 * (acc int64 (n_ref), caller-zeroed, summed over batches / all-reduced over GPUs as integers),
 * then score = score_multiplier * (acc / units_per_one) / n_include, zero below min_score.
 * Same bits for any batch order and any number of GPUs; within 1e-14 relative of
 * nabo_mapping_scores. */
int nabo_score_accumulate(const int32_t* tgt_knn, const uint8_t* counts, const long long* int_weights,
                          int n_query, int k, int n_ref, const uint8_t* include, long long* acc,
                          void* stream);
int nabo_scores_finalize(const long long* acc, int n_ref, double units_per_one, double score_multiplier,
                         long long n_include, double min_score, double* out_scores, void* stream);

/* Per-target cluster vote: array form of Graph.classify_target (nabo/_graph.py:722-792).
 * ref_labels int32 (n_ref), -1 = unlabelled; out_label -1 = na_label. */
int nabo_classify_targets(const int32_t* tgt_knn, const uint8_t* counts, const double* lut,
                          int n_query, int k, const int32_t* ref_labels, int n_labels,
                          double weight_frac, int min_degree, double min_weight,
                          int32_t* out_label, void* stream);

/* Mapping specificity: array form of Graph.get_mapping_specificity (nabo/_graph.py:794-824).
 * For every target, the unweighted shortest-path lengths in the reference graph (CSR, symmetric:
 * indptr int64 (n_ref + 1), indices int32) between all pairs of reference cells it has an edge to
 * (tgt_knn[t][j] with counts[t][j] > 0).  out_sum[t] = sum of d(i, j) over ORDERED pairs (twice the
 * reference's sum), out_pairs[t] = ordered pairs connected, out_nmapped[t] = mapped cells; the mean is
 * (out_sum / 2) / (nmapped (nmapped - 1) / 2); out_pairs < nmapped (nmapped - 1) means "no path"
 * (the reference raises NetworkXNoPath), nmapped < 2 means "no pairs" (the reference's NaN).
 * One bit-parallel multi-source BFS per target instead of one BFS per pair; k <= 64. */
size_t nabo_specificity_workspace_bytes(int n_ref, int n_query);
int nabo_mapping_specificity(const long long* indptr, const int32_t* indices, int n_ref,
                             const int32_t* tgt_knn, const uint8_t* counts, int n_query, int k,
                             long long* out_sum, int32_t* out_pairs, int32_t* out_nmapped,
                             void* workspace, size_t workspace_bytes, void* stream);

/* Per-row float32 statistics of a sparse count matrix in NumPy's pairwise summation order: the device
 * form of Dataset.set_sf (nabo/_dataset.py:573-583: temp[keepGenesIdx].sum() per cell) and
 * Dataset.set_gene_stats (:609-622: temp.mean(), temp[temp > 0].mean(), temp.var(), (temp > 0).sum() per
 * gene, temp = densified counts of the kept cells times their size factors).  CSR rows (indptr int64,
 * idx int32 ascending within a row, val float32); pos_of_col[n_cols] = position of a column in the dense
 * vector of length n_dense or -1; scale (n_dense) or NULL.  want_moments = 0 fills out_sum only.
 * Results are bit-identical to NumPy's float32 reductions of the dense vector. */
int nabo_sparse_row_stats(const long long* indptr, const int32_t* idx, const float* val, int n_rows,
                          int n_cols, const int32_t* pos_of_col, const float* scale, long long n_dense,
                          int want_moments, float* out_sum, float* out_mean, float* out_nzmean,
                          float* out_var, int32_t* out_npos, void* stream);

/* Connected components of an undirected graph (edge list int32): out_labels[i] = smallest node id of
 * i's component.  Device form of the nx.connected_components call inside the reference-graph repair
 * (_fix_disconnected_graph, nabo/_mapping.py:203-249).  workspace >= n_nodes * 4 + 512 bytes.
 * Synchronises the stream (one flag read per sweep over the edges). */
int nabo_connected_components(const int32_t* edge_a, const int32_t* edge_b, long long n_edges, int n_nodes,
                              int32_t* out_labels, void* workspace, size_t workspace_bytes, void* stream);

/* ---- (6) scaling + PCA projection: replaces get_scaled_values + transform_pca ---
 * nabo/_dataset.py:905-913 and :1028 (sklearn IncrementalPCA.transform):
 *   a = counts as float32; z = ((a * sf_i) [float32] - mu) / sigma   [float64]
 *   P = z @ components.T - mean @ components.T                       [float64]
 * Dense form: counts (n_cells x ld) float32, gene_idx[G] selects/reorders columns
 * (the reference's `goi`; -1 = gene missing in this dataset -> value 0, :909-910).
 * CSR form: indptr int64 (n_cells+1), col int32, val float32 over ALL genes of
 * the dataset; gene_pos[n_genes_total] = position in the model's gene order or -1.
 * components (n_comps x G) row-major, mean (G).  out (n_cells x ldo) FP64. */
/* z alone (n_cells x G, FP64), bit-identical to get_scaled_values (nabo/_dataset.py:912). */
int nabo_scale_dense(const float* counts, int ld, int n_cells, const int32_t* gene_idx, int G,
                     const float* sf, const double* mu, const double* sigma, double* out, int ldo,
                     void* stream);
int nabo_project_dense(const float* counts, int ld, int n_cells, const int32_t* gene_idx, int G,
                       const float* sf, const double* mu, const double* sigma,
                       const double* components, const double* mean, int n_comps, double* out,
                       int ldo, void* stream);
/* The same dense projection as ONE FP64 tensor-core GEMM (DMMA m8n8k4): the per-gene constants are folded into
 * W[g][c] = C[c][g] / sigma_g and bias[c] = sum_g (mu_g / sigma_g + mean_g) C[c][g] once per call (workspace),
 * so P = (a * sf)[f32 -> f64] . W - bias; FP64 accumulate, equal to nabo_project_dense to ~1e-15 relative. */
size_t nabo_project_dense_workspace_bytes(int G, int n_comps);
int nabo_project_dense_mma(const float* counts, int ld, int n_cells, const int32_t* gene_idx, int G,
                           const float* sf, const double* mu, const double* sigma,
                           const double* components, const double* mean, int n_comps, double* out,
                           int ldo, void* workspace, size_t workspace_bytes, void* stream);
size_t nabo_project_csr_workspace_bytes(int G, int n_comps);
int nabo_project_csr(const int64_t* indptr, const int32_t* col, const float* val, int n_cells,
                     const int32_t* gene_pos, int n_genes_total, int G, const float* sf,
                     const double* mu, const double* sigma, const double* components,
                     const double* mean, int n_comps, double* out, int ldo, void* workspace,
                     size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* NABO_B200_H */
