// Internal (non-ABI) entry points shared between the kNN translation units.
#pragma once
#include "common.cuh"

// Routed result rows (reference-sharded mode): result row t of a kNN call goes to part p with
// bounds[p] <= t < bounds[p + 1], at row t - bounds[p] of that part's (rows x k) idx / dist blocks.  The blocks
// may be anywhere the device can store to - slices of a local all-to-all send buffer, or the receive buffers of
// the peer GPUs mapped over NVLink - so the kernel that produces a row also delivers it.  n_parts == 0: plain
// contiguous out_idx / out_dist.
#define NABO_MAX_PARTS 16
struct NaboRoute {
    int n_parts;
    int bounds[NABO_MAX_PARTS + 1];
    int32_t* idx[NABO_MAX_PARTS];
    double* dist[NABO_MAX_PARTS];
};
__device__ __forceinline__ void nabo_route_row(const NaboRoute& rt, long long row, int k, int32_t* out_idx,
                                               double* out_dist, int32_t*& ri, double*& rd) {
    if (rt.n_parts == 0) {
        ri = out_idx + row * k;
        rd = out_dist + row * k;
        return;
    }
    int p = 0;
    while (p + 1 < rt.n_parts && row >= rt.bounds[p + 1]) ++p;
    const long long local = row - rt.bounds[p];
    ri = rt.idx[p] + local * k;
    rd = rt.dist[p] + local * k;
}

// Split fallback: with at most NABO_FALLBACK_SPLIT_ROWS uncertified rows the exact engine splits the
// reference range over blockIdx.y and merges the partial lists (a single block would otherwise scan
// the whole reference alone and dominate the call).
#define NABO_FALLBACK_SPLIT_ROWS 2048
// A handful of uncertified rows against a large reference: the range is cut into many more pieces (two per SM) and
// the partial lists are merged by a whole block per row - one row at 1.25 M references: 5.2 -> under 1 ms.
#define NABO_FALLBACK_FEW_ROWS 64
#define NABO_FALLBACK_FEW_ENTRIES 16384       /* pieces x (k + drop_first) of the few-rows merge */
#define NABO_FALLBACK_FEW_MIN_REF 262144
struct NaboExactSplit {
    int mode;            // 0 = plain, 1 = split partial pass (runs iff f_min < rows <= f_max), 2 = plain iff rows > f_max
    int nsplit, f_max, f_min;
    int32_t* part_idx;   // [nsplit][f_max][ksel]
    double* part_dist;
};
int nabo_exact_split_count(int ksel);
size_t nabo_exact_split_workspace(int ksel);
int nabo_knn_exact_launch_ex(const double* q, int ldq, const double* r, int ldr, int n_query, int n_ref, int g,
                             int k, int metric, double f, const uint8_t* mask, int drop_first, int idx_offset,
                             const int* row_ids, const int* n_rows_dev, const NaboExactSplit& sp, int32_t* out_idx,
                             double* out_dist, const NaboRoute& route, cudaStream_t st);
int nabo_knn_exact_fallback(const double* q, int ldq, const double* r, int ldr, int n_query, int n_ref, int g, int k,
                            int metric, double f, const uint8_t* mask, int drop_first, int idx_offset,
                            const int* row_ids, const int* n_rows_dev, void* split_ws, int32_t* out_idx,
                            double* out_dist, const NaboRoute& route, cudaStream_t st);

int nabo_knn_exact_launch(const double* q, int ldq, const double* r, int ldr, int n_query, int n_ref, int g,
                          int k, int metric, double f, const uint8_t* mask, int drop_first, int idx_offset,
                          const int* row_ids, const int* n_rows_dev, int32_t* out_idx, double* out_dist,
                          const NaboRoute& route, cudaStream_t st);

// Candidate certificate evaluated by the re-rank (see rerank_kernel).
#define NABO_CERT_NONE 0
#define NABO_CERT_EUCLID 1   // L = sqrt(tau + |q~|^2 - eps) / sc - slack
#define NABO_CERT_COSINE 2   // chord on unit vectors -> e^2 / 2
#define NABO_CERT_LINEAR 3   // L = tau - c_acc  (candidate score is a lower bound of the distance)
struct NaboCert {
    int kind;
    const float* tau;      // [n_query] final candidate threshold (score space), +inf = nothing rejected
    const double* qn2;     // [n_query] |q~|^2 in scaled units (Euclid / cosine)
    const double* scal;    // {sc, 1/sc, max scaled reference norm, cosine flag}
    double c_acc;          // accumulation-error constant (Euclid / cosine) or absolute slack (linear)
    double abs_slack;      // Euclid: absolute split error in scaled units, 2 sqrt(g) 2^-24 (the FP16 low halves are
                           // subnormal below |x| ~ 0.25, where the split error stops being relative)
};

// Candidates straight from the buffers the tensor-core sweep left behind (one 128-key buffer per query, query i at
// slot i): the re-rank kernel makes the final K' selection itself (histogram cut + rank inside the cut bin) - no emit kernel, no
// candidate-index round trip.  buf == NULL: candidates come from the `cand` lists.
struct NaboCandBuf {
    const unsigned long long* buf;   // [n_query][128] keys (score bits << 32 | reference row)
    const int* cnt;                  // [n_query] live keys
    const float* tau;                // [n_query] running threshold at the end of the sweep
    int kprime;
};
// row0: the launch covers the queries [row0, n_query) (all pointers are those of row 0); dependent: launched with
// programmatic stream serialisation behind a kernel that signals (NaboTailSplit)
int nabo_rerank_launch(const double* q, int ldq, const double* r, int ldr, int n_query, int n_ref, int g, int k,
                       int metric, double f, const uint8_t* mask, int drop_first, int idx_offset,
                       const int32_t* cand, int n_cand, const NaboCert& cert, int* fail_rows, int* fail_count,
                       int32_t* out_idx, double* out_dist, const NaboRoute& route, cudaStream_t st,
                       const NaboCandBuf* from_buf = nullptr, int row0 = 0, bool dependent = false);

// Partly filled last wave of the persistent candidate kernel (tc_candidates.cu; only where it does not cut items at
// CTA boundaries, i.e. packed references larger than half of L2): every CTA executes
// griddepcontrol.launch_dependents once its full-wave items are done, so a kernel launched right behind it on the same
// stream with programmatic stream serialisation - the re-rank of the first rows_full queries - runs while the last wave is
// still busy, on the SMs that wave leaves idle.  rows_full = 0: nothing to overlap.  When rows_full > 0 the candidate pass
// has NOT closed its timing stage: the caller does, after the dependent launch.
struct NaboTailSplit {
    int dry;                   // in: 1 = only report (the per-stage timing pass measures the candidate kernel alone)
    int rows_full;             // out: queries the dependent launch may take (0 with dry)
    int applies;               // out: 1 when the shape qualifies (with or without dry)
};

struct NaboStageTimer;
bool nabo_tc_supported(int g, int k, int drop_first);
int nabo_tc_kprime(int k, int drop_first);
size_t nabo_tc_workspace_bytes(int n_query, int n_ref, int g, int k, int drop_first);
#define NABO_TC_MAX_SPLIT 3
int nabo_tc_split(int n_query, int n_ref, int g);
int nabo_tc_candidates(const double* q, int ldq, const double* r, int ldr, int n_query, int n_ref, int g, int k,
                       int metric, const uint8_t* mask, int drop_first, int* n_split_io, NaboArena& ar, int32_t** cand_idx_out,
                       int* kprime_out, float** cert_tau_out, double** qn2_out, double** scal_out, int* launches,
                       NaboStageTimer& tm, cudaStream_t st, NaboCandBuf* raw_out = nullptr, NaboTailSplit* tail = nullptr);

bool nabo_cb_supported(int g, int k, int drop_first);
int nabo_cb_kprime(int k, int drop_first);
double nabo_cb_eps(int g);
size_t nabo_cb_pretile_floats(int n, int g);
size_t nabo_cb_extra_bytes(int n_ref, int g);
int nabo_cb_candidates(const double* q, int ldq, const double* r, int ldr, int n_query, int n_ref, int g, int k,
                       double f, const uint8_t* mask, int drop_first, float* qt, float* rt, void* extra, int32_t* cand,
                       float* tau, cudaStream_t st);

int nabo_cb_pretile_launch(const double* x, int ld, int n, int g, float* out, cudaStream_t st);
// bit-sliced Canberra pass (canberra_sliced.cu); same outputs as nabo_cb_candidates
bool nabo_cbs_supported(int g, int k, int drop_first);
size_t nabo_cbs_extra_bytes(int n_query, int n_ref, int g);
#define NABO_CBS_MAX_SPLIT 3
int nabo_cbs_split(int n_query, int n_ref, int g, int k, int drop_first);
int nabo_cbs_candidates(const double* q, int ldq, const double* r, int ldr, int n_query, int n_ref, int g, int k,
                        double f, const uint8_t* mask, int drop_first, int n_split, float* rt, void* extra,
                        size_t extra_bytes, int32_t* cand, float* tau, cudaStream_t st);
int nabo_tau_min_launch(float* tau, int n_query, int n_split, cudaStream_t st);

size_t nabo_fast_workspace_bytes(int n_query, int n_ref, int g, int k, int metric);
int nabo_knn_fast(const double* q, int ldq, const double* r, int ldr, int n_query, int n_ref, int g, int k,
                  int metric, double f, const uint8_t* mask, int drop_first, int idx_offset, int32_t* out_idx,
                  double* out_dist, const NaboRoute& route, void* workspace, size_t workspace_bytes,
                  int64_t* stats_host, cudaStream_t st);

// CUDA-event stage timer, active only when the caller asked for stats (stats_host != NULL).
// Usage: begin(); <launch stage 0>; end(0); <launch stage 1>; end(1); ... sync; ns(i).
struct NaboStageTimer {
    static constexpr int MAXS = 4;
    bool on;
    cudaStream_t st;
    cudaEvent_t start;
    cudaEvent_t stop[MAXS];
    int prev[MAXS];
    bool used[MAXS];
    int last;
    NaboStageTimer(bool enable, cudaStream_t s) : on(enable), st(s), last(-1) {
        for (int i = 0; i < MAXS; ++i) { prev[i] = -1; used[i] = false; }
        if (on) {
            cudaEventCreate(&start);
            for (int i = 0; i < MAXS; ++i) cudaEventCreate(&stop[i]);
        }
    }
    ~NaboStageTimer() {
        if (on) {
            cudaEventDestroy(start);
            for (int i = 0; i < MAXS; ++i) cudaEventDestroy(stop[i]);
        }
    }
    void begin() { if (on) cudaEventRecord(start, st); }
    void end(int i) {          // stage i ran since the previous begin()/end()
        if (!on) return;
        cudaEventRecord(stop[i], st);
        used[i] = true;
        prev[i] = last;
        last = i;
    }
    long long ns(int i) {      // valid after the stream has been synchronised
        if (!on || !used[i]) return 0;
        float ms = 0.f;
        cudaEventElapsedTime(&ms, prev[i] < 0 ? start : stop[prev[i]], stop[i]);
        return (long long)((double)ms * 1e6);
    }
};
