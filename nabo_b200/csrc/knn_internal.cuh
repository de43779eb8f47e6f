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
int nabo_knn_exact_launch_ex(const double* q, int ldq, const double* r, int ldr, int n_query, int n_ref, int g,
                             int k, int metric, double f, const uint8_t* mask, int drop_first, int idx_offset,
                             const int* row_ids, const int* n_rows_dev, const NaboExactSplit& sp, int32_t* out_idx,
                             double* out_dist, const NaboRoute& route, cudaStream_t st);
// Partial-list regions of the split fallback: the split pass and, against n_ref >= NABO_FALLBACK_FEW_MIN_REF, the
// few-rows pass (few->nsplit = 0 otherwise).
void nabo_exact_split_carve(NaboArena& ar, int n_ref, int ksel, NaboExactSplit* split, NaboExactSplit* few);
int nabo_knn_exact_fallback(const double* q, int ldq, const double* r, int ldr, int n_query, int n_ref, int g, int k,
                            int metric, double f, const uint8_t* mask, int drop_first, int idx_offset,
                            const int* row_ids, const int* n_rows_dev, const NaboExactSplit& split,
                            const NaboExactSplit& few, int32_t* out_idx, double* out_dist, const NaboRoute& route,
                            cudaStream_t st);

int nabo_knn_exact_launch(const double* q, int ldq, const double* r, int ldr, int n_query, int n_ref, int g,
                          int k, int metric, double f, const uint8_t* mask, int drop_first, int idx_offset,
                          const int* row_ids, const int* n_rows_dev, int32_t* out_idx, double* out_dist,
                          const NaboRoute& route, cudaStream_t st);
// The exact engine on every row with its stats (one launch, all of it timed as the candidate stage).
int nabo_knn_exact_call(const double* q, int ldq, const double* r, int ldr, int n_query, int n_ref, int g, int k,
                        int metric, double f, const uint8_t* mask, int drop_first, int idx_offset, int32_t* out_idx,
                        double* out_dist, const NaboRoute& route, int64_t* stats_host, cudaStream_t st);

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
// programmatic stream serialisation behind a kernel that signals (NaboCandidates::rows_full)
int nabo_rerank_launch(const double* q, int ldq, const double* r, int ldr, int n_query, int n_ref, int g, int k,
                       int metric, double f, const uint8_t* mask, int drop_first, int idx_offset,
                       const int32_t* cand, int n_cand, const NaboCert& cert, int* fail_rows, int* fail_count,
                       int32_t* out_idx, double* out_dist, const NaboRoute& route, cudaStream_t st,
                       const NaboCandBuf* from_buf = nullptr, int row0 = 0, bool dependent = false);

// Which pass of the fast engine serves a call, and its parameters (nabo_fast_plan, fast.cu).  The passes, the
// workspace carves and the workspace-size functions all take these values from the plan and change none of them.
#define NABO_PATH_EXACT 0        // the exact engine on every row
#define NABO_PATH_TC 1           // tensor-core candidate pass (Euclidean / cosine)
#define NABO_PATH_SLICED 2       // bit-sliced modified-Canberra pass
struct NaboFastPlan {
    int path;
    int kprime;       // K': candidates per list
    int cap;          // tensor core: keys per candidate buffer (128 or 256)
    int n_split;      // reference pieces, each with its own K' list and threshold per query
    bool fused;       // tensor core: the re-rank makes the final K' selection from the raw buffers (no emit kernel)
    bool prepared;    // a prepared reference's operands replace the reference half of the pass
};
NaboFastPlan nabo_fast_plan(int n_query, int n_ref, int g, int k, int metric, double f, int drop_first, bool pre);

// What a candidate pass hands to the fast engine's re-rank.
struct NaboCandidates {
    const int32_t* cand;       // [n_query][n_cand] candidate lists (K' per reference piece)
    int n_cand;
    NaboCert cert;             // cert.tau: [n_split][n_query] thresholds; the engine reduces them to row 0 when split
    NaboCandBuf raw;           // fused path: raw.buf != NULL, the re-rank selects from the candidate buffers
    // Partly filled last wave of the persistent tensor-core kernel (only where it does not cut items at CTA
    // boundaries, i.e. packed references larger than half of L2): every CTA executes griddepcontrol.launch_dependents
    // once its full-wave items are done, so the re-rank of the first rows_full queries, launched right behind it with
    // programmatic stream serialisation, runs while the last wave is still busy, on the SMs that wave leaves idle.
    // 0: nothing to overlap.  When rows_full > 0 the pass has NOT closed the candidate stage of the timer.
    int rows_full;
    int launches;              // kernels the pass reports in stats_host[3]
};

// Reference half of the tensor-core operands, built once by nabo_tc_prepare_ref (prepared reference, knn.cu):
// the packed tiles in the layout the one-shot path writes, and the scale {sc, 1/sc, max scaled reference norm, cosine}.
struct NaboTcRef {
    const void* rb;
    const double* scal;
};

// Each pass takes its regions with one carve function; the size functions run the same carve on a measuring arena.
// With a prepared reference (plan.prepared) the reference half is not carved and those pointers stay NULL.
struct NaboStageTimer;
bool nabo_tc_supported(int g, int k, int drop_first);
int nabo_tc_kprime(int k, int drop_first, int* cap = nullptr);    // cap: keys per candidate buffer of the plan
int nabo_tc_split(int n_query, int n_ref, int g);
#define NABO_TC_MAX_SPLIT 3
struct NaboTcWork {
    void *qa, *rb;                 // packed query and reference tiles
    double *qnorm, *qn2, *rnorm, *scal;
    unsigned long long* cbuf;      // per query slot and reference piece: cap keys, live count (ccnt), threshold (ctau)
    int* ccnt;
    float *ctau, *tau;             // tau: [n_split][n_query]
    int32_t* cand;                 // [n_query][n_split][K']
    unsigned int* maxbits;         // 2 norm maxima, CTA ticket, head flags
};
void nabo_tc_carve(NaboArena& ar, int n_query, int n_ref, int g, const NaboFastPlan& p, NaboTcWork* w);
size_t nabo_tc_prepared_bytes(int n_ref, int g);
int nabo_tc_prepare_ref(const double* r, int ldr, int n_ref, int g, int metric, const uint8_t* mask, void* buffer,
                        NaboTcRef* out, cudaStream_t st);
// timed: the caller times the stages, so the candidate kernel runs alone (rows_full = 0)
int nabo_tc_candidates(const double* q, int ldq, const double* r, int ldr, int n_query, int n_ref, int g, int metric,
                       const uint8_t* mask, const NaboFastPlan& p, const NaboTcWork& w, bool timed, NaboStageTimer& tm,
                       cudaStream_t st, const NaboTcRef* pre, NaboCandidates* out);

// bit-sliced modified-Canberra pass (canberra_sliced.cu)
// Reference half of the sliced pass, built once by nabo_cbs_prepare_ref: FP32 copy, cumulative planes, bin edges.
struct NaboCbsRef {
    const float* rt;
    const uint32_t* planes;
    const float* edges;
};
bool nabo_cbs_supported(int g, int k, int drop_first);
int nabo_cbs_kprime(int k, int drop_first);
int nabo_cbs_split(int n_query, int n_ref, int g, int k, int drop_first);
#define NABO_CBS_MAX_SPLIT 3
struct NaboCbsWork {
    int32_t* cand;                 // [n_query][n_split][K']
    float *tau, *rt, *edges, *qx;  // tau: [n_split][n_query]; reference FP32 copy and bin edges; queries' FP32 copy
    uint32_t *planes, *ctrl;       // reference bit planes; queries' bin controls
    unsigned long long* cbuf;      // per warp of the grid: CAP keys
};
void nabo_cbs_carve(NaboArena& ar, int n_query, int n_ref, int g, const NaboFastPlan& p, NaboCbsWork* w);
size_t nabo_cbs_prepared_bytes(int n_ref, int g);
int nabo_cbs_prepare_ref(const double* r, int ldr, int n_ref, int g, const uint8_t* mask, void* buffer, NaboCbsRef* out,
                         cudaStream_t st);
int nabo_cbs_candidates(const double* q, int ldq, const double* r, int ldr, int n_query, int n_ref, int g, double f,
                        const uint8_t* mask, const NaboFastPlan& p, const NaboCbsWork& w, cudaStream_t st,
                        const NaboCbsRef* pre, NaboCandidates* out);
int nabo_tau_min_launch(float* tau, int n_query, int n_split, cudaStream_t st);

// Reference-side operands of a prepared reference (knn.cu): the tensor-core tiles (Euclidean / cosine) or the
// sliced-pass state (modified Canberra); the pointers of the other engine are NULL.
struct NaboFastRef {
    NaboTcRef tc;
    NaboCbsRef cbs;
};
// Workspace of nabo_knn_fast, the largest carve over drop_first: pre = false for the one-shot call, which has no
// dist_factor (f is not read; modified Canberra is sized for the sliced pass), true for a prepared reference with
// dist_factor f.  0 when every drop_first runs the exact engine.
size_t nabo_fast_workspace_bytes(int n_query, int n_ref, int g, int k, int metric, bool pre, double f);
int nabo_knn_fast(const double* q, int ldq, const double* r, int ldr, int n_query, int n_ref, int g, int k,
                  int metric, double f, const uint8_t* mask, int drop_first, int idx_offset, int32_t* out_idx,
                  double* out_dist, const NaboRoute& route, void* workspace, size_t workspace_bytes,
                  int64_t* stats_host, cudaStream_t st, const NaboFastRef* pre = nullptr);

// Correlation metric (correlation.cu): out (n x g, contiguous) = the rows of x (stride ld) minus their means, in the
// arithmetic the header pins.  One launch.
int nabo_centre_rows(const double* x, int ld, int n, int g, double* out, cudaStream_t st);

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
