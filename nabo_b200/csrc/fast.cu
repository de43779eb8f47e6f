// Fast kNN engine: candidate pass -> exact FP64 re-rank + certificate -> exact brute force
// for the rows the certificate could not clear.  Results are identical to the exact engine
// (and hence to the reference) by construction; only the amount of FP64 work changes.
//   Euclidean / cosine : tensor-core candidate pass (tc_candidates.cu)
//   modified Canberra  : bit-sliced count bound + FP32 evaluation (canberra_sliced.cu, g <= 128), or the two-phase
//                        FP16 / FP32 CUDA-core pass (canberra_candidates.cu, g <= 77) for a vanishing dist_factor
#include "knn_internal.cuh"

// Accumulation-error constant of the tensor-core score relative to (4|q||r| + |r|^2 + |q|^2);
// measured on B200 by tests/test_gpu_tc.py::test_tc_score_error_bound, which asserts a >= 4x margin.
static const double kCAcc = 1.52587890625e-05;   // 2^-16

static size_t cb_extra_bytes(int n_query, int n_ref, int g) {
    const size_t a = nabo_cb_extra_bytes(n_ref, g), b = nabo_cbs_extra_bytes(n_query, n_ref, g);
    return a > b ? a : b;
}

// Tensor-core share of the workspace for every drop_first: with drop_first the buffer plan may be the 256-key one
// (k + 1 >= 89) while k alone still takes the 128-key plan with its reference splits, so the larger of the two.
static size_t tc_workspace_any_drop(int n_query, int n_ref, int g, int k, bool with_ref) {
    const size_t a = nabo_tc_workspace_bytes(n_query, n_ref, g, k, 1, with_ref);
    const size_t b = nabo_tc_workspace_bytes(n_query, n_ref, g, k, 0, with_ref);
    return a > b ? a : b;
}

size_t nabo_fast_workspace_bytes(int n_query, int n_ref, int g, int k, int metric) {
    if (metric == NABO_MOD_CANBERRA)
        return nabo_align_up((size_t)n_query * nabo_cb_kprime(k, 1) * 4 * NABO_CBS_MAX_SPLIT, 256) +
               (2 + NABO_CBS_MAX_SPLIT) * nabo_align_up((size_t)n_query * 4, 256) +
               nabo_align_up(nabo_cb_pretile_floats(n_query, g) * 4, 256) + nabo_align_up(nabo_cb_pretile_floats(n_ref, g) * 4, 256) +
               nabo_align_up(nabo_exact_split_workspace(k + 1), 256) + nabo_align_up(cb_extra_bytes(n_query, n_ref, g), 256) + 4096;
    return tc_workspace_any_drop(n_query, n_ref, g, k, true) + nabo_align_up((size_t)n_query * 4, 256) +
           nabo_align_up(nabo_exact_split_workspace(k + 1), 256) + 1024;
}

// The prepared operands serve a call when its engine is the one they were built for; the size below covers every
// drop_first, so it is the query half only where both take that engine (else the full one-shot size).
static bool cbs_prepared_used(int g, int k, int drop_first, double f) { return f >= 1e-6 && nabo_cbs_supported(g, k, drop_first); }

size_t nabo_fast_prepared_workspace_bytes(int n_query, int n_ref, int g, int k, int metric, double f) {
    if (metric == NABO_MOD_CANBERRA) {
        if (!cbs_prepared_used(g, k, 1, f)) return nabo_fast_workspace_bytes(n_query, n_ref, g, k, metric);
        return nabo_align_up((size_t)n_query * nabo_cb_kprime(k, 1) * 4 * NABO_CBS_MAX_SPLIT, 256) +
               (2 + NABO_CBS_MAX_SPLIT) * nabo_align_up((size_t)n_query * 4, 256) +
               nabo_align_up(nabo_exact_split_workspace(k + 1), 256) +
               nabo_align_up(nabo_cbs_extra_bytes(n_query, n_ref, g, false), 256) + 4096;
    }
    if (!nabo_tc_supported(g, k, 1)) return nabo_fast_workspace_bytes(n_query, n_ref, g, k, metric);
    return tc_workspace_any_drop(n_query, n_ref, g, k, false) + nabo_align_up((size_t)n_query * 4, 256) +
           nabo_align_up(nabo_exact_split_workspace(k + 1), 256) + 1024;
}

int nabo_knn_fast(const double* q, int ldq, const double* r, int ldr, int n_query, int n_ref, int g, int k,
                  int metric, double f, const uint8_t* mask, int drop_first, int idx_offset, int32_t* out_idx,
                  double* out_dist, const NaboRoute& route, void* workspace, size_t workspace_bytes,
                  int64_t* stats_host, cudaStream_t st, const NaboFastRef* pre) {
    NaboStageTimer tm(stats_host != nullptr, st);
    tm.begin();
    const bool use_tc = (metric == NABO_EUCLIDEAN || metric == NABO_COSINE) && nabo_tc_supported(g, k, drop_first) &&
                        n_ref > nabo_tc_kprime(k, drop_first);
    // the interval ends of the sliced pass carry a 1e-6 relative margin over f|x|; it must dominate the FP64
    // rounding of x -+ f|x| (~1e-16 |x|), so a vanishing dist_factor goes to the FP16 two-phase pass instead
    const bool sliced_ok = metric == NABO_MOD_CANBERRA && nabo_cbs_supported(g, k, drop_first) && f >= 1e-6;
    const bool use_cb = metric == NABO_MOD_CANBERRA && (sliced_ok || nabo_cb_supported(g, k, drop_first)) &&
                        n_ref > nabo_cb_kprime(k, drop_first);
    if (use_cb) {
        // a prepared reference's sliced operands replace the FP32 copy, planes and edges of this call
        const NaboCbsRef* pre_cb = sliced_ok && pre && pre->cbs.planes ? &pre->cbs : nullptr;
        const size_t need = pre ? nabo_fast_prepared_workspace_bytes(n_query, n_ref, g, k, metric, f)
                                : nabo_fast_workspace_bytes(n_query, n_ref, g, k, metric);
        if (workspace_bytes < need) return nabo_set_error(NABO_EWORKSPACE, "knn: workspace too small");
        NaboArena ar(workspace, workspace_bytes);
        const int kprime = nabo_cb_kprime(k, drop_first);
        const int n_split = sliced_ok ? nabo_cbs_split(n_query, n_ref, g, k, drop_first) : 1;
        int32_t* cand = ar.take<int32_t>((size_t)n_query * kprime * n_split);
        float* tau = ar.take<float>((size_t)n_query * n_split);
        int* fail_rows = ar.take<int>(n_query);
        int* fail_count = ar.take<int>(1);
        float* qt = pre_cb ? nullptr : ar.take<float>(nabo_cb_pretile_floats(n_query, g));
        float* rt = pre_cb ? nullptr : ar.take<float>(nabo_cb_pretile_floats(n_ref, g));
        char* split_ws = ar.take<char>(nabo_exact_split_workspace(k + (drop_first ? 1 : 0)));
        const size_t extra_bytes = pre_cb ? nabo_cbs_extra_bytes(n_query, n_ref, g, false) : cb_extra_bytes(n_query, n_ref, g);
        char* extra = ar.take<char>(extra_bytes);
        if (!ar.ok) return nabo_set_error(NABO_EWORKSPACE, "knn: workspace too small");
        NABO_CUDA(cudaMemsetAsync(fail_count, 0, sizeof(int), st));
        int rc = sliced_ok
                     ? nabo_cbs_candidates(q, ldq, r, ldr, n_query, n_ref, g, k, f, mask, drop_first, n_split, rt, extra,
                                           extra_bytes, cand, tau, st, pre_cb)
                     : nabo_cb_candidates(q, ldq, r, ldr, n_query, n_ref, g, k, f, mask, drop_first, qt, rt, extra, cand,
                                          tau, st);
        if (rc) return rc;
        if (n_split > 1) {
            rc = nabo_tau_min_launch(tau, n_query, n_split, st);
            if (rc) return rc;
        }
        tm.end(0);
        NaboCert cert;
        cert.kind = NABO_CERT_LINEAR; cert.tau = tau; cert.qn2 = nullptr; cert.scal = nullptr; cert.c_acc = nabo_cb_eps(g); cert.abs_slack = 0.0;
        rc = nabo_rerank_launch(q, ldq, r, ldr, n_query, n_ref, g, k, metric, f, mask, drop_first, idx_offset, cand,
                                kprime * n_split, cert, fail_rows, fail_count, out_idx, out_dist, route, st);
        if (rc) return rc;
        tm.end(1);
        rc = nabo_knn_exact_fallback(q, ldq, r, ldr, n_query, n_ref, g, k, metric, f, mask, drop_first, idx_offset,
                                     fail_rows, fail_count, split_ws, out_idx, out_dist, route, st);
        if (rc) return rc;
        tm.end(2);
        if (stats_host) {
            int nfail = 0;
            NABO_CUDA(cudaMemcpyAsync(&nfail, fail_count, sizeof(int), cudaMemcpyDeviceToHost, st));
            NABO_CUDA(cudaStreamSynchronize(st));
            stats_host[0] = n_query; stats_host[1] = nfail; stats_host[2] = kprime;
            stats_host[3] = sliced_ok ? 10 : 11;      // preparation + candidate pass + re-rank + 3 fallback kernels
            stats_host[4] = tm.ns(0); stats_host[5] = tm.ns(1); stats_host[6] = tm.ns(2);
        }
        return 0;
    }
    if (!use_tc) {
        int rc = nabo_knn_exact_launch(q, ldq, r, ldr, n_query, n_ref, g, k, metric, f, mask, drop_first, idx_offset,
                                       nullptr, nullptr, out_idx, out_dist, route, st);
        tm.end(0);
        if (rc) return rc;
        if (stats_host) {
            NABO_CUDA(cudaStreamSynchronize(st));
            stats_host[1] = n_query;
            stats_host[3] = 1;
            stats_host[4] = tm.ns(0);
        }
        return 0;
    }
    const NaboTcRef* pre_tc = pre && pre->tc.rb ? &pre->tc : nullptr;
    const size_t need = pre ? nabo_fast_prepared_workspace_bytes(n_query, n_ref, g, k, metric, f)
                            : nabo_fast_workspace_bytes(n_query, n_ref, g, k, metric);
    if (workspace_bytes < need)
        return nabo_set_error(NABO_EWORKSPACE, "knn: workspace too small (%zu < %zu)", workspace_bytes, need);
    NaboArena ar(workspace, workspace_bytes);
    int32_t* cand = nullptr;
    float* tau = nullptr;
    double *qn2 = nullptr, *scal = nullptr;
    int kprime = 0, launches = 0;
    NaboCandBuf raw;
    raw.buf = nullptr;
    int n_split = nabo_tc_split(n_query, n_ref, g);              // > 1 only when there are fewer query items than SMs
    // split lists stay within 128 candidates per query: every K' > 64 (and the whole 256-key plan) runs unsplit
    while (n_split > 1 && n_split * nabo_tc_kprime(k, drop_first) > 128) --n_split;
    // the failure list first: the re-rank of the full waves may start while the candidate pass is still running
    int* fail_rows = ar.take<int>(n_query);
    int* fail_count = ar.take<int>(1);
    char* split_ws = ar.take<char>(nabo_exact_split_workspace(k + (drop_first ? 1 : 0)));
    if (!ar.ok) return nabo_set_error(NABO_EWORKSPACE, "knn: workspace too small");
    NABO_CUDA(cudaMemsetAsync(fail_count, 0, sizeof(int), st));
    NaboTailSplit tail;
    tail.rows_full = 0; tail.applies = 0;
    tail.dry = stats_host != nullptr;      // stage timing asked for: the candidate kernel is timed on its own
    int rc = nabo_tc_candidates(q, ldq, r, ldr, n_query, n_ref, g, k, metric, mask, drop_first, &n_split, ar, &cand,
                                &kprime, &tau, &qn2, &scal, &launches, tm, st, &raw, &tail, pre_tc);  // n_split out: K' lists per query
    if (rc) return rc;
    if (!ar.ok) return nabo_set_error(NABO_EWORKSPACE, "knn: workspace too small");
    NaboCert cert;
    cert.kind = metric == NABO_COSINE ? NABO_CERT_COSINE : NABO_CERT_EUCLID;
    cert.tau = tau; cert.qn2 = qn2; cert.scal = scal; cert.c_acc = kCAcc;
    cert.abs_slack = 2.0 * sqrt((double)g) * 5.9604644775390625e-08;
    int row0 = 0;
    if (tail.rows_full > 0) {
        // queries of the full waves: their re-rank is a dependent launch right behind the candidate kernel and runs
        // under its last, partly filled wave
        rc = nabo_rerank_launch(q, ldq, r, ldr, tail.rows_full, n_ref, g, k, metric, f, mask, drop_first, idx_offset, cand,
                                kprime * n_split, cert, fail_rows, fail_count, out_idx, out_dist, route, st, &raw, 0, true);
        if (rc) return rc;
        tm.end(0);
        row0 = tail.rows_full;
    }
    launches += tail.applies;
    rc = nabo_rerank_launch(q, ldq, r, ldr, n_query, n_ref, g, k, metric, f, mask, drop_first, idx_offset, cand,
                            kprime * n_split, cert, fail_rows, fail_count, out_idx, out_dist, route, st,
                            raw.buf ? &raw : nullptr, row0);
    if (rc) return rc;
    tm.end(1);
    // rows the certificate did not clear: exact brute force (grid sized for the worst case,
    // blocks beyond the device-side row count exit immediately)
    rc = nabo_knn_exact_fallback(q, ldq, r, ldr, n_query, n_ref, g, k, metric, f, mask, drop_first, idx_offset,
                                 fail_rows, fail_count, split_ws, out_idx, out_dist, route, st);
    if (rc) return rc;
    tm.end(2);
    if (stats_host) {
        int nfail = 0;
        NABO_CUDA(cudaMemcpyAsync(&nfail, fail_count, sizeof(int), cudaMemcpyDeviceToHost, st));
        NABO_CUDA(cudaStreamSynchronize(st));
        stats_host[0] = n_query;
        stats_host[1] = nfail;
        stats_host[2] = kprime;
        stats_host[3] = launches + 4;
        stats_host[4] = tm.ns(0);
        stats_host[5] = tm.ns(1);
        stats_host[6] = tm.ns(2);
        stats_host[7] = tm.ns(3);
    }
    return 0;
}
