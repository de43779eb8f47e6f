// Fast kNN engine: candidate pass -> exact FP64 re-rank + certificate -> exact brute force
// for the rows the certificate could not clear.  Results are identical to the exact engine
// (and hence to the reference) by construction; only the amount of FP64 work changes.
//   Euclidean / cosine : tensor-core candidate pass (tc_candidates.cu)
//   modified Canberra  : bit-sliced count bound + FP32 evaluation (canberra_sliced.cu, g <= 128, dist_factor >= 1e-6)
#include "knn_internal.cuh"

NaboFastPlan nabo_fast_plan(int n_query, int n_ref, int g, int k, int metric, double f, int drop_first, bool pre) {
    NaboFastPlan p;
    p.path = NABO_PATH_EXACT;
    p.kprime = 0; p.cap = 0; p.n_split = 1; p.fused = false; p.prepared = false;
    if (metric == NABO_EUCLIDEAN || metric == NABO_COSINE) {
        if (!nabo_tc_supported(g, k, drop_first)) return p;
        const int kprime = nabo_tc_kprime(k, drop_first, &p.cap);
        if (n_ref <= kprime) return p;
        p.path = NABO_PATH_TC;
        p.kprime = kprime;
        p.n_split = nabo_tc_split(n_query, n_ref, g);       // > 1 only when there are fewer query items than SMs
        // split lists stay within 128 candidates per query: every K' > 64 (and the whole 256-key plan) runs unsplit
        while (p.n_split > 1 && p.n_split * kprime > 128) --p.n_split;
        p.fused = p.n_split == 1 && kprime <= 64;
        p.prepared = pre;
        return p;
    }
    if (metric != NABO_MOD_CANBERRA) return p;
    // the interval ends of the sliced pass carry a 1e-6 relative margin over f|x|; it must dominate the FP64
    // rounding of x -+ f|x| (~1e-16 |x|), so a vanishing dist_factor runs on the exact engine.  No candidate pass would
    // help there: nearly every pair is at d = g, so the K'-th candidate ties the threshold and the certificate fails.
    if (!nabo_cbs_supported(g, k, drop_first) || f < 1e-6) return p;
    const int kprime = nabo_cbs_kprime(k, drop_first);
    if (n_ref <= kprime) return p;
    p.path = NABO_PATH_SLICED;
    p.kprime = kprime;
    p.n_split = nabo_cbs_split(n_query, n_ref, g, k, drop_first);
    if (nabo_sm_count() < p.n_split) p.n_split = 1;     // the pieces of a query block run on CTAs of their own
    p.prepared = pre;
    return p;
}

struct FastWork {
    int* fail_rows;
    int* fail_count;
    NaboExactSplit split, few;
    NaboTcWork tc;
    NaboCbsWork cbs;
};

// The regions of one call: the failure list first (the re-rank of the full waves may start while the tensor-core pass
// is still running), the partial lists of the split fallback, then the candidate pass's own.
static void fast_carve(NaboArena& ar, int n_query, int n_ref, int g, int k, int drop_first, const NaboFastPlan& p,
                       FastWork* w) {
    if (p.path == NABO_PATH_EXACT) return;
    w->fail_rows = ar.take<int>(n_query);
    w->fail_count = ar.take<int>(1);
    nabo_exact_split_carve(ar, n_ref, k + (drop_first ? 1 : 0), &w->split, &w->few);
    if (p.path == NABO_PATH_TC) nabo_tc_carve(ar, n_query, n_ref, g, p, &w->tc);
    else nabo_cbs_carve(ar, n_query, n_ref, g, p, &w->cbs);
}

size_t nabo_fast_workspace_bytes(int n_query, int n_ref, int g, int k, int metric, bool pre, double f) {
    // the one-shot size has no dist_factor: the sliced carve, the same for every f >= 1e-6
    const double fv = pre ? f : 1.0;
    size_t need = 0;
    for (int drop_first = 0; drop_first <= 1; ++drop_first) {
        NaboArena m = NaboArena::measure();
        FastWork w;
        fast_carve(m, n_query, n_ref, g, k, drop_first, nabo_fast_plan(n_query, n_ref, g, k, metric, fv, drop_first, pre),
                   &w);
        if (m.off > need) need = m.off;
    }
    return need;
}

int nabo_knn_fast(const double* q, int ldq, const double* r, int ldr, int n_query, int n_ref, int g, int k,
                  int metric, double f, const uint8_t* mask, int drop_first, int idx_offset, int32_t* out_idx,
                  double* out_dist, const NaboRoute& route, void* workspace, size_t workspace_bytes,
                  int64_t* stats_host, cudaStream_t st, const NaboFastRef* pre) {
    const NaboFastPlan p = nabo_fast_plan(n_query, n_ref, g, k, metric, f, drop_first, pre != nullptr);
    const size_t need = nabo_fast_workspace_bytes(n_query, n_ref, g, k, metric, pre != nullptr, f);
    if (workspace_bytes < need)
        return nabo_set_error(NABO_EWORKSPACE, "knn: workspace too small (%zu < %zu)", workspace_bytes, need);
    if (p.path == NABO_PATH_EXACT)
        return nabo_knn_exact_call(q, ldq, r, ldr, n_query, n_ref, g, k, metric, f, mask, drop_first, idx_offset,
                                   out_idx, out_dist, route, stats_host, st);
    NaboStageTimer tm(stats_host != nullptr, st);
    tm.begin();
    NaboArena ar(workspace, workspace_bytes);
    FastWork w;
    fast_carve(ar, n_query, n_ref, g, k, drop_first, p, &w);
    if (!ar.ok) return nabo_set_error(NABO_EWORKSPACE, "knn: workspace too small");
    NABO_CUDA(cudaMemsetAsync(w.fail_count, 0, sizeof(int), st));
    NaboCandidates c;
    int rc;
    if (p.path == NABO_PATH_TC)        // stage timing asked for: the candidate kernel is timed on its own
        rc = nabo_tc_candidates(q, ldq, r, ldr, n_query, n_ref, g, metric, mask, p, w.tc, stats_host != nullptr, tm, st,
                                p.prepared ? &pre->tc : nullptr, &c);
    else
        rc = nabo_cbs_candidates(q, ldq, r, ldr, n_query, n_ref, g, f, mask, p, w.cbs, st, p.prepared ? &pre->cbs : nullptr,
                                 &c);
    if (rc) return rc;
    if (p.n_split > 1) {               // the re-rank certifies against the smallest threshold of the pieces
        rc = nabo_tau_min_launch(const_cast<float*>(c.cert.tau), n_query, p.n_split, st);
        if (rc) return rc;
    }
    int row0 = 0;
    if (c.rows_full > 0) {
        // queries of the full waves: their re-rank is a dependent launch right behind the candidate kernel and runs
        // under its last, partly filled wave
        rc = nabo_rerank_launch(q, ldq, r, ldr, c.rows_full, n_ref, g, k, metric, f, mask, drop_first, idx_offset,
                                c.cand, c.n_cand, c.cert, w.fail_rows, w.fail_count, out_idx, out_dist, route, st,
                                &c.raw, 0, true);
        if (rc) return rc;
        row0 = c.rows_full;
    }
    if (!tm.used[0]) tm.end(0);        // unless the pass closed the candidate stage ahead of its own selection kernels
    rc = nabo_rerank_launch(q, ldq, r, ldr, n_query, n_ref, g, k, metric, f, mask, drop_first, idx_offset, c.cand,
                            c.n_cand, c.cert, w.fail_rows, w.fail_count, out_idx, out_dist, route, st,
                            c.raw.buf ? &c.raw : nullptr, row0);
    if (rc) return rc;
    tm.end(1);
    // rows the certificate did not clear: exact brute force (grid sized for the worst case,
    // blocks beyond the device-side row count exit immediately)
    rc = nabo_knn_exact_fallback(q, ldq, r, ldr, n_query, n_ref, g, k, metric, f, mask, drop_first, idx_offset,
                                 w.fail_rows, w.fail_count, w.split, w.few, out_idx, out_dist, route, st);
    if (rc) return rc;
    tm.end(2);
    if (stats_host) {
        int nfail = 0;
        NABO_CUDA(cudaMemcpyAsync(&nfail, w.fail_count, sizeof(int), cudaMemcpyDeviceToHost, st));
        NABO_CUDA(cudaStreamSynchronize(st));
        stats_host[0] = n_query;
        stats_host[1] = nfail;
        stats_host[2] = p.kprime;
        stats_host[3] = c.launches + 4;      // + re-rank and the 3 fallback kernels
        stats_host[4] = tm.ns(0);
        stats_host[5] = tm.ns(1);
        stats_host[6] = tm.ns(2);
        stats_host[7] = tm.ns(3);
    }
    return 0;
}
