// nabo_knn: engine selection and workspace layout for the fused distance + top-k path
// (replaces _calc_dist, nabo/_mapping.py:48-148).
#include "common.cuh"
#include "knn_internal.cuh"

#include <string.h>

// Workspace of the engine that serves a call: 256 bytes for the exact engine, the fast engine's carve otherwise.
static size_t engine_bytes(int n_query, int n_ref, int g, int k, int metric, int mode, bool pre, double f) {
    if (mode == NABO_MODE_EXACT) return 256;
    return nabo_fast_workspace_bytes(n_query, n_ref, g, k, metric, pre, f);
}

// ------------------------------------------------------------------ correlation
// Correlation distance is the cosine distance of the row-centred vectors (include/nabo_b200.h).  Metric 3 is resolved
// here and only here: the centred FP64 copies take the head of the workspace (the reference's copy only without a
// prepared reference, whose buffer holds it), then the call continues as cosine on the copies with the rest of the
// workspace.  The plans, the carves of the passes and the kernels never see metric 3.
struct CorrCopies {
    double *q, *r;
};
static void corr_carve(NaboArena& ar, int n_query, int n_ref, int g, bool ref_copy, CorrCopies* c) {
    c->q = ar.take<double>((size_t)n_query * g);
    c->r = ref_copy ? ar.take<double>((size_t)n_ref * g) : nullptr;
}
// bytes of the copies; the cosine call's workspace starts there
static size_t corr_head_bytes(int n_query, int n_ref, int g, bool ref_copy) {
    if (n_query < 0 || n_ref < 0 || g < 1) return 0;
    NaboArena m = NaboArena::measure();
    CorrCopies c;
    corr_carve(m, n_query, n_ref, g, ref_copy, &c);
    return nabo_align_up(m.off, 256);
}

extern "C" size_t nabo_knn_workspace_bytes(int n_query, int n_ref, int g, int k, int metric, int mode) {
    if (metric == NABO_CORRELATION)
        return corr_head_bytes(n_query, n_ref, g, true) + engine_bytes(n_query, n_ref, g, k, NABO_COSINE, mode, false, 0.0);
    return engine_bytes(n_query, n_ref, g, k, metric, mode, false, 0.0);
}

static int knn_impl(const double* q, int ldq, const double* r, int ldr, int n_query, int n_ref, int g, int k,
                    int metric, double dist_factor, const uint8_t* ref_mask, int drop_first, int idx_offset,
                    int mode, int32_t* out_idx, double* out_dist, const NaboRoute& route, void* workspace,
                    size_t workspace_bytes, int64_t* stats_host, void* stream, const NaboFastRef* pre = nullptr);

static int parse_route(int n_query, int n_parts, const int* part_bounds_host, int32_t* const* part_idx_host,
                       double* const* part_dist_host, NaboRoute& route) {
    NABO_ARG(n_parts >= 1 && n_parts <= NABO_MAX_PARTS, "knn_routed: n_parts=%d outside 1..%d", n_parts, NABO_MAX_PARTS);
    NABO_ARG(part_bounds_host && part_idx_host && part_dist_host, "knn_routed: null table");
    NABO_ARG(part_bounds_host[0] == 0 && part_bounds_host[n_parts] == n_query,
             "knn_routed: part bounds must run from 0 to n_query");
    route.n_parts = n_parts;
    for (int p = 0; p <= n_parts; ++p) route.bounds[p] = part_bounds_host[p];
    for (int p = 0; p < n_parts; ++p) {
        NABO_ARG(route.bounds[p] <= route.bounds[p + 1], "knn_routed: part bounds must not decrease");
        NABO_ARG(route.bounds[p] == route.bounds[p + 1] || (part_idx_host[p] && part_dist_host[p]),
                 "knn_routed: part %d has rows but no buffers", p);
        route.idx[p] = part_idx_host[p];
        route.dist[p] = part_dist_host[p];
    }
    return 0;
}

extern "C" int nabo_knn(const double* q, int ldq, const double* r, int ldr, int n_query, int n_ref, int g, int k,
                        int metric, double dist_factor, const uint8_t* ref_mask, int drop_first, int idx_offset,
                        int mode, int32_t* out_idx, double* out_dist, void* workspace, size_t workspace_bytes,
                        int64_t* stats_host, void* stream) {
    NaboRoute plain;
    plain.n_parts = 0;
    return knn_impl(q, ldq, r, ldr, n_query, n_ref, g, k, metric, dist_factor, ref_mask, drop_first, idx_offset, mode,
                    out_idx, out_dist, plain, workspace, workspace_bytes, stats_host, stream);
}

extern "C" int nabo_knn_routed(const double* q, int ldq, const double* r, int ldr, int n_query, int n_ref, int g,
                               int k, int metric, double dist_factor, const uint8_t* ref_mask, int drop_first,
                               int idx_offset, int mode, int n_parts, const int* part_bounds_host,
                               int32_t* const* part_idx_host, double* const* part_dist_host, void* workspace,
                               size_t workspace_bytes, int64_t* stats_host, void* stream) {
    NaboRoute route;
    int rc = parse_route(n_query, n_parts, part_bounds_host, part_idx_host, part_dist_host, route);
    if (rc) return rc;
    return knn_impl(q, ldq, r, ldr, n_query, n_ref, g, k, metric, dist_factor, ref_mask, drop_first, idx_offset, mode,
                    nullptr, nullptr, route, workspace, workspace_bytes, stats_host, stream);
}

static int knn_impl(const double* q, int ldq, const double* r, int ldr, int n_query, int n_ref, int g, int k,
                    int metric, double dist_factor, const uint8_t* ref_mask, int drop_first, int idx_offset,
                    int mode, int32_t* out_idx, double* out_dist, const NaboRoute& route, void* workspace,
                    size_t workspace_bytes, int64_t* stats_host, void* stream, const NaboFastRef* pre) {
    cudaStream_t st = (cudaStream_t)stream;
    NABO_ARG(n_query >= 0 && n_ref >= 1 && g >= 1 && k >= 1, "knn: bad sizes n_query=%d n_ref=%d g=%d k=%d",
             n_query, n_ref, g, k);
    NABO_ARG(ldq >= g && ldr >= g, "knn: leading dimension smaller than g");
    NABO_ARG(metric == NABO_EUCLIDEAN || metric == NABO_MOD_CANBERRA || metric == NABO_COSINE ||
             metric == NABO_CORRELATION, "knn: unknown metric %d", metric);
    NABO_ARG(metric != NABO_MOD_CANBERRA || dist_factor > 0.0, "knn: dist_factor must be > 0");
    if (n_query == 0) return 0;
    NABO_ARG(q && r && (route.n_parts > 0 || (out_idx && out_dist)), "knn: null pointer");
    if (stats_host) for (int i = 0; i < 8; ++i) stats_host[i] = 0;
    if (metric == NABO_CORRELATION) {
        NABO_ARG(mode == NABO_MODE_EXACT || mode == NABO_MODE_FAST, "knn: unknown mode %d", mode);
        // a prepared reference's rows are its centred copy already
        const bool ref_copy = pre == nullptr;
        const size_t head = corr_head_bytes(n_query, n_ref, g, ref_copy);
        const size_t need = head + engine_bytes(n_query, n_ref, g, k, NABO_COSINE, mode, pre != nullptr, dist_factor);
        if (!workspace || workspace_bytes < need)
            return nabo_set_error(NABO_EWORKSPACE, "knn: workspace too small (%zu < %zu)", workspace_bytes, need);
        NaboArena ar(workspace, workspace_bytes);
        CorrCopies c;
        corr_carve(ar, n_query, n_ref, g, ref_copy, &c);
        NaboStageTimer tm(stats_host != nullptr, st);
        tm.begin();
        int rc = nabo_centre_rows(q, ldq, n_query, g, c.q, st);
        if (rc == 0 && ref_copy) rc = nabo_centre_rows(r, ldr, n_ref, g, c.r, st);
        if (rc) return rc;
        tm.end(0);
        rc = knn_impl(c.q, g, ref_copy ? c.r : r, ref_copy ? g : ldr, n_query, n_ref, g, k, NABO_COSINE, dist_factor,
                      ref_mask, drop_first, idx_offset, mode, out_idx, out_dist, route, (char*)workspace + head,
                      workspace_bytes - head, stats_host, stream, pre);
        if (rc) return rc;
        if (stats_host) {
            NABO_CUDA(cudaStreamSynchronize(st));
            stats_host[3] += ref_copy ? 2 : 1;
            stats_host[7] += tm.ns(0);
        }
        return 0;
    }
    if (mode == NABO_MODE_EXACT)
        return nabo_knn_exact_call(q, ldq, r, ldr, n_query, n_ref, g, k, metric, dist_factor, ref_mask, drop_first,
                                   idx_offset, out_idx, out_dist, route, stats_host, st);
    NABO_ARG(mode == NABO_MODE_FAST, "knn: unknown mode %d", mode);
    return nabo_knn_fast(q, ldq, r, ldr, n_query, n_ref, g, k, metric, dist_factor, ref_mask, drop_first,
                         idx_offset, out_idx, out_dist, route, workspace, workspace_bytes, stats_host, st, pre);
}

// ------------------------------------------------------------------ prepared reference
// Buffer layout: the reference half of the fast engine's operands for the metric (tc_candidates.cu /
// canberra_sliced.cu own the layout inside), at offset 0; correlation puts the centred copy of the rows in front of
// them.  The descriptor keeps the device addresses.
// The plan is the pass the fast engine takes for the metric at k = 1 against a large reference: the tensor-core or the
// sliced pass, whose operands then serve every call that takes the same pass.
static bool prepared_plan(int g, int metric, int* plan) {
    if (metric == NABO_CORRELATION) metric = NABO_COSINE;   // the tensor-core operands of the centred copy
    const int path = nabo_fast_plan(1, 1 << 30, g, 1, metric, 1.0, 0, true).path;
    *plan = path == NABO_PATH_TC ? NABO_PLAN_TC : NABO_PLAN_SLICED;
    return path == NABO_PATH_TC || path == NABO_PATH_SLICED;
}

extern "C" size_t nabo_ref_prepared_bytes(int n_ref, int g, int metric) {
    int plan = 0;
    if (n_ref < 1 || !prepared_plan(g, metric, &plan)) return 0;
    if (metric == NABO_CORRELATION) return corr_head_bytes(0, n_ref, g, true) + nabo_tc_prepared_bytes(n_ref, g);
    return plan == NABO_PLAN_TC ? nabo_tc_prepared_bytes(n_ref, g) : nabo_cbs_prepared_bytes(n_ref, g);
}

extern "C" int nabo_ref_prepare(const double* r, int ldr, int n_ref, int g, int metric, const uint8_t* ref_mask,
                                void* buffer, size_t buffer_bytes, nabo_prepared_ref* prepared_host, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    NABO_ARG(prepared_host, "ref_prepare: null descriptor");
    memset(prepared_host, 0, sizeof(*prepared_host));
    int plan = 0;
    if (!prepared_plan(g, metric, &plan))
        return nabo_set_error(NABO_EUNSUPPORTED, "ref_prepare: metric %d with g=%d has no fast plan (1 <= g <= 128)",
                              metric, g);
    NABO_ARG(n_ref >= 1 && ldr >= g, "ref_prepare: bad sizes n_ref=%d ldr=%d g=%d", n_ref, ldr, g);
    NABO_ARG(r && buffer, "ref_prepare: null pointer");
    const size_t need = nabo_ref_prepared_bytes(n_ref, g, metric);
    NABO_ARG(buffer_bytes >= need, "ref_prepare: buffer too small (%zu < %zu)", buffer_bytes, need);
    nabo_prepared_ref d;
    memset(&d, 0, sizeof(d));
    d.magic = NABO_PREPARED_MAGIC;
    d.abi_version = NABO_ABI_VERSION;
    d.n_ref = n_ref; d.g = g; d.metric = metric; d.plan = plan;
    d.r = r; d.ldr = ldr; d.ref_mask = ref_mask;
    d.buffer = buffer; d.buffer_bytes = buffer_bytes;
    if (plan == NABO_PLAN_TC) {
        // correlation: the buffer starts with the centred copy; the operands that follow are those of the copy as cosine
        const double* rows = r;
        void* ops = buffer;
        if (metric == NABO_CORRELATION) {
            NaboArena ar(buffer, buffer_bytes);
            CorrCopies c;
            corr_carve(ar, 0, n_ref, g, true, &c);
            int rc = nabo_centre_rows(r, ldr, n_ref, g, c.r, st);
            if (rc) return rc;
            rows = d.r = c.r;
            d.ldr = g;
            ops = (char*)buffer + corr_head_bytes(0, n_ref, g, true);
        }
        NaboTcRef t;
        int rc = nabo_tc_prepare_ref(rows, d.ldr, n_ref, g, metric == NABO_CORRELATION ? NABO_COSINE : metric, ref_mask,
                                     ops, &t, st);
        if (rc) return rc;
        d.ops[0] = t.rb; d.ops[1] = t.scal;
    } else {
        NaboCbsRef c;
        int rc = nabo_cbs_prepare_ref(r, ldr, n_ref, g, ref_mask, buffer, &c, st);
        if (rc) return rc;
        d.ops[0] = c.rt; d.ops[1] = c.planes; d.ops[2] = c.edges;
    }
    *prepared_host = d;
    return 0;
}

// A descriptor this library prepared, unchanged: NABO_EINVAL otherwise (NABO_EUNSUPPORTED for another ABI version).
static int check_prepared(const nabo_prepared_ref* pr, NaboFastRef* ops) {
    NABO_ARG(pr, "knn_prepared: null descriptor");
    NABO_ARG(pr->magic == NABO_PREPARED_MAGIC, "knn_prepared: not a prepared reference (bad magic)");
    if (pr->abi_version != NABO_ABI_VERSION)
        return nabo_set_error(NABO_EUNSUPPORTED, "knn_prepared: prepared by ABI version %d, this library is %d",
                              pr->abi_version, NABO_ABI_VERSION);
    int plan = 0;
    if (!prepared_plan(pr->g, pr->metric, &plan))
        return nabo_set_error(NABO_EUNSUPPORTED, "knn_prepared: metric %d with g=%d has no fast plan", pr->metric, pr->g);
    NABO_ARG(pr->plan == plan, "knn_prepared: plan %d does not match metric %d", pr->plan, pr->metric);
    NABO_ARG(pr->n_ref >= 1 && pr->ldr >= pr->g, "knn_prepared: bad descriptor sizes");
    NABO_ARG(pr->r && pr->buffer, "knn_prepared: descriptor without rows or buffer");
    NABO_ARG(pr->metric != NABO_CORRELATION || (pr->r == pr->buffer && pr->ldr == pr->g),
             "knn_prepared: the rows of a correlation descriptor must be the centred copy at the start of its buffer");
    NABO_ARG(pr->buffer_bytes >= nabo_ref_prepared_bytes(pr->n_ref, pr->g, pr->metric),
             "knn_prepared: descriptor buffer smaller than its shape needs");
    memset(ops, 0, sizeof(*ops));
    for (int i = 0; i < (plan == NABO_PLAN_TC ? 2 : 3); ++i) {
        const char* a = (const char*)pr->ops[i];
        NABO_ARG(a >= (const char*)pr->buffer && a < (const char*)pr->buffer + pr->buffer_bytes,
                 "knn_prepared: operand %d outside the buffer", i);
    }
    if (plan == NABO_PLAN_TC) {
        ops->tc.rb = pr->ops[0];
        ops->tc.scal = (const double*)pr->ops[1];
    } else {
        ops->cbs.rt = (const float*)pr->ops[0];
        ops->cbs.planes = (const uint32_t*)pr->ops[1];
        ops->cbs.edges = (const float*)pr->ops[2];
    }
    return 0;
}

extern "C" size_t nabo_knn_prepared_workspace_bytes(int n_query, const nabo_prepared_ref* prepared_host, int k,
                                                    double dist_factor, int mode) {
    NaboFastRef ops;
    if (check_prepared(prepared_host, &ops) != 0) return 0;
    const nabo_prepared_ref* pr = prepared_host;
    if (pr->metric == NABO_CORRELATION)
        return corr_head_bytes(n_query, pr->n_ref, pr->g, false) +
               engine_bytes(n_query, pr->n_ref, pr->g, k, NABO_COSINE, mode, true, dist_factor);
    return engine_bytes(n_query, pr->n_ref, pr->g, k, pr->metric, mode, true, dist_factor);
}

static int knn_prepared_impl(const double* q, int ldq, int n_query, const nabo_prepared_ref* pr, int k,
                             double dist_factor, int drop_first, int idx_offset, int mode, int32_t* out_idx,
                             double* out_dist, const NaboRoute& route, void* workspace, size_t workspace_bytes,
                             int64_t* stats_host, void* stream) {
    NaboFastRef ops;
    int rc = check_prepared(pr, &ops);
    if (rc) return rc;
    if (k < 1 || k + (drop_first ? 1 : 0) > 128)
        return nabo_set_error(NABO_EUNSUPPORTED, "knn_prepared: k=%d outside the kNN plans (k + drop_first <= 128)", k);
    return knn_impl(q, ldq, pr->r, pr->ldr, n_query, pr->n_ref, pr->g, k, pr->metric, dist_factor, pr->ref_mask,
                    drop_first, idx_offset, mode, out_idx, out_dist, route, workspace, workspace_bytes, stats_host,
                    stream, &ops);
}

extern "C" int nabo_knn_prepared(const double* q, int ldq, int n_query, const nabo_prepared_ref* prepared_host, int k,
                                 double dist_factor, int drop_first, int idx_offset, int mode, int32_t* out_idx,
                                 double* out_dist, void* workspace, size_t workspace_bytes, int64_t* stats_host,
                                 void* stream) {
    NaboRoute plain;
    plain.n_parts = 0;
    return knn_prepared_impl(q, ldq, n_query, prepared_host, k, dist_factor, drop_first, idx_offset, mode, out_idx,
                             out_dist, plain, workspace, workspace_bytes, stats_host, stream);
}

extern "C" int nabo_knn_prepared_routed(const double* q, int ldq, int n_query, const nabo_prepared_ref* prepared_host,
                                        int k, double dist_factor, int drop_first, int idx_offset, int mode, int n_parts,
                                        const int* part_bounds_host, int32_t* const* part_idx_host,
                                        double* const* part_dist_host, void* workspace, size_t workspace_bytes,
                                        int64_t* stats_host, void* stream) {
    NaboRoute route;
    int rc = parse_route(n_query, n_parts, part_bounds_host, part_idx_host, part_dist_host, route);
    if (rc) return rc;
    return knn_prepared_impl(q, ldq, n_query, prepared_host, k, dist_factor, drop_first, idx_offset, mode, nullptr,
                             nullptr, route, workspace, workspace_bytes, stats_host, stream);
}
