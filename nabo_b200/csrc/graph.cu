// SNN neighbour weights, per-reference mapping scores, target classification and the
// shard merge.  Integer / gather work bounded by HBM, not by any FP pipe.
//   nabo_snn_weights      <- _calc_snn                      nabo/_mapping.py:151-200
//   nabo_mapping_scores   <- Graph.get_mapping_score core   nabo/_graph.py:643-653, 690-693
//   nabo_classify_targets <- Graph.classify_target          nabo/_graph.py:722-792
//   nabo_merge_topk       (reference-sharded mode; result must equal the unsharded top-k)
#include "common.cuh"

#define NABO_MERGE_MAX_SHARDS 16

// ------------------------------------------------------------------ SNN counts + weights
// One warp per query.  A = the query's k neighbours go into a 256- (k <= 32) or 1024-slot open-addressing hash table in
// shared memory; one neighbour's own kNN row per iteration, lanes over its entries (one coalesced row read): an
// entry is a member of A iff a probe sequence of ~1.3 loads finds it, and the row's intersection size is the
// popcount of the warp's hit ballot (no atomics in the counting, no index arithmetic).  The gathers of 16 rows are
// issued back to back before any of them is consumed: the kernel is bound by L2 latency, not by arithmetic.
// multiplicative hash, top bits: shift = 32 - log2(table size)
__device__ __forceinline__ unsigned snn_hash(int v, int shift) { return ((unsigned)v * 2654435761u) >> shift; }

constexpr int SNN_PAD = 32;      // table[tsize] mirrors table[0]: a lookup's second probe needs no wrap

__global__ void __launch_bounds__(256)
snn_kernel(const int32_t* __restrict__ tgt_knn, int n_query, int k, int tsize, int shift, const int32_t* __restrict__ ref_knn,
           int n_ref, int k_ref, int k_use, const double* __restrict__ lut, uint8_t* __restrict__ counts,
           double* __restrict__ weights) {
    extern __shared__ int sm_snn[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int t = blockIdx.x * 8 + warp;
    if (t >= n_query) return;
    const int kp = (k + 31) & ~31;
    int* table = sm_snn + warp * (tsize + SNN_PAD + 2 * kp);   // [tsize (+1)] hash table of A, -1 = empty
    int* a_row = table + tsize + SNN_PAD;                      // [kp] the row in its own order
    int* hits = a_row + kp;                                    // [kp] per-neighbour intersection size
    const unsigned mask = (unsigned)tsize - 1u;
    for (int i = lane; i < tsize; i += 32) table[i] = -1;
    for (int i = lane; i < kp; i += 32) {
        a_row[i] = i < k ? tgt_knn[(long long)t * k + i] : -1;
        hits[i] = 0;
    }
    __syncwarp();
    // insert; the warp remembers the LONGEST displacement of any key, so that a lookup is a fixed number of
    // independent probes (no data-dependent loop, no divergence): 1 + disp slots, disp is 0 or 1 at this load factor
    int disp = 0;
    for (int i = lane; i < kp; i += 32) {
        const int v = a_row[i];
        if (v >= 0) {
            unsigned s_ = snn_hash(v, shift);
            int dd = 0;
            for (;;) {
                const int old = atomicCAS(&table[s_], -1, v);
                if (old == -1 || old == v) break;
                s_ = (s_ + 1) & mask;
                ++dd;
            }
            disp = max(disp, dd);
        }
        if (!(v >= 0 && v < n_ref)) a_row[i] = -1;       // from here on a_row holds the rows of ref_knn to walk
    }
    disp = __reduce_max_sync(0xffffffffu, disp);
    __syncwarp();
    if (lane == 0) table[tsize] = table[0];
    __syncwarp();
    // the ballot count of a row is warp-uniform: row r0 + u of a block of 16 accumulates in lane (r0 & 31) + u
    for (int c0 = 0; c0 < k_use; c0 += 32) {
        const int col = c0 + lane;
        const bool col_ok = col < k_use;
        const int32_t* colp = ref_knn + col;
        for (int r0 = 0; r0 < k; r0 += 16) {
            int bv[16];                                   // -2 = nothing to look up (never equals a key or an empty slot)
#pragma unroll
            for (int u = 0; u < 16; ++u) {
                const int j = a_row[r0 + u];              // r0 + u < kp
                const int raw = (j >= 0 && col_ok) ? __ldg(colp + (size_t)j * k_ref) : -2;
                bv[u] = raw >= 0 ? raw : -2;               // a missing neighbour (-1) must not match an empty slot
            }
            const int base = r0 & 31;
            int blk = 0;
            if (disp <= 1) {
#pragma unroll
                for (int u = 0; u < 16; ++u) {
                    const int b = bv[u];
                    const unsigned s_ = snn_hash(b, shift);
                    const bool hit = (table[s_] == b) | (table[s_ + 1] == b);
                    const int cnt = __popc(__ballot_sync(0xffffffffu, hit));
                    if (lane == base + u) blk += cnt;
                }
            } else {
#pragma unroll 1
                for (int u = 0; u < 16; ++u) {
                    int b = bv[0];
#pragma unroll
                    for (int w = 1; w < 16; ++w) b = (w == u) ? bv[w] : b;
                    const unsigned s_ = snn_hash(b, shift);
                    bool hit = false;
                    for (int dd = 0; dd <= disp; ++dd) hit |= table[(s_ + dd) & mask] == b;
                    const int cnt = __popc(__ballot_sync(0xffffffffu, hit));
                    if (lane == base + u) blk += cnt;
                }
            }
            const int mine = r0 + lane - base;
            if (lane >= base && lane < base + 16 && mine < k) hits[mine] += blk;
        }
    }
    __syncwarp();
    for (int i = lane; i < k; i += 32) {
        const int c = hits[i];
        if (counts) counts[(long long)t * k + i] = (uint8_t)c;
        if (weights) weights[(long long)t * k + i] = lut[c];
    }
}

extern "C" int nabo_snn_weights(const int32_t* tgt_knn, int n_query, int k, const int32_t* ref_knn, int n_ref,
                                int k_ref, const double* lut, uint8_t* out_counts, double* out_weights,
                                void* stream) {
    NABO_ARG(k >= 1 && k <= 255 && k_ref >= 1, "snn: k=%d k_ref=%d unsupported (1..255)", k, k_ref);
    NABO_ARG(n_query >= 0 && n_ref >= 1, "snn: bad sizes");
    if (n_query == 0) return 0;
    NABO_ARG(tgt_knn && ref_knn && (out_counts || out_weights), "snn: null pointer");
    NABO_ARG(!out_weights || lut, "snn: weights requested without a lut");
    int k_use = k < k_ref ? k : k_ref;   // ref_data[ref_c][:k], _mapping.py:193
    const int tsize = k <= 32 ? 256 : 1024;          // load factor <= 1/4: the warp walks the LONGEST probe sequence of its lanes
    const int shift = k <= 32 ? 24 : 22;             // 32 - log2(tsize)
    const int kp = (k + 31) & ~31;
    snn_kernel<<<(n_query + 7) / 8, 256, 8 * (tsize + SNN_PAD + 2 * kp) * sizeof(int), (cudaStream_t)stream>>>(
        tgt_knn, n_query, k, tsize, shift, ref_knn, n_ref, k_ref, k_use, lut, out_counts, out_weights);
    NABO_LAUNCH_CHECK("snn_kernel");
    return 0;
}

// ------------------------------------------------------------------ stable LSD radix sort (keys u32, payload u32)
constexpr int RS_THREADS = 256;
constexpr int RS_ROUNDS = 8;
constexpr int RS_BLOCK = RS_THREADS * RS_ROUNDS;   // elements per block, order = (round, thread)

__global__ void __launch_bounds__(RS_THREADS)
rs_hist_kernel(const uint32_t* __restrict__ keys, int n, int shift, uint32_t* __restrict__ hist, int nblocks) {
    __shared__ uint32_t h[256];
    h[threadIdx.x] = 0;
    __syncthreads();
    const long long base = (long long)blockIdx.x * RS_BLOCK;
    for (int r = 0; r < RS_ROUNDS; ++r) {
        long long i = base + r * RS_THREADS + threadIdx.x;
        if (i < n) atomicAdd(&h[(keys[i] >> shift) & 255u], 1u);
    }
    __syncthreads();
    hist[(size_t)threadIdx.x * nblocks + blockIdx.x] = h[threadIdx.x];   // digit-major
}

// Exclusive scan of the digit-major counter matrix hist[256][nblocks] in two parallel steps:
//   (1) one block per digit: exclusive scan of that digit's row, row total -> totals[d]
//   (2) the scatter kernel adds the exclusive prefix of totals[] (256 values, scanned per block there)
__global__ void __launch_bounds__(256) rs_scan_rows_kernel(uint32_t* __restrict__ hist, int nblocks,
                                                           uint32_t* __restrict__ totals) {
    __shared__ uint32_t warp_sum[8];
    __shared__ uint32_t carry_s;
    uint32_t* row = hist + (size_t)blockIdx.x * nblocks;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) carry_s = 0;
    __syncthreads();
    for (int base = 0; base < nblocks; base += 256) {
        const int i = base + threadIdx.x;
        const uint32_t v = i < nblocks ? row[i] : 0;
        uint32_t incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t u = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += u;
        }
        if (lane == 31) warp_sum[warp] = incl;
        __syncthreads();
        uint32_t before = carry_s;
        for (int w = 0; w < warp; ++w) before += warp_sum[w];
        if (i < nblocks) row[i] = before + incl - v;
        __syncthreads();
        if (threadIdx.x == 255) carry_s = before + incl;
        __syncthreads();
    }
    if (threadIdx.x == 0) totals[blockIdx.x] = carry_s;
}

__global__ void __launch_bounds__(RS_THREADS)
rs_scatter_kernel(const uint32_t* __restrict__ keys, const uint32_t* __restrict__ vals, int n, int shift,
                  const uint32_t* __restrict__ offs, const uint32_t* __restrict__ totals, int nblocks,
                  uint32_t* __restrict__ okeys, uint32_t* __restrict__ ovals) {
    __shared__ uint32_t running[256];           // elements of each digit placed by earlier rounds
    __shared__ uint16_t wcnt[RS_THREADS / 32][256];
    __shared__ uint32_t wtot[RS_THREADS / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    {   // exclusive prefix of the 256 digit totals (thread = digit)
        const uint32_t v = totals[threadIdx.x];
        uint32_t incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t u = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += u;
        }
        if (lane == 31) wtot[warp] = incl;
        __syncthreads();
        uint32_t before = 0;
        for (int w = 0; w < warp; ++w) before += wtot[w];
        running[threadIdx.x] = before + incl - v + offs[(size_t)threadIdx.x * nblocks + blockIdx.x];
    }
    const long long base = (long long)blockIdx.x * RS_BLOCK;
    for (int r = 0; r < RS_ROUNDS; ++r) {
        for (int w = 0; w < RS_THREADS / 32; ++w) wcnt[w][threadIdx.x] = 0;
        __syncthreads();
        const long long i = base + r * RS_THREADS + threadIdx.x;
        const bool live = i < n;
        uint32_t key = live ? keys[i] : 0xFFFFFFFFu;
        uint32_t val = live ? vals[i] : 0u;
        const uint32_t digit = live ? ((key >> shift) & 255u) : 256u;   // 256 = idle lane group
        const uint32_t peers = __match_any_sync(0xffffffffu, digit);
        const int rank_in_warp = __popc(peers & ((1u << lane) - 1u));
        if (live && rank_in_warp == 0) wcnt[warp][digit] = (uint16_t)__popc(peers);
        __syncthreads();
        if (live) {
            uint32_t before = 0;
            for (int w = 0; w < warp; ++w) before += wcnt[w][digit];
            const uint32_t pos = running[digit] + before + rank_in_warp;
            okeys[pos] = key;
            ovals[pos] = val;
        }
        __syncthreads();
        {
            uint32_t tot = 0;
            for (int w = 0; w < RS_THREADS / 32; ++w) tot += wcnt[w][threadIdx.x];
            running[threadIdx.x] += tot;
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------ mapping scores
__global__ void __launch_bounds__(256)
score_edges_kernel(const int32_t* __restrict__ tgt_knn, const uint8_t* __restrict__ counts,
                   const double* __restrict__ lut, long long n_edges, int k, int n_ref,
                   const uint8_t* __restrict__ include, double min_weight, int weighted,
                   uint32_t* __restrict__ keys, uint32_t* __restrict__ vals) {
    long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_edges) return;
    const int t = (int)(e / k);
    const int r = tgt_knn[e];
    const int c = counts[e];
    bool keep = c > 0 && r >= 0 && r < n_ref && (!include || include[t]);
    if (keep && weighted) keep = lut[c] > min_weight;      // _graph.py:647-648
    keys[e] = keep ? (uint32_t)r : (uint32_t)n_ref;         // dropped edges sort past every reference
    vals[e] = (uint32_t)e;
}

__global__ void __launch_bounds__(256)
score_reduce_kernel(const uint32_t* __restrict__ keys, const uint32_t* __restrict__ vals, long long n_edges,
                    const uint8_t* __restrict__ counts, const double* __restrict__ lut, int n_ref,
                    int weighted, double mult, double denom, double min_score, double* __restrict__ out) {
    int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_ref) return;
    // lower_bound(keys, r)
    long long lo = 0, hi = n_edges;
    while (lo < hi) {
        long long mid = (lo + hi) >> 1;
        if (keys[mid] < (uint32_t)r) lo = mid + 1; else hi = mid;
    }
    double acc = 0.0;
    for (long long p = lo; p < n_edges && keys[p] == (uint32_t)r; ++p) {
        // edges arrive in target order (stable sort of a target-major list) = the
        // reference's adjacency insertion order
        acc = weighted ? __dadd_rn(acc, lut[counts[vals[p]]]) : __dadd_rn(acc, 1.0);
    }
    double v = __ddiv_rn(__dmul_rn(mult, acc), denom);       // score_multiplier * v / len(include_nodes)
    out[r] = v >= min_score ? v : 0.0;
}

extern "C" size_t nabo_scores_workspace_bytes(int n_query, int k, int n_ref) {
    size_t e = (size_t)n_query * (size_t)k;
    size_t nblocks = (e + RS_BLOCK - 1) / RS_BLOCK;
    (void)n_ref;
    return 4 * nabo_align_up(e * sizeof(uint32_t), 256) + nabo_align_up(256 * nblocks * sizeof(uint32_t), 256) + 4096;
}

extern "C" int nabo_mapping_scores(const int32_t* tgt_knn, const uint8_t* counts, const double* lut, int n_query,
                                   int k, int n_ref, const uint8_t* include, int n_include, double min_weight,
                                   int weighted, double score_multiplier, double min_score, double* out_scores,
                                   void* workspace, size_t workspace_bytes, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    NABO_ARG(n_query >= 0 && k >= 1 && n_ref >= 1, "scores: bad sizes");
    NABO_ARG((long long)n_query * k < (1ll << 31), "scores: more than 2^31 edges in one call; shard the targets");
    NABO_ARG(out_scores && (n_query == 0 || (tgt_knn && counts && lut)), "scores: null pointer");
    NABO_ARG(n_include > 0 || n_query == 0, "scores: n_include must be positive");
    if (n_query == 0) {
        NABO_CUDA(cudaMemsetAsync(out_scores, 0, sizeof(double) * n_ref, st));
        return 0;
    }
    const long long e = (long long)n_query * k;
    const int nblocks = (int)((e + RS_BLOCK - 1) / RS_BLOCK);
    if (workspace_bytes < nabo_scores_workspace_bytes(n_query, k, n_ref))
        return nabo_set_error(NABO_EWORKSPACE, "scores: workspace too small (%zu < %zu)", workspace_bytes,
                              nabo_scores_workspace_bytes(n_query, k, n_ref));
    NaboArena ar(workspace, workspace_bytes);
    uint32_t* k0 = ar.take<uint32_t>(e);
    uint32_t* v0 = ar.take<uint32_t>(e);
    uint32_t* k1 = ar.take<uint32_t>(e);
    uint32_t* v1 = ar.take<uint32_t>(e);
    uint32_t* hist = ar.take<uint32_t>((size_t)256 * nblocks);
    uint32_t* totals = ar.take<uint32_t>(256);
    if (!ar.ok) return nabo_set_error(NABO_EWORKSPACE, "scores: workspace too small");
    score_edges_kernel<<<(unsigned)((e + 255) / 256), 256, 0, st>>>(tgt_knn, counts, lut, e, k, n_ref, include,
                                                                   min_weight, weighted, k0, v0);
    NABO_LAUNCH_CHECK("score_edges_kernel");
    int bits = 1;
    while ((1ll << bits) <= n_ref) ++bits;          // keys go up to n_ref inclusive
    for (int shift = 0; shift < bits; shift += 8) {
        rs_hist_kernel<<<nblocks, RS_THREADS, 0, st>>>(k0, (int)e, shift, hist, nblocks);
        rs_scan_rows_kernel<<<256, 256, 0, st>>>(hist, nblocks, totals);
        rs_scatter_kernel<<<nblocks, RS_THREADS, 0, st>>>(k0, v0, (int)e, shift, hist, totals, nblocks, k1, v1);
        NABO_LAUNCH_CHECK("radix pass");
        uint32_t* t = k0; k0 = k1; k1 = t;
        t = v0; v0 = v1; v1 = t;
    }
    score_reduce_kernel<<<(n_ref + 255) / 256, 256, 0, st>>>(k0, v0, e, counts, lut, n_ref, weighted,
                                                             score_multiplier, (double)n_include, min_score,
                                                             out_scores);
    NABO_LAUNCH_CHECK("score_reduce_kernel");
    return 0;
}

// ------------------------------------------------------------------ classify_target
__global__ void __launch_bounds__(128)
classify_kernel(const int32_t* __restrict__ tgt_knn, const uint8_t* __restrict__ counts,
                const double* __restrict__ lut, int n_query, int k, const int32_t* __restrict__ ref_labels,
                int n_labels, double weight_frac, int min_degree, double min_weight,
                int32_t* __restrict__ out) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_query) return;
    const int32_t* nb = tgt_knn + (long long)t * k;
    const uint8_t* cn = counts + (long long)t * k;
    int deg = 0;
    double tot = 0.0;
    for (int j = 0; j < k; ++j)
        if (cn[j] > 0 && nb[j] >= 0) { ++deg; tot = __dadd_rn(tot, lut[cn[j]]); }   // every edge counts (:771)
    int best = -1;
    double best_w = -1.0;
    if (deg >= min_degree) {
        for (int j = 0; j < k; ++j) {
            if (!(cn[j] > 0 && nb[j] >= 0)) continue;
            const double wj = lut[cn[j]];
            if (!(wj > min_weight)) continue;
            const int lab = ref_labels[nb[j]];
            if (lab < 0 || lab >= n_labels) continue;
            bool first = true;
            for (int i = 0; i < j; ++i)
                if (cn[i] > 0 && nb[i] >= 0 && lut[cn[i]] > min_weight && ref_labels[nb[i]] == lab) { first = false; break; }
            if (!first) continue;
            double s = 0.0;
            for (int i = j; i < k; ++i)
                if (cn[i] > 0 && nb[i] >= 0 && lut[cn[i]] > min_weight && ref_labels[nb[i]] == lab)
                    s = __dadd_rn(s, lut[cn[i]]);
            if (s > best_w || (s == best_w && lab < best)) { best_w = s; best = lab; }
        }
        if (best < 0) {          // no voting edge: every cluster has weight 0; argmax -> label 0
            best = n_labels > 0 ? 0 : -1;
            best_w = 0.0;
        }
        if (!(best_w > __dmul_rn(weight_frac, tot))) best = -1;
    }
    out[t] = best;
}

extern "C" int nabo_classify_targets(const int32_t* tgt_knn, const uint8_t* counts, const double* lut, int n_query,
                                     int k, const int32_t* ref_labels, int n_labels, double weight_frac,
                                     int min_degree, double min_weight, int32_t* out_label, void* stream) {
    NABO_ARG(n_query >= 0 && k >= 1, "classify: bad sizes");
    if (n_query == 0) return 0;
    NABO_ARG(tgt_knn && counts && lut && ref_labels && out_label, "classify: null pointer");
    classify_kernel<<<(n_query + 127) / 128, 128, 0, (cudaStream_t)stream>>>(
        tgt_knn, counts, lut, n_query, k, ref_labels, n_labels, weight_frac, min_degree, min_weight, out_label);
    NABO_LAUNCH_CHECK("classify_kernel");
    return 0;
}

// ------------------------------------------------------------------ shard merge
// One warp per query: the k-lists of all shards (one (n_query x k) idx / dist block per shard, anywhere in
// device-visible memory: slices of an all-gather result or the per-source blocks of an all-to-all / peer-written
// receive buffer, consumed in place) are sorted by (distance, index) in shared memory.
struct MergeParts {
    const int32_t* idx[NABO_MERGE_MAX_SHARDS];
    const double* dist[NABO_MERGE_MAX_SHARDS];
};

__global__ void __launch_bounds__(128)
merge_kernel(const MergeParts parts, int n_shards, int n_query, int k, int capp, int drop_first,
             int32_t* __restrict__ out_idx, double* __restrict__ out_dist) {
    extern __shared__ double smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int qi = blockIdx.x * 4 + warp;
    if (qi >= n_query) return;
    double* d = smem + (size_t)warp * capp;
    int* ix = (int*)(smem + (size_t)4 * capp) + (size_t)warp * capp;
    const int tot = n_shards * k;
    for (int c = lane; c < capp; c += 32) {
        double dv = CUDART_INF;
        int id = 0x7fffffff;
        if (c < tot) {
            const int s = c / k, j = c - s * k;
            const long long off = (long long)qi * k + j;
            const int i0 = parts.idx[s][off];
            if (i0 >= 0) {
                id = i0;
                dv = parts.dist[s][off];
                if (dv != dv) dv = CUDART_INF;
            }
        }
        d[c] = dv; ix[c] = id;
    }
    __syncwarp();
    warp_bitonic_sort(d, ix, capp, lane);
    const int ko = k - drop_first;                          // drop_first: the global "self" entry goes after the merge
    for (int t = lane; t < ko; t += 32) {
        int id = ix[t + drop_first];
        double dv = d[t + drop_first];
        if (id == 0x7fffffff) { id = -1; dv = CUDART_NAN; }
        else if (dv == CUDART_INF) dv = CUDART_NAN;
        out_idx[(long long)qi * ko + t] = id;
        out_dist[(long long)qi * ko + t] = dv;
    }
}

static int merge_launch(const MergeParts& parts, int n_shards, int n_query, int k, int drop_first, int32_t* out_idx,
                        double* out_dist, cudaStream_t st) {
    int capp = nabo_next_pow2(n_shards * k);
    if (capp < 32) capp = 32;
    size_t smem = (size_t)4 * capp * (sizeof(double) + sizeof(int));
    NABO_CUDA(cudaFuncSetAttribute(merge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    merge_kernel<<<(n_query + 3) / 4, 128, smem, st>>>(parts, n_shards, n_query, k, capp, drop_first ? 1 : 0, out_idx,
                                                       out_dist);
    NABO_LAUNCH_CHECK("merge_kernel");
    return 0;
}

extern "C" int nabo_merge_topk(const int32_t* idx, const double* dist, int n_shards, int n_query, int k,
                               int32_t* out_idx, double* out_dist, void* stream) {
    NABO_ARG(n_shards >= 1 && n_shards <= NABO_MERGE_MAX_SHARDS && k >= 1 && n_query >= 0, "merge: bad sizes");
    NABO_ARG((long long)n_shards * k <= 2048, "merge: n_shards*k=%d exceeds 2048", n_shards * k);
    if (n_query == 0) return 0;
    NABO_ARG(idx && dist && out_idx && out_dist, "merge: null pointer");
    MergeParts parts;
    for (int s = 0; s < n_shards; ++s) {
        parts.idx[s] = idx + (size_t)s * n_query * k;
        parts.dist[s] = dist + (size_t)s * n_query * k;
    }
    return merge_launch(parts, n_shards, n_query, k, 0, out_idx, out_dist, (cudaStream_t)stream);
}

extern "C" int nabo_merge_topk_parts(int n_shards, const int32_t* const* shard_idx_host,
                                     const double* const* shard_dist_host, int n_query, int k, int drop_first,
                                     int32_t* out_idx, double* out_dist, void* stream) {
    NABO_ARG(n_shards >= 1 && n_shards <= NABO_MERGE_MAX_SHARDS && k >= 1 && n_query >= 0, "merge_parts: bad sizes");
    NABO_ARG((long long)n_shards * k <= 2048, "merge_parts: n_shards*k=%d exceeds 2048", n_shards * k);
    NABO_ARG(!drop_first || k >= 2, "merge_parts: drop_first needs k >= 2");
    if (n_query == 0) return 0;
    NABO_ARG(shard_idx_host && shard_dist_host && out_idx && out_dist, "merge_parts: null pointer");
    MergeParts parts;
    for (int s = 0; s < n_shards; ++s) {
        NABO_ARG(shard_idx_host[s] && shard_dist_host[s], "merge_parts: shard %d has no buffers", s);
        parts.idx[s] = shard_idx_host[s];
        parts.dist[s] = shard_dist_host[s];
    }
    return merge_launch(parts, n_shards, n_query, k, drop_first, out_idx, out_dist, (cudaStream_t)stream);
}

// ------------------------------------------------------------------ GPU-count-independent mapping scores
// Every SNN weight is one of k + 1 table values, so the sum over a reference cell's edges is an INTEGER
// combination of them: acc[r] += iw[counts] with iw = the table in integer units (for the reference's table,
// round(w, 2) in hundredths: exact).  Integer atomics commute, so acc - and with it the score - has the same
// bits for any launch geometry, any order of target batches and any number of GPUs (acc is what the sharded
// modes all-reduce, as int64).  nabo_mapping_scores (sorted, target order) stays the single-GPU default of the
// Graph facade; the two agree to ~1e-15 relative (one rounding here, one per edge there).
__global__ void __launch_bounds__(256)
score_accumulate_kernel(const int32_t* __restrict__ tgt_knn, const uint8_t* __restrict__ counts,
                        const long long* __restrict__ iw, long long n_edges, int k, int n_ref,
                        const uint8_t* __restrict__ include, unsigned long long* __restrict__ acc) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_edges) return;
    const int c = counts[e];
    if (c == 0) return;
    const int r = tgt_knn[e];
    if (r < 0 || r >= n_ref) return;
    if (include && !include[e / k]) return;
    const long long w = iw[c];
    if (w != 0) atomicAdd(acc + r, (unsigned long long)w);
}

__global__ void __launch_bounds__(256)
score_finalize_kernel(const long long* __restrict__ acc, int n_ref, double unit, double mult, double denom,
                      double min_score, double* __restrict__ out) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_ref) return;
    const double sum = __ddiv_rn((double)acc[r], unit);           // exact integer / units per 1.0
    const double v = __ddiv_rn(__dmul_rn(mult, sum), denom);
    out[r] = v >= min_score ? v : 0.0;
}

extern "C" int nabo_score_accumulate(const int32_t* tgt_knn, const uint8_t* counts, const long long* int_weights,
                                     int n_query, int k, int n_ref, const uint8_t* include, long long* acc,
                                     void* stream) {
    NABO_ARG(n_query >= 0 && k >= 1 && n_ref >= 1, "score_accumulate: bad sizes");
    if (n_query == 0) return 0;
    NABO_ARG(tgt_knn && counts && int_weights && acc, "score_accumulate: null pointer");
    const long long e = (long long)n_query * k;
    score_accumulate_kernel<<<(unsigned)((e + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        tgt_knn, counts, int_weights, e, k, n_ref, include, (unsigned long long*)acc);
    NABO_LAUNCH_CHECK("score_accumulate_kernel");
    return 0;
}

extern "C" int nabo_scores_finalize(const long long* acc, int n_ref, double units_per_one, double score_multiplier,
                                    long long n_include, double min_score, double* out_scores, void* stream) {
    NABO_ARG(n_ref >= 1 && units_per_one > 0.0 && n_include > 0, "scores_finalize: bad arguments");
    NABO_ARG(acc && out_scores, "scores_finalize: null pointer");
    score_finalize_kernel<<<(n_ref + 255) / 256, 256, 0, (cudaStream_t)stream>>>(acc, n_ref, units_per_one,
                                                                               score_multiplier, (double)n_include,
                                                                               min_score, out_scores);
    NABO_LAUNCH_CHECK("score_finalize_kernel");
    return 0;
}

// ------------------------------------------------------------------ connected components
// Labels of the connected components of an undirected graph given as an edge list: union-find with
// atomicMin hooking (the root with the larger id is hooked under the smaller one) and path halving, swept
// over the edges until a sweep changes nothing; label[i] = smallest node id of i's component, so the
// result does not depend on scheduling.  Used by the reference-graph repair (_fix_disconnected_graph,
// nabo/_mapping.py:203-249, works on nx.connected_components).
__device__ __forceinline__ int cc_find(int* parent, int x) {
    int p = parent[x];
    while (p != x) {
        const int gp = parent[p];
        if (gp != p) parent[x] = gp;          // path halving (benign race: every written value is an ancestor)
        x = p;
        p = gp;
    }
    return x;
}

__global__ void cc_init_kernel(int* parent, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) parent[i] = i;
}

__global__ void cc_hook_kernel(const int32_t* __restrict__ ea, const int32_t* __restrict__ eb, long long n_edges,
                               int n_nodes, int* parent, int* changed) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_edges) return;
    const int a = ea[e], b = eb[e];
    if (a < 0 || b < 0 || a >= n_nodes || b >= n_nodes || a == b) return;
    int ra = cc_find(parent, a), rb = cc_find(parent, b);
    while (ra != rb) {
        const int hi = ra > rb ? ra : rb, lo = ra > rb ? rb : ra;
        const int old = atomicMin(&parent[hi], lo);
        if (old == hi) { *changed = 1; break; }       // hooked a root
        ra = cc_find(parent, old);                     // hi was no longer a root: retry from its new parent
        rb = lo;
        *changed = 1;
    }
}

__global__ void cc_flatten_kernel(int* parent, int n, int32_t* labels) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) labels[i] = cc_find(parent, i);
}

extern "C" int nabo_connected_components(const int32_t* edge_a, const int32_t* edge_b, long long n_edges, int n_nodes,
                                         int32_t* out_labels, void* workspace, size_t workspace_bytes, void* stream) {
    NABO_ARG(n_nodes >= 1 && n_edges >= 0, "connected_components: bad sizes");
    NABO_ARG(out_labels && (n_edges == 0 || (edge_a && edge_b)), "connected_components: null pointer");
    if (workspace == nullptr || workspace_bytes < (size_t)n_nodes * sizeof(int) + 256)
        return nabo_set_error(NABO_EWORKSPACE, "connected_components: workspace too small (need %zu bytes)",
                              (size_t)n_nodes * sizeof(int) + 256);
    cudaStream_t st = (cudaStream_t)stream;
    int* parent = (int*)workspace;
    int* changed = (int*)((char*)workspace + nabo_align_up((size_t)n_nodes * sizeof(int), 256));
    cc_init_kernel<<<(n_nodes + 255) / 256, 256, 0, st>>>(parent, n_nodes);
    NABO_LAUNCH_CHECK("cc_init_kernel");
    for (int sweep = 0; sweep < 64 && n_edges > 0; ++sweep) {
        int h = 0;
        NABO_CUDA(cudaMemsetAsync(changed, 0, sizeof(int), st));
        cc_hook_kernel<<<(unsigned)((n_edges + 255) / 256), 256, 0, st>>>(edge_a, edge_b, n_edges, n_nodes, parent, changed);
        NABO_LAUNCH_CHECK("cc_hook_kernel");
        NABO_CUDA(cudaMemcpyAsync(&h, changed, sizeof(int), cudaMemcpyDeviceToHost, st));
        NABO_CUDA(cudaStreamSynchronize(st));
        if (!h) break;
    }
    cc_flatten_kernel<<<(n_nodes + 255) / 256, 256, 0, st>>>(parent, n_nodes, out_labels);
    NABO_LAUNCH_CHECK("cc_flatten_kernel");
    return 0;
}
