// Mapping specificity (nabo/_graph.py:794-824): for every target cell, the mean of the unweighted
// shortest-path lengths, in the reference graph, between all pairs of reference cells it maps to.
// The reference runs one networkx BFS per pair (k(k-1)/2 per target); here ONE bit-parallel multi-source
// search per target finds all pair distances at once:
//
//   * source i of the target owns bit i of a W-word mask (W = 1 up to 64 sources, W = 2 up to 128; bit i is
//     bit i % 64 of word i / 64); cur[v] = sources whose ball contains node v;
//   * level L: every frontier node u pushes the bits that reached it at level L-1 (delta[u]) to its
//     neighbours: acc[v] |= delta[u] & ~cur[v]; v joins the next frontier once per level (W = 1: the writer
//     whose atomicOr found acc zero; W = 2: the writer that swaps the level into v's stamp);
//   * commit: delta[v] = acc[v] & ~cur[v].  All balls grow in lock step, so the first time bit i arrives
//     at a node that already holds bit j the pair is 2L - 1 apart, and two bits arriving together are 2L
//     apart (pass A before pass B, so the shorter meeting always wins): every pair is settled after
//     ceil(d / 2) levels - the balls stay small - instead of the d levels a one-sided search needs;
//   * a source that has met every partner stops propagating; the search ends when all k(k-1)/2 pairs
//     are settled (or the frontier dies: no path, reported to the host, where the reference would raise
//     NetworkXNoPath).
//
// One CTA per target at a time, persistent over the targets; per-CTA scratch (cur, acc, frontier lists)
// lives in the caller's workspace and is cleaned by walking the list of touched nodes, so the arrays are
// zero again when the next target starts.  Integer outputs (sum of distances, pairs found): exact and
// independent of scheduling.
#include "common.cuh"

namespace spec {

constexpr int NT = 256;
constexpr int MAXK = 128;

// W words of source bits; W = 2 is 16-byte aligned so that a node's mask is one load or store
template <int W>
struct alignas(8 * W) Mask {
    unsigned long long w[W];
};

template <int W>
__device__ __forceinline__ Mask<W> operator&(Mask<W> a, const Mask<W>& b) {
#pragma unroll
    for (int i = 0; i < W; ++i) a.w[i] &= b.w[i];
    return a;
}
template <int W>
__device__ __forceinline__ Mask<W> operator|(Mask<W> a, const Mask<W>& b) {
#pragma unroll
    for (int i = 0; i < W; ++i) a.w[i] |= b.w[i];
    return a;
}
template <int W>
__device__ __forceinline__ Mask<W> and_not(Mask<W> a, const Mask<W>& b) {
#pragma unroll
    for (int i = 0; i < W; ++i) a.w[i] &= ~b.w[i];
    return a;
}
template <int W>
__device__ __forceinline__ bool any(const Mask<W>& a) {
    unsigned long long o = a.w[0];
#pragma unroll
    for (int i = 1; i < W; ++i) o |= a.w[i];
    return o != 0ull;
}
template <int W>
__device__ __forceinline__ bool two_or_more(const Mask<W>& a) {
    if constexpr (W == 1) return (a.w[0] & (a.w[0] - 1)) != 0ull;
    else return ((a.w[0] & (a.w[0] - 1)) | (a.w[1] & (a.w[1] - 1))) != 0ull || (a.w[0] != 0ull && a.w[1] != 0ull);
}
// source i alone
template <int W>
__device__ __forceinline__ Mask<W> single(int i) {
    Mask<W> m;
    if constexpr (W == 1) m.w[0] = 1ull << i;
    else { m.w[0] = i < 64 ? 1ull << i : 0ull; m.w[1] = i < 64 ? 0ull : 1ull << (i - 64); }
    return m;
}
// index of the lowest set bit of a non-empty mask, which is cleared
template <int W>
__device__ __forceinline__ int pop_lowest(Mask<W>& a) {
    if constexpr (W == 1) {
        const int i = __ffsll((long long)a.w[0]) - 1;
        a.w[0] &= a.w[0] - 1;
        return i;
    } else {
        if (a.w[0]) {
            const int i = __ffsll((long long)a.w[0]) - 1;
            a.w[0] &= a.w[0] - 1;
            return i;
        }
        const int i = __ffsll((long long)a.w[1]) - 1;
        a.w[1] &= a.w[1] - 1;
        return 64 + i;
    }
}

template <int W>
struct Scratch {
    Mask<W>* cur;                // [m]
    Mask<W>* acc;                // [m]
    Mask<W>* dl[2];              // [m] delta of the frontier entries (parallel to fr[])
    int* fr[2];                  // [m] frontier node lists
    int* touched;                // [m]
    uint8_t* tpos;               // [m] 0 = not a mapped cell of the current target, else position + 1
};

// per node: cur, acc, two deltas (8 W bytes each), two frontier entries, touched, tpos; W = 2 adds the int
// enqueue stamp (the level at which the node last joined a frontier).  45 bytes at W = 1, 81 at W = 2.
static size_t scratch_bytes(int m, int W) {
    const size_t mm = nabo_align_up((size_t)m, 64);
    return mm * (32 * W + 8 + 4 + 1 + (W > 1 ? 4 : 0)) + 1024;
}

static int words_for(int k) { return k <= 64 ? 1 : 2; }

template <int W>
__global__ void __launch_bounds__(NT)
specificity_kernel(const long long* __restrict__ indptr, const int32_t* __restrict__ indices, int m,
                   const int32_t* __restrict__ tgt_knn, const uint8_t* __restrict__ counts, int n_query, int k,
                   long long* __restrict__ out_sum, int32_t* __restrict__ out_pairs, int32_t* __restrict__ out_nmapped,
                   unsigned char* __restrict__ ws, size_t per_block) {
    constexpr int NS = 64 * W;                    // sources a target can have
    __shared__ int s_src[NS];
    __shared__ int s_nt, s_nf[2], s_ntouched;
    __shared__ unsigned long long s_sum;
    __shared__ int s_pairs;
    __shared__ Mask<W> s_found[NS];               // s_found[lo] bit hi: pair {lo, hi} has its distance (lo < hi)
    __shared__ int s_nfound[NS];                  // partners found per source
    __shared__ Mask<W> s_active;                  // sources still missing a partner: only their bits keep travelling

    Scratch<W> sc;
    int* stamp = nullptr;                         // [m], W = 2 only
    {
        const size_t mm = ((size_t)m + 63) / 64 * 64;
        unsigned char* b = ws + (size_t)blockIdx.x * per_block;
        sc.cur = reinterpret_cast<Mask<W>*>(b); b += mm * 8 * W;
        sc.acc = reinterpret_cast<Mask<W>*>(b); b += mm * 8 * W;
        sc.dl[0] = reinterpret_cast<Mask<W>*>(b); b += mm * 8 * W;
        sc.dl[1] = reinterpret_cast<Mask<W>*>(b); b += mm * 8 * W;
        sc.fr[0] = reinterpret_cast<int*>(b); b += mm * 4;
        sc.fr[1] = reinterpret_cast<int*>(b); b += mm * 4;
        sc.touched = reinterpret_cast<int*>(b); b += mm * 4;
        if constexpr (W > 1) { stamp = reinterpret_cast<int*>(b); b += mm * 4; }
        sc.tpos = b;
    }

    // pair {i, j} met with total path length dist: count it once
    auto record = [&](int i, int j, int dist) {
        const int lo = i < j ? i : j, hi = i < j ? j : i;
        const unsigned long long bit = 1ull << (W == 1 ? hi : hi & 63);
        if (!(atomicOr(&s_found[lo].w[W == 1 ? 0 : hi >> 6], bit) & bit)) {
            atomicAdd(&s_sum, (unsigned long long)dist);
            atomicAdd(&s_pairs, 1);
            atomicAdd(&s_nfound[lo], 1);
            atomicAdd(&s_nfound[hi], 1);
        }
    };

    for (int t = blockIdx.x; t < n_query; t += gridDim.x) {
        // ---- the target's mapped reference cells = its edges (snn count > 0), nabo/_mapping.py:195-198
        if (threadIdx.x == 0) {
            int nt = 0;
            for (int j = 0; j < k; ++j) {
                const int r = tgt_knn[(size_t)t * k + j];
                if (r >= 0 && r < m && counts[(size_t)t * k + j] > 0) s_src[nt++] = r;
            }
            s_nt = nt;
            s_sum = 0ull;
            s_pairs = 0;
            s_nf[0] = nt;
            s_nf[1] = 0;
            s_ntouched = nt;
#pragma unroll
            for (int w = 0; w < W; ++w) {
                const int r = nt - 64 * w;                              // sources in word w (clamped below)
                s_active.w[w] = (w > 0 && r <= 0) ? 0ull : r >= 64 ? ~0ull : ((1ull << r) - 1ull);
            }
        }
        if (threadIdx.x < NS) { s_found[threadIdx.x] = Mask<W>{}; s_nfound[threadIdx.x] = 0; }
        __syncthreads();
        const int nt = s_nt;
        if (nt < 2) {
            if (threadIdx.x == 0) { out_sum[t] = 0; out_pairs[t] = 0; out_nmapped[t] = nt; }
            __syncthreads();
            continue;
        }
        if (threadIdx.x < nt) {
            const int v = s_src[threadIdx.x];
            sc.cur[v] = single<W>(threadIdx.x);
            sc.fr[0][threadIdx.x] = v;
            sc.dl[0][threadIdx.x] = single<W>(threadIdx.x);
            sc.touched[threadIdx.x] = v;
        }
        __syncthreads();

        // All sources grow their balls in lock step.  When ball i (radius L) first meets ball j at a node, the
        // pair's distance is 2L - 1 if j was there since the level before, 2L if both arrive now: every pair is
        // settled after ceil(d / 2) levels, long before a one-sided search from i would reach j.
        const int want = nt * (nt - 1) / 2;
        int cb = 0;
        for (int level = 1;; ++level) {
            const int nf = s_nf[cb];
            const Mask<W> active = s_active;
            // ---- expand: one warp per frontier node, lanes over its adjacency
            const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
            for (int f = warp; f < nf; f += NT / 32) {
                const int u = sc.fr[cb][f];
                const Mask<W> du = sc.dl[cb][f] & active;              // a source that has found every partner stops here
                if (!any(du)) continue;
                const long long e0 = indptr[u], e1 = indptr[u + 1];
                for (long long e = e0 + lane; e < e1; e += 32) {
                    const int v = indices[e];
                    const Mask<W> nb = and_not(du, sc.cur[v]);
                    if (any(nb)) {
                        bool first;
                        if constexpr (W == 1) {
                            first = atomicOr(&sc.acc[v].w[0], nb.w[0]) == 0ull;
                        } else {
                            // two separate word atomics cannot tell who was first: the level stamp decides
#pragma unroll
                            for (int w = 0; w < W; ++w)
                                if (nb.w[w]) atomicOr(&sc.acc[v].w[w], nb.w[w]);
                            first = atomicExch(&stamp[v], level) != level;
                        }
                        if (first) {
                            const int pos = atomicAdd(&s_nf[cb ^ 1], 1);
                            NABO_DEV_ASSERT(pos < m);
                            sc.fr[cb ^ 1][pos] = v;
                        }
                    }
                }
            }
            __syncthreads();
            // ---- commit pass A: new bits meet the bits that were already there (distance 2L - 1)
            const int nn = s_nf[cb ^ 1];
            for (int f = threadIdx.x; f < nn; f += NT) {
                const int v = sc.fr[cb ^ 1][f];
                const Mask<W> c = sc.cur[v];
                const Mask<W> d = and_not(sc.acc[v], c);
                sc.acc[v] = Mask<W>{};
                sc.cur[v] = c | d;
                sc.dl[cb ^ 1][f] = d;
                if (!any(c)) sc.touched[atomicAdd(&s_ntouched, 1)] = v;  // first visit of v
                if (any(c)) {
                    Mask<W> di = d;
                    while (any(di)) {
                        const int i = pop_lowest(di);
                        Mask<W> cj = c;
                        while (any(cj)) {
                            const int j = pop_lowest(cj);
                            record(i, j, 2 * level - 1);
                        }
                    }
                }
            }
            __syncthreads();
            // ---- commit pass B: bits that arrive together (distance 2L), after every 2L - 1 meeting is known
            if (s_pairs < want) {
                for (int f = threadIdx.x; f < nn; f += NT) {
                    Mask<W> di = sc.dl[cb ^ 1][f];
                    if (two_or_more(di)) {
                        while (any(di)) {
                            const int i = pop_lowest(di);
                            Mask<W> dj = di;
                            while (any(dj)) {
                                const int j = pop_lowest(dj);
                                record(i, j, 2 * level);
                            }
                        }
                    }
                }
            }
            __syncthreads();
            if (threadIdx.x < nt && s_nfound[threadIdx.x] >= nt - 1)
                atomicAnd(&s_active.w[W == 1 ? 0 : threadIdx.x >> 6], ~(1ull << (W == 1 ? threadIdx.x : threadIdx.x & 63)));
            if (threadIdx.x == 0) s_nf[cb] = 0;
            cb ^= 1;
            const bool done = s_pairs >= want || nn == 0;
            __syncthreads();
            if (done) break;
        }
        // ---- clean the scratch for the next target
        const int ntouched = s_ntouched;
        for (int f = threadIdx.x; f < ntouched; f += NT) {
            const int v = sc.touched[f];
            sc.cur[v] = Mask<W>{};
            sc.acc[v] = Mask<W>{};
            if constexpr (W > 1) stamp[v] = 0;        // every node that joined a frontier was committed, so touched
        }
        if (threadIdx.x == 0) {
            out_sum[t] = 2 * (long long)s_sum;          // ordered-pair convention of the interface
            out_pairs[t] = 2 * s_pairs;
            out_nmapped[t] = nt;
            s_nf[0] = 0;
            s_nf[1] = 0;
        }
        __syncthreads();
    }
}

}  // namespace spec

static int spec_blocks(int m, size_t workspace_bytes, int n_query, int W) {
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    long long b = (long long)(workspace_bytes / spec::scratch_bytes(m, W));
    if (b > 4LL * sms) b = 4LL * sms;
    if (b > n_query) b = n_query;
    return (int)b;
}

extern "C" size_t nabo_specificity_workspace_bytes_k(int n_ref, int n_query, int k) {
    if (k > spec::MAXK) return 0;
    const size_t per_block = spec::scratch_bytes(n_ref, spec::words_for(k));
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    long long b = 4LL * sms;
    if (b > n_query) b = n_query;
    if (b < 1) b = 1;
    // cap the request at 8 GB: fewer CTAs are used for very large graphs
    size_t need = (size_t)b * per_block;
    const size_t cap = (size_t)8 << 30;
    if (need > cap) {
        need = cap;
        if (need < per_block) need = per_block;
    }
    return need;
}

extern "C" size_t nabo_specificity_workspace_bytes(int n_ref, int n_query) {
    return nabo_specificity_workspace_bytes_k(n_ref, n_query, 64);
}

extern "C" int nabo_mapping_specificity(const long long* indptr, const int32_t* indices, int n_ref,
                                        const int32_t* tgt_knn, const uint8_t* counts, int n_query, int k,
                                        long long* out_sum, int32_t* out_pairs, int32_t* out_nmapped,
                                        void* workspace, size_t workspace_bytes, void* stream) {
    NABO_ARG(n_ref > 0 && n_query >= 0 && k > 0, "mapping_specificity: bad sizes");
    NABO_ARG(k <= spec::MAXK, "mapping_specificity: at most %d mapped cells per target", spec::MAXK);
    NABO_ARG(indptr && indices && tgt_knn && counts && out_sum && out_pairs && out_nmapped, "mapping_specificity: null pointer");
    if (n_query == 0) return 0;
    const int W = spec::words_for(k);
    const size_t per_block = spec::scratch_bytes(n_ref, W);
    const int blocks = spec_blocks(n_ref, workspace_bytes, n_query, W);
    if (workspace == nullptr || blocks < 1)
        return nabo_set_error(NABO_EWORKSPACE, "mapping_specificity: workspace too small (need %zu bytes per CTA)",
                              per_block);
    cudaStream_t st = (cudaStream_t)stream;
    NABO_CUDA(cudaMemsetAsync(workspace, 0, (size_t)blocks * per_block, st));
    if (W == 1)
        spec::specificity_kernel<1><<<blocks, spec::NT, 0, st>>>(indptr, indices, n_ref, tgt_knn, counts, n_query, k,
                                                                 out_sum, out_pairs, out_nmapped,
                                                                 (unsigned char*)workspace, per_block);
    else
        spec::specificity_kernel<2><<<blocks, spec::NT, 0, st>>>(indptr, indices, n_ref, tgt_knn, counts, n_query, k,
                                                                 out_sum, out_pairs, out_nmapped,
                                                                 (unsigned char*)workspace, per_block);
    NABO_LAUNCH_CHECK("specificity_kernel");
    return 0;
}
