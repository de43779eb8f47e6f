// Exact FP64 kernels in the reference's arithmetic order.
//   * full distance tiles  (replace _euclidean_dist / _mod_canberra_dist, nabo/_mapping.py:16-45)
//   * brute-force distance + fused per-query top-k  (replace _calc_dist, :48-148)
//   * exact re-rank of nominated candidates
// All accumulate over dimensions k = 0..g-1 sequentially with separate multiply and
// add (__dmul_rn/__dadd_rn forbid FMA contraction), so results are bit-identical to the
// numba loops.  The brute-force kernel never writes the N x M matrix: each 64x64 tile
// is filtered against the running k-th best of its query and only survivors reach a
// per-query shared-memory buffer that a warp compacts with a bitonic sort.
#include <stdarg.h>
#include <stdio.h>

#include "common.cuh"
#include "knn_internal.cuh"
#include "select.cuh"

// ------------------------------------------------------------------ error channel
static thread_local char g_err[512] = "";
int nabo_set_error(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}
extern "C" const char* nabo_last_error(void) { return g_err; }
extern "C" int nabo_abi_version(void) { return NABO_ABI_VERSION; }
extern "C" int nabo_device_check(int* sm_count) {
    int dev = 0;
    NABO_CUDA(cudaGetDevice(&dev));
    cudaDeviceProp p;
    NABO_CUDA(cudaGetDeviceProperties(&p, dev));
    if (sm_count) *sm_count = p.multiProcessorCount;
    if (p.major != 10)
        return nabo_set_error(NABO_EUNSUPPORTED, "device %s is sm_%d%d; this library is built for sm_100a only",
                              p.name, p.major, p.minor);
    return 0;
}

// ------------------------------------------------------------------ per-pair arithmetic
template <int METRIC>
struct Pair {
    // one dimension
    static __device__ __forceinline__ double step(double acc, double x, double y, double f) {
        if (METRIC == NABO_EUCLIDEAN) {
            double t = __dsub_rn(x, y);
            return __dadd_rn(acc, __dmul_rn(t, t));
        } else if (METRIC == NABO_MOD_CANBERRA) {
            double absx = fabs(x);
            double num = fabs(__dsub_rn(x, y));
            if (num < __dmul_rn(f, absx)) {
                double den = __dadd_rn(__dadd_rn(absx, fabs(y)), 0.01);
                return __dadd_rn(acc, __ddiv_rn(num, den));
            }
            return __dadd_rn(acc, 1.0);
        } else {
            return __dadd_rn(acc, __dmul_rn(x, y));
        }
    }
    // nq, nr: squared norms (cosine only)
    static __device__ __forceinline__ double finish(double acc, double nq, double nr) {
        if (METRIC == NABO_EUCLIDEAN) return __dsqrt_rn(acc);
        if (METRIC == NABO_MOD_CANBERRA) return acc;
        return __dsub_rn(1.0, __ddiv_rn(acc, __dmul_rn(__dsqrt_rn(nq), __dsqrt_rn(nr))));
    }
};

__device__ __forceinline__ double seq_sqnorm(const double* v, int g) {
    double s = 0.0;
    for (int k = 0; k < g; ++k) s = __dadd_rn(s, __dmul_rn(v[k], v[k]));
    return s;
}

// ------------------------------------------------------------------ tile geometry
constexpr int TQ = 64;          // queries per block
constexpr int TR = 64;          // references per step
constexpr int NT = 256;         // threads: 16 x 16, each owns a 4 x 4 micro tile
constexpr int LDS_T = TQ + 2;   // padded row stride of the k-major tiles (keeps 16 B alignment)

__device__ __forceinline__ void load_tile_kmajor(double* s, const double* __restrict__ src, int ld,
                                                 int row0, int nrows, int g, const int* row_ids, int k0 = 0) {
    // s[k * LDS_T + r] = src[row(row0 + r)][k0 + k], k < g; rows past nrows are zero-filled
    for (int e = threadIdx.x; e < TQ * g; e += NT) {
        int r = e / g, k = e - r * g;
        int row = row0 + r;
        double v = 0.0;
        if (row < nrows) {
            long long rr = row_ids ? row_ids[row] : row;
            v = src[rr * (long long)ld + k0 + k];
        }
        s[k * LDS_T + r] = v;
    }
}

// ------------------------------------------------------------------ (1) distance tiles
template <int METRIC>
__global__ void __launch_bounds__(NT) dist_tile_kernel(const double* __restrict__ x, int ldx,
                                                       const double* __restrict__ y, int ldy,
                                                       double* __restrict__ d, int ldd, int m, int n,
                                                       int g, double f) {
    extern __shared__ double smem[];
    double* xs = smem;
    double* ys = smem + (size_t)g * LDS_T;
    __shared__ double nqs[TQ], nrs[TR];
    const int q0 = blockIdx.y * TQ, r0 = blockIdx.x * TR;
    load_tile_kmajor(xs, x, ldx, q0, m, g, nullptr);
    load_tile_kmajor(ys, y, ldy, r0, n, g, nullptr);
    __syncthreads();
    // correlation = cosine of the centred rows: one thread per tile row (padding rows included) centres it in place
    constexpr bool COS_LIKE = METRIC == NABO_COSINE || METRIC == NABO_CORRELATION;
    if (METRIC == NABO_CORRELATION && threadIdx.x < TQ + TR) {
        double* col = threadIdx.x < TQ ? xs + threadIdx.x : ys + (threadIdx.x - TQ);
        double s = 0.0;
        for (int k = 0; k < g; ++k) s = __dadd_rn(s, col[k * LDS_T]);
        const double mu = __ddiv_rn(s, (double)g);
        for (int k = 0; k < g; ++k) col[k * LDS_T] = __dsub_rn(col[k * LDS_T], mu);
    }
    if (METRIC == NABO_CORRELATION) __syncthreads();
    if (COS_LIKE) {
        if (threadIdx.x < TQ) {
            double s = 0.0;
            for (int k = 0; k < g; ++k) { double v = xs[k * LDS_T + threadIdx.x]; s = __dadd_rn(s, __dmul_rn(v, v)); }
            nqs[threadIdx.x] = s;
        } else if (threadIdx.x < TQ + TR) {
            int t = threadIdx.x - TQ;
            double s = 0.0;
            for (int k = 0; k < g; ++k) { double v = ys[k * LDS_T + t]; s = __dadd_rn(s, __dmul_rn(v, v)); }
            nrs[t] = s;
        }
        __syncthreads();
    }
    const int tr = threadIdx.x & 15, tq = threadIdx.x >> 4;
    double acc[4][4];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) acc[a][b] = 0.0;
    for (int k = 0; k < g; ++k) {
        double xv[4], yv[4];
#pragma unroll
        for (int a = 0; a < 4; ++a) xv[a] = xs[k * LDS_T + tq * 4 + a];
#pragma unroll
        for (int b = 0; b < 4; ++b) yv[b] = ys[k * LDS_T + tr * 4 + b];
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
            for (int b = 0; b < 4; ++b) acc[a][b] = Pair<METRIC>::step(acc[a][b], xv[a], yv[b], f);
    }
#pragma unroll
    for (int a = 0; a < 4; ++a) {
        int qi = q0 + tq * 4 + a;
        if (qi >= m) continue;
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            int rj = r0 + tr * 4 + b;
            if (rj < n) {
                double nq = COS_LIKE ? nqs[tq * 4 + a] : 0.0;
                double nr = COS_LIKE ? nrs[tr * 4 + b] : 0.0;
                d[(long long)qi * ldd + rj] = Pair<METRIC>::finish(acc[a][b], nq, nr);
            }
        }
    }
}

template <int METRIC>
static int launch_dist_tiles(const double* x, int ldx, const double* y, int ldy, double* d, int ldd,
                             int m, int n, int g, double f, cudaStream_t s) {
    NABO_ARG(m >= 0 && n >= 0 && g >= 1, "dist: bad shape m=%d n=%d g=%d", m, n, g);
    NABO_ARG(ldx >= g && ldy >= g && ldd >= n, "dist: leading dimension smaller than row length");
    if (m == 0 || n == 0) return 0;
    NABO_ARG(x && y && d, "dist: null pointer");
    size_t smem = 2 * (size_t)g * LDS_T * sizeof(double);
    NABO_ARG(smem <= 200 * 1024, "dist: g=%d exceeds the shared-memory tile (max %d dims)", g,
             (int)(200 * 1024 / (2 * LDS_T * sizeof(double))));
    NABO_CUDA(cudaFuncSetAttribute(dist_tile_kernel<METRIC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dim3 grid((n + TR - 1) / TR, (m + TQ - 1) / TQ);
    dist_tile_kernel<METRIC><<<grid, NT, smem, s>>>(x, ldx, y, ldy, d, ldd, m, n, g, f);
    NABO_LAUNCH_CHECK("dist_tile_kernel");
    return 0;
}

extern "C" int nabo_euclidean_dist(const double* x, int ldx, const double* y, int ldy, double* d, int ldd,
                                   int m, int n, int g, void* stream) {
    return launch_dist_tiles<NABO_EUCLIDEAN>(x, ldx, y, ldy, d, ldd, m, n, g, 0.0, (cudaStream_t)stream);
}
extern "C" int nabo_mod_canberra_dist(const double* x, int ldx, const double* y, int ldy, double* d, int ldd,
                                      int m, int n, int g, double f, void* stream) {
    return launch_dist_tiles<NABO_MOD_CANBERRA>(x, ldx, y, ldy, d, ldd, m, n, g, f, (cudaStream_t)stream);
}
extern "C" int nabo_cosine_dist(const double* x, int ldx, const double* y, int ldy, double* d, int ldd,
                                int m, int n, int g, void* stream) {
    return launch_dist_tiles<NABO_COSINE>(x, ldx, y, ldy, d, ldd, m, n, g, 0.0, (cudaStream_t)stream);
}
extern "C" int nabo_correlation_dist(const double* x, int ldx, const double* y, int ldy, double* d, int ldd,
                                     int m, int n, int g, void* stream) {
    return launch_dist_tiles<NABO_CORRELATION>(x, ldx, y, ldy, d, ldd, m, n, g, 0.0, (cudaStream_t)stream);
}

// ------------------------------------------------------------------ (2) brute force + fused top-k
// Per-query candidate buffer of CAP (d, i) pairs in shared memory.  A tile appends at
// most TR entries per query, so compacting whenever count > CAP - TR keeps it in bounds.
struct ExactSmem {
    double* xs;     // [g][LDS_T]
    double* ys;     // [g][LDS_T]
    double* bd;     // [TQ][CAP]
    int* bi;        // [TQ][CAP]
    double* tau_d;  // [TQ]
    double* nq;     // [TQ]
    double* nr;     // [TR]
    int* tau_i;     // [TQ]
    int* cnt;       // [TQ]
};

__device__ __forceinline__ ExactSmem carve_exact(double* base, int g, int cap) {
    ExactSmem s;
    s.xs = base;
    s.ys = s.xs + (size_t)g * LDS_T;
    s.bd = s.ys + (size_t)g * LDS_T;
    s.tau_d = s.bd + (size_t)TQ * cap;
    s.nq = s.tau_d + TQ;
    s.nr = s.nq + TQ;
    s.bi = (int*)(s.nr + TR);
    s.tau_i = s.bi + (size_t)TQ * cap;
    s.cnt = s.tau_i + TQ;
    return s;
}
static size_t exact_smem_bytes(int g, int cap) {
    return (2 * (size_t)g * LDS_T + (size_t)TQ * cap + 3 * TQ) * sizeof(double) +
           ((size_t)TQ * cap + 2 * TQ) * sizeof(int);
}

// one warp: sort the buffer of query q, keep the best ksel, refresh tau
__device__ __forceinline__ void compact_query(const ExactSmem& s, int q, int cap, int ksel, int lane) {
    double* d = s.bd + (size_t)q * cap;
    int* ix = s.bi + (size_t)q * cap;
    int n = s.cnt[q];
    for (int t = n + lane; t < cap; t += 32) { d[t] = CUDART_INF; ix[t] = 0x7fffffff; }
    __syncwarp();
    warp_bitonic_sort(d, ix, cap, lane);
    if (lane == 0) {
        if (n >= ksel) {
            s.cnt[q] = ksel;
            s.tau_d[q] = d[ksel - 1];
            s.tau_i[q] = ix[ksel - 1];
        }
    }
    __syncwarp();
}

template <int METRIC>
__global__ void __launch_bounds__(NT, 1)
knn_exact_kernel(const double* __restrict__ q, int ldq, const double* __restrict__ r, int ldr, int n_query,
                 int n_ref, int g, int k, double f, const uint8_t* __restrict__ mask, int drop_first,
                 int idx_offset, const int* __restrict__ row_ids, const int* __restrict__ n_rows_dev,
                 int cap, int gc, const NaboExactSplit sp, int32_t* __restrict__ out_idx, double* __restrict__ out_dist,
                 const NaboRoute route) {
    // gc = dimensions per shared-memory tile chunk (gc == g: the whole vectors, query tile loaded once; gc < g:
    // both tiles are streamed in chunks, the accumulators carry over - same sequential order of additions)
    extern __shared__ double smem[];
    const ExactSmem s = carve_exact(smem, gc, cap);
    const bool chunked = gc < g;
    const int nq_total = n_rows_dev ? *n_rows_dev : n_query;   // fallback mode: row list on device
    // fallback for FEW rows: the reference range is split over blockIdx.y and the partial lists are
    // merged afterwards (mode 1); with many rows the plain row-parallel kernel is used (mode 2)
    if (sp.mode == 1 && (nq_total > sp.f_max || nq_total <= sp.f_min)) return;
    if (sp.mode == 2 && nq_total <= sp.f_max) return;
    const int r_lo = sp.mode == 1 ? (int)((long long)n_ref * blockIdx.y / sp.nsplit) / TR * TR : 0;
    const int r_hi = sp.mode == 1 ? (blockIdx.y + 1 == (unsigned)sp.nsplit
                                         ? n_ref
                                         : (int)((long long)n_ref * (blockIdx.y + 1) / sp.nsplit) / TR * TR)
                                  : n_ref;
    const int q0 = blockIdx.x * TQ;
    if (q0 >= nq_total) return;
    const int ksel = k + (drop_first ? 1 : 0);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int tr = threadIdx.x & 15, tq = threadIdx.x >> 4;

    if (threadIdx.x < TQ) {
        s.cnt[threadIdx.x] = 0;
        s.tau_d[threadIdx.x] = CUDART_INF;
        s.tau_i[threadIdx.x] = 0x7fffffff;
    }
    if (!chunked) {
        load_tile_kmajor(s.xs, q, ldq, q0, nq_total, g, row_ids);
        __syncthreads();
        if (METRIC == NABO_COSINE && threadIdx.x < TQ) {
            double acc = 0.0;
            for (int kk = 0; kk < g; ++kk) { double v = s.xs[kk * LDS_T + threadIdx.x]; acc = __dadd_rn(acc, __dmul_rn(v, v)); }
            s.nq[threadIdx.x] = acc;
        }
    } else if (METRIC == NABO_COSINE) {
        double acc = 0.0;                                   // squared norm of the queries, chunk by chunk, same order
        for (int kc = 0; kc < g; kc += gc) {
            const int gn = min(gc, g - kc);
            __syncthreads();
            load_tile_kmajor(s.xs, q, ldq, q0, nq_total, gn, row_ids, kc);
            __syncthreads();
            if (threadIdx.x < TQ)
                for (int kk = 0; kk < gn; ++kk) { double v = s.xs[kk * LDS_T + threadIdx.x]; acc = __dadd_rn(acc, __dmul_rn(v, v)); }
        }
        if (threadIdx.x < TQ) s.nq[threadIdx.x] = acc;
    }

    for (int r0 = r_lo; r0 < r_hi; r0 += TR) {
        double acc[4][4];
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
            for (int b = 0; b < 4; ++b) acc[a][b] = 0.0;
        for (int kc = 0; kc < g; kc += gc) {
            const int gn = min(gc, g - kc);
            __syncthreads();   // previous tile / chunk fully consumed (and compaction finished)
            if (chunked) load_tile_kmajor(s.xs, q, ldq, q0, nq_total, gn, row_ids, kc);
            load_tile_kmajor(s.ys, r, ldr, r0, r_hi, gn, nullptr, kc);
            __syncthreads();
            if (METRIC == NABO_COSINE && threadIdx.x < TR) {
                double nacc = kc == 0 ? 0.0 : s.nr[threadIdx.x];
                for (int kk = 0; kk < gn; ++kk) { double v = s.ys[kk * LDS_T + threadIdx.x]; nacc = __dadd_rn(nacc, __dmul_rn(v, v)); }
                s.nr[threadIdx.x] = nacc;
            }
            // a thread whose four query rows all lie beyond the row count has nothing to accumulate (the fallback for a
            // few rows runs 64-row tiles with one or two live rows: 15 of 16 threads skip the FP64 work)
            if (q0 + tq * 4 < nq_total)
            for (int kk = 0; kk < gn; ++kk) {
                double xv[4], yv[4];
#pragma unroll
                for (int a = 0; a < 4; ++a) xv[a] = s.xs[kk * LDS_T + tq * 4 + a];
#pragma unroll
                for (int b = 0; b < 4; ++b) yv[b] = s.ys[kk * LDS_T + tr * 4 + b];
#pragma unroll
                for (int a = 0; a < 4; ++a)
#pragma unroll
                    for (int b = 0; b < 4; ++b) acc[a][b] = Pair<METRIC>::step(acc[a][b], xv[a], yv[b], f);
            }
        }
        if (METRIC == NABO_COSINE) __syncthreads();        // reference norms complete
        // filter against the running k-th best and append survivors
#pragma unroll
        for (int a = 0; a < 4; ++a) {
            const int ql = tq * 4 + a;
            if (q0 + ql >= nq_total) continue;
            const double td = s.tau_d[ql];
            const int ti = s.tau_i[ql];
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                const int j = r0 + tr * 4 + b;
                if (j >= r_hi) continue;
                double d = Pair<METRIC>::finish(acc[a][b], METRIC == NABO_COSINE ? s.nq[ql] : 0.0,
                                                METRIC == NABO_COSINE ? s.nr[tr * 4 + b] : 0.0);
                if (d != d || (mask && mask[j])) d = CUDART_INF;   // NaN / ignored -> last
                if (nabo_less(d, j, td, ti)) {
                    int pos = atomicAdd(&s.cnt[ql], 1);
                    s.bd[(size_t)ql * cap + pos] = d;
                    s.bi[(size_t)ql * cap + pos] = j;
                }
            }
        }
        __syncthreads();
        for (int ql = warp; ql < TQ; ql += NT / 32)
            if (s.cnt[ql] > cap - TR) compact_query(s, ql, cap, ksel, lane);
    }
    __syncthreads();
    // final sort + write-out
    for (int ql = warp; ql < TQ; ql += NT / 32) {
        const int qi = q0 + ql;
        if (qi >= nq_total) continue;
        const int n_have = s.cnt[ql];
        {
            double* d = s.bd + (size_t)ql * cap;
            int* ix = s.bi + (size_t)ql * cap;
            for (int t = n_have + lane; t < cap; t += 32) { d[t] = CUDART_INF; ix[t] = 0x7fffffff; }
            __syncwarp();
            warp_bitonic_sort(d, ix, cap, lane);
        }
        if (sp.mode == 1) {
            // partial list of this reference range: raw keys (NaN / masked = +inf), local indices
            for (int t = lane; t < ksel; t += 32) {
                const bool have = t < n_have && t < cap;
                const size_t o = ((size_t)blockIdx.y * sp.f_max + qi) * ksel + t;
                sp.part_idx[o] = have ? s.bi[(size_t)ql * cap + t] : -1;
                sp.part_dist[o] = have ? s.bd[(size_t)ql * cap + t] : CUDART_INF;
            }
            continue;
        }
        const long long orow = row_ids ? row_ids[qi] : qi;
        int32_t* oi;
        double* od;
        nabo_route_row(route, orow, k, out_idx, out_dist, oi, od);
        const int skip = drop_first ? 1 : 0;
        for (int t = lane; t < k; t += 32) {
            int src = t + skip;
            int id = -1;
            double dv = CUDART_NAN;
            if (src < n_have && src < cap) {
                id = s.bi[(size_t)ql * cap + src];
                dv = s.bd[(size_t)ql * cap + src];
                if (mask && mask[id]) dv = CUDART_NAN;
                else if (dv == CUDART_INF) {
                    // NaN distances were keyed as +inf: recompute to tell them from a true inf
                    dv = CUDART_NAN;
                }
                id += idx_offset;
            }
            oi[t] = id;
            od[t] = dv;
        }
    }
}

static int exact_cap_for(int ksel) {
    int kp = nabo_next_pow2(ksel);
    int cap = 2 * kp;
    if (cap < 128) cap = 128;
    return cap;
}

// merge the per-range partial lists of the split fallback: one warp per failing row
__global__ void __launch_bounds__(128)
fallback_merge_kernel(const NaboExactSplit sp, const int* __restrict__ row_ids, const int* __restrict__ n_rows_dev,
                      int k, int drop_first, int idx_offset, const uint8_t* __restrict__ mask, int capp,
                      int32_t* __restrict__ out_idx, double* __restrict__ out_dist, const NaboRoute route) {
    extern __shared__ double smem[];
    const int n_rows = *n_rows_dev;
    if (n_rows > sp.f_max || n_rows <= sp.f_min) return;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int qi = blockIdx.x * 4 + warp;
    if (qi >= n_rows) return;
    const int ksel = k + (drop_first ? 1 : 0);
    double* d = smem + (size_t)warp * capp;
    int* ix = (int*)(smem + (size_t)4 * capp) + (size_t)warp * capp;
    const int tot = sp.nsplit * ksel;
    int n_valid = 0;
    for (int c = lane; c < capp; c += 32) {
        double dv = CUDART_INF;
        int id = 0x7fffffff;
        if (c < tot) {
            const int sidx = c / ksel, j = c - sidx * ksel;
            const size_t o = ((size_t)sidx * sp.f_max + qi) * ksel + j;
            const int i0 = sp.part_idx[o];
            if (i0 >= 0) { id = i0; dv = sp.part_dist[o]; ++n_valid; }
        }
        d[c] = dv; ix[c] = id;
    }
    for (int o = 16; o > 0; o >>= 1) n_valid += __shfl_xor_sync(0xffffffffu, n_valid, o);
    __syncwarp();
    warp_bitonic_sort(d, ix, capp, lane);
    const long long orow = row_ids[qi];
    int32_t* oi;
    double* od;
    nabo_route_row(route, orow, k, out_idx, out_dist, oi, od);
    const int skip = drop_first ? 1 : 0;
    for (int t = lane; t < k; t += 32) {
        const int src = t + skip;
        int id = -1;
        double dv = CUDART_NAN;
        if (src < n_valid) {
            id = ix[src];
            dv = d[src];
            if (dv == CUDART_INF || (mask && mask[id])) dv = CUDART_NAN;
            id += idx_offset;
        }
        oi[t] = id;
        od[t] = dv;
    }
}

// the same merge for the few-rows split (up to NABO_FALLBACK_FEW_ENTRIES partial entries per row): one block per row,
// block-wide bitonic sort in shared memory
__global__ void __launch_bounds__(256)
fallback_merge_few_kernel(const NaboExactSplit sp, const int* __restrict__ row_ids, const int* __restrict__ n_rows_dev,
                          int k, int drop_first, int idx_offset, const uint8_t* __restrict__ mask, int capp,
                          int32_t* __restrict__ out_idx, double* __restrict__ out_dist, const NaboRoute route) {
    extern __shared__ double smem[];
    const int n_rows = *n_rows_dev;
    if (n_rows > sp.f_max || n_rows <= sp.f_min) return;
    const int qi = blockIdx.x;
    if (qi >= n_rows) return;
    const int ksel = k + (drop_first ? 1 : 0);
    double* d = smem;
    int* ix = (int*)(smem + capp);
    __shared__ int s_valid;
    if (threadIdx.x == 0) s_valid = 0;
    __syncthreads();
    const int tot = sp.nsplit * ksel;
    int n_valid = 0;
    for (int c = threadIdx.x; c < capp; c += blockDim.x) {
        double dv = CUDART_INF;
        int id = 0x7fffffff;
        if (c < tot) {
            const int sidx = c / ksel, j = c - sidx * ksel;
            const size_t o = ((size_t)sidx * sp.f_max + qi) * ksel + j;
            const int i0 = sp.part_idx[o];
            if (i0 >= 0) { id = i0; dv = sp.part_dist[o]; ++n_valid; }
        }
        d[c] = dv; ix[c] = id;
    }
    atomicAdd(&s_valid, n_valid);
    __syncthreads();
    for (int size = 2; size <= capp; size <<= 1)
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int t = threadIdx.x; t < (capp >> 1); t += blockDim.x) {
                const int lo = 2 * t - (t & (stride - 1)), hi = lo + stride;
                const bool up = (lo & size) == 0;
                const double dl = d[lo], dh = d[hi];
                const int il = ix[lo], ih = ix[hi];
                if (up ? nabo_less(dh, ih, dl, il) : nabo_less(dl, il, dh, ih)) { d[lo] = dh; d[hi] = dl; ix[lo] = ih; ix[hi] = il; }
            }
            __syncthreads();
        }
    const long long orow = row_ids[qi];
    int32_t* oi;
    double* od;
    nabo_route_row(route, orow, k, out_idx, out_dist, oi, od);
    const int skip = drop_first ? 1 : 0;
    for (int t = threadIdx.x; t < k; t += blockDim.x) {
        const int src = t + skip;
        int id = -1;
        double dv = CUDART_NAN;
        if (src < s_valid) {
            id = ix[src];
            dv = d[src];
            if (dv == CUDART_INF || (mask && mask[id])) dv = CUDART_NAN;
            id += idx_offset;
        }
        oi[t] = id;
        od[t] = dv;
    }
}

static void split_carve(NaboArena& ar, int nsplit, int f_max, int ksel, NaboExactSplit* sp) {
    sp->mode = 1;
    sp->nsplit = nsplit;
    sp->f_max = f_max;
    sp->f_min = 0;
    sp->part_dist = ar.take<double>((size_t)nsplit * f_max * ksel);
    sp->part_idx = ar.take<int32_t>((size_t)nsplit * f_max * ksel);
}

void nabo_exact_split_carve(NaboArena& ar, int n_ref, int ksel, NaboExactSplit* split, NaboExactSplit* few) {
    // (b) up to NABO_FALLBACK_SPLIT_ROWS rows: up to 48 pieces, one warp merges a row
    const int s = 2048 / ksel;
    split_carve(ar, s > 48 ? 48 : (s < 1 ? 1 : s), NABO_FALLBACK_SPLIT_ROWS, ksel, split);
    few->nsplit = 0;
    if (n_ref < NABO_FALLBACK_FEW_MIN_REF) return;
    // (a) a handful of rows against a large reference: two pieces per SM, block-wide merge
    const int sms2 = 2 * nabo_sm_count();
    split_carve(ar, NABO_FALLBACK_FEW_ENTRIES / ksel < sms2 ? NABO_FALLBACK_FEW_ENTRIES / ksel : sms2,
                NABO_FALLBACK_FEW_ROWS, ksel, few);
    split->f_min = NABO_FALLBACK_FEW_ROWS;
}

// Exact engine on the rows listed in row_ids[0 .. *n_rows_dev): split over the reference when the rows
// are few (one block would otherwise scan the whole reference alone), row-parallel otherwise.  All
// variants are launched; each checks the device-side row count and exits at once if it is not its turn,
// so no host synchronisation is needed.
int nabo_knn_exact_fallback(const double* q, int ldq, const double* r, int ldr, int n_query, int n_ref, int g, int k,
                            int metric, double f, const uint8_t* mask, int drop_first, int idx_offset,
                            const int* row_ids, const int* n_rows_dev, const NaboExactSplit& split,
                            const NaboExactSplit& few, int32_t* out_idx, double* out_dist, const NaboRoute& route,
                            cudaStream_t st) {
    const int ksel = k + (drop_first ? 1 : 0);
    if (few.nsplit > 0) {
        int rc0 = nabo_knn_exact_launch_ex(q, ldq, r, ldr, NABO_FALLBACK_FEW_ROWS, n_ref, g, ksel, metric, f, mask, 0, 0,
                                           row_ids, n_rows_dev, few, out_idx, out_dist, route, st);
        if (rc0) return rc0;
        const int cappf = nabo_next_pow2(few.nsplit * ksel);
        const size_t smf = (size_t)cappf * (sizeof(double) + sizeof(int));
        NABO_CUDA(cudaFuncSetAttribute(fallback_merge_few_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smf));
        fallback_merge_few_kernel<<<NABO_FALLBACK_FEW_ROWS, 256, smf, st>>>(few, row_ids, n_rows_dev, k, drop_first,
                                                                         idx_offset, mask, cappf, out_idx, out_dist,
                                                                         route);
        NABO_LAUNCH_CHECK("fallback_merge_few_kernel");
    }
    int rc = nabo_knn_exact_launch_ex(q, ldq, r, ldr, NABO_FALLBACK_SPLIT_ROWS, n_ref, g, ksel, metric, f, mask, 0, 0,
                                      row_ids, n_rows_dev, split, out_idx, out_dist, route, st);
    if (rc) return rc;
    int capp = nabo_next_pow2(split.nsplit * ksel);
    if (capp < 32) capp = 32;
    const size_t smem = (size_t)4 * capp * (sizeof(double) + sizeof(int));
    NABO_CUDA(cudaFuncSetAttribute(fallback_merge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    fallback_merge_kernel<<<(NABO_FALLBACK_SPLIT_ROWS + 3) / 4, 128, smem, st>>>(split, row_ids, n_rows_dev, k, drop_first,
                                                                               idx_offset, mask, capp, out_idx, out_dist,
                                                                               route);
    NABO_LAUNCH_CHECK("fallback_merge_kernel");
    NaboExactSplit rest = split;
    rest.mode = 2;
    return nabo_knn_exact_launch_ex(q, ldq, r, ldr, n_query, n_ref, g, k, metric, f, mask, drop_first, idx_offset,
                                    row_ids, n_rows_dev, rest, out_idx, out_dist, route, st);
}

int nabo_knn_exact_launch(const double* q, int ldq, const double* r, int ldr, int n_query, int n_ref, int g,
                          int k, int metric, double f, const uint8_t* mask, int drop_first, int idx_offset,
                          const int* row_ids, const int* n_rows_dev, int32_t* out_idx, double* out_dist,
                          const NaboRoute& route, cudaStream_t st) {
    NaboExactSplit sp;
    sp.mode = 0; sp.nsplit = 1; sp.f_max = 0; sp.f_min = 0; sp.part_idx = nullptr; sp.part_dist = nullptr;
    return nabo_knn_exact_launch_ex(q, ldq, r, ldr, n_query, n_ref, g, k, metric, f, mask, drop_first, idx_offset,
                                    row_ids, n_rows_dev, sp, out_idx, out_dist, route, st);
}

int nabo_knn_exact_call(const double* q, int ldq, const double* r, int ldr, int n_query, int n_ref, int g, int k,
                        int metric, double f, const uint8_t* mask, int drop_first, int idx_offset, int32_t* out_idx,
                        double* out_dist, const NaboRoute& route, int64_t* stats_host, cudaStream_t st) {
    NaboStageTimer tm(stats_host != nullptr, st);
    tm.begin();
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

int nabo_knn_exact_launch_ex(const double* q, int ldq, const double* r, int ldr, int n_query, int n_ref, int g,
                             int k, int metric, double f, const uint8_t* mask, int drop_first, int idx_offset,
                             const int* row_ids, const int* n_rows_dev, const NaboExactSplit& sp, int32_t* out_idx,
                             double* out_dist, const NaboRoute& route, cudaStream_t st) {
    const int ksel = k + (drop_first ? 1 : 0);
    NABO_ARG(k >= 1 && ksel <= 128, "knn: k=%d unsupported (1 <= k, k + drop_first <= 128)", k);
    NABO_ARG(g >= 1, "knn: g=%d", g);
    if (n_query == 0) return 0;
    const int cap = exact_cap_for(ksel);
    // whole vectors in shared memory when they fit next to the candidate buffers, else chunks of gc dimensions
    int gc = g;
    while (gc > 8 && exact_smem_bytes(gc, cap) > (size_t)227 * 1024) gc = (gc + 1) / 2;
    size_t smem = exact_smem_bytes(gc, cap);
    NABO_ARG(smem <= 227 * 1024, "knn: g=%d with k=%d needs %zu B of shared memory (max 232448)", g, k, smem);
    dim3 grid((n_query + TQ - 1) / TQ, sp.mode == 1 ? sp.nsplit : 1);
#define LAUNCH(M)                                                                                         \
    NABO_CUDA(cudaFuncSetAttribute(knn_exact_kernel<M>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    knn_exact_kernel<M><<<grid, NT, smem, st>>>(q, ldq, r, ldr, n_query, n_ref, g, k, f, mask, drop_first, \
                                                idx_offset, row_ids, n_rows_dev, cap, gc, sp, out_idx, out_dist, route);
    if (metric == NABO_EUCLIDEAN) { LAUNCH(NABO_EUCLIDEAN) }
    else if (metric == NABO_MOD_CANBERRA) { LAUNCH(NABO_MOD_CANBERRA) }
    else if (metric == NABO_COSINE) { LAUNCH(NABO_COSINE) }
    else return nabo_set_error(NABO_EINVAL, "knn: unknown metric %d", metric);
#undef LAUNCH
    NABO_LAUNCH_CHECK("knn_exact_kernel");
    return 0;
}

// ------------------------------------------------------------------ exact re-rank of candidates
// One warp per query.  cand (n_query x n_cand) holds LOCAL reference indices, -1 = empty,
// all distinct.  With a certificate (NaboCert.kind != 0) the kernel also proves that no
// reference outside the candidate list can belong to the top ksel: every such reference
// had candidate-pass score >= tau[q], which bounds its exact distance from below by L(q);
// the row passes iff its ksel-th exact distance is strictly below L(q).  Rows that fail are
// appended to fail_rows for the exact brute-force engine.
__device__ __forceinline__ double cert_lower_bound(const NaboCert& c, int qi, float tau) {
    if (c.kind == NABO_CERT_LINEAR) return (double)tau - c.c_acc;     // score = lower bound of the distance
    const double sc_inv = c.scal[1], rmax = c.scal[2];
    const double qn2 = c.qn2[qi];
    const double qn = sqrt(qn2);
    const double eps = c.c_acc * (4.0 * qn * rmax + rmax * rmax + qn2);       // accumulation error (scaled^2)
    const double l2 = (double)tau + qn2 - eps;
    if (c.kind == NABO_CERT_EUCLID) {
        if (!(l2 > 0.0)) return 0.0;
        // |d~ - d| <= 2^-21 (|q| + |r|) from the two-term FP16 split of the inputs
        return sqrt(l2) * sc_inv * (1.0 - 1e-7) - (9.6e-7 * (qn + rmax) + c.abs_slack) * sc_inv;
    }
    // cosine: unit vectors, chord e -> distance e^2 / 2.  The FP64 distance 1 - dot / (|q| |r|) itself lies up to
    // (g + 5) 2^-53 below the true one (below zero for parallel vectors, e.g. every centred row at g = 2 under
    // correlation), so the bound keeps 1e-12 below it: a non-candidate at a rounded-down distance cannot pass.
    double e = l2 > 0.0 ? sqrt(l2) * sc_inv - 1.0e-6 : 0.0;
    if (!(e > 0.0)) e = 0.0;
    return 0.5 * e * e * (1.0 - 1e-9) - 1e-12;
}

// acc[u] = sum over the dimensions of the pair terms of (x, row jj[u] of r), u < NU, all slots in one sweep over the
// dimensions.  Slots without a candidate (jj < 0) read row 0 and are ignored by the caller.  vec2: r is 16-byte
// aligned with an even leading dimension, rows are read as double2.
template <int METRIC, int NU>
__device__ __forceinline__ void pair_rows(const double* __restrict__ x, const double* __restrict__ r, int ldr,
                                          const int* jj, int g, double f, bool vec2, double* acc) {
    const double* y[NU];
#pragma unroll
    for (int u = 0; u < NU; ++u) y[u] = r + (long long)(jj[u] >= 0 ? jj[u] : 0) * ldr;
    double a[NU];
#pragma unroll
    for (int u = 0; u < NU; ++u) a[u] = 0.0;
    int kk = 0;
    if (vec2) {
#pragma unroll 4
        for (; kk + 2 <= g; kk += 2) {
            const double x0 = x[kk], x1 = x[kk + 1];
#pragma unroll
            for (int u = 0; u < NU; ++u) {
                const double2 v = __ldg(reinterpret_cast<const double2*>(y[u] + kk));
                a[u] = Pair<METRIC>::step(a[u], x0, v.x, f);
                a[u] = Pair<METRIC>::step(a[u], x1, v.y, f);
            }
        }
    }
#pragma unroll 4
    for (; kk < g; ++kk) {
        const double xv = x[kk];
#pragma unroll
        for (int u = 0; u < NU; ++u) a[u] = Pair<METRIC>::step(a[u], xv, __ldg(y[u] + kk), f);
    }
#pragma unroll
    for (int u = 0; u < NU; ++u) acc[u] = a[u];
}

#ifdef NABO_RR_STATS      // development counters: [0] rows [1] rows on the sort path [2] sum of cut-bin sizes [3] sum of buffer
__device__ unsigned long long g_rr_stats[8];   // counts [4] sum of keys ranked away
extern "C" int nabo_dbg_rr_stats(unsigned long long* out_host, int reset) {
    cudaDeviceSynchronize();
    cudaMemcpyFromSymbol(out_host, g_rr_stats, sizeof(unsigned long long) * 8);
    if (reset) { unsigned long long z[8] = {0}; cudaMemcpyToSymbol(g_rr_stats, z, sizeof(z)); }
    return 0;
}
#endif
// NS: candidate slots per lane - 4 for capp <= 128; 8 for capp = 256 (Euclidean / cosine without FROM_BUF: the
// 256-key tensor-core plan, K' up to 160)
template <int METRIC, bool FROM_BUF, int NS = 4>
__global__ void __launch_bounds__(128)
rerank_kernel(const double* __restrict__ q, int ldq, const double* __restrict__ r, int ldr, int n_query,
              int n_ref, int g, int k, double f, const uint8_t* __restrict__ mask, int drop_first,
              int idx_offset, const int32_t* __restrict__ cand, int n_cand, int capp, const NaboCert cert,
              int* __restrict__ fail_rows, int* __restrict__ fail_count,
              int32_t* __restrict__ out_idx, double* __restrict__ out_dist, const NaboRoute route,
              const NaboCandBuf cb, int xs_dims, bool vec2, int row0) {
    static_assert(NS == 4 || (NS == 8 && !FROM_BUF), "8 slots per lane: candidate lists only (capp = 256)");
    extern __shared__ double smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int qi = row0 + blockIdx.x * 4 + warp;
    if (qi >= n_query) return;
    int32_t* oi;
    double* od;
    nabo_route_row(route, qi, k, out_idx, out_dist, oi, od);
    double* d = smem + (size_t)warp * capp;
    int* ix = (int*)(smem + (size_t)4 * capp) + (size_t)warp * capp;
    const size_t hist_off = (size_t)6 * capp + (size_t)4 * xs_dims;      // FROM_BUF only: 256 counters per warp
    const double* x = q + (long long)qi * ldq;
    double nq = 0.0;
    if (METRIC == NABO_COSINE) nq = seq_sqnorm(x, g);
    // FROM_BUF: final K' selection of the query's candidate buffer (what tc::emit_kernel does otherwise).  One
    // histogram pass over the scores finds the bin that holds the K'-th best key; the keys of lower bins and the best
    // of that bin (ranked by pairwise comparison) are the K' candidates, the threshold is the largest kept score.
    // If the cut bin holds more than 48 keys (a big tie class), the 128 keys are sorted by score in registers
    // instead.  Either way the list ends up in ix[0 .. nc), nc <= K' <= capp.
    int nc = 0;
    float tau_q = CUDART_INF_F;
    if (FROM_BUF) {
        const int n = __ldcg(cb.cnt + qi);            // through L2: the producer may still be running (dependent launch)
        const unsigned long long* gb = cb.buf + (size_t)qi * sel::CAP;
        float fv[4];
        uint32_t kpl[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int i = u * 32 + lane;
            const unsigned long long kv = i < n ? __ldcg(gb + i) : 0ull;
            fv[u] = __uint_as_float((uint32_t)(kv >> 32));
            kpl[u] = (uint32_t)kv;
        }
        uint32_t* hist = reinterpret_cast<uint32_t*>(smem + hist_off) + warp * 256;
        int bin[4], cut_bin, kept;
        bool reach;
        sel::histogram_cut(fv, n, lane, cb.kprime, hist, bin, cut_bin, kept, reach);
        // keys of the cut bin beyond the K' needed: ranked among themselves (score, then buffer position), so that
        // exactly K' stay - every extra candidate is a 400-byte row gather from HBM once the reference outgrows L2
        const int c_cut = reach ? (int)hist[cut_bin] : 0;
        const int need = cb.kprime - (kept - c_cut);             // keys still wanted from the cut bin: 1 .. c_cut
#ifdef NABO_RR_STATS
        if (lane == 0) {
            atomicAdd(&g_rr_stats[0], 1ull); atomicAdd(&g_rr_stats[1], (unsigned long long)(reach && c_cut > 48));
            atomicAdd(&g_rr_stats[2], (unsigned long long)c_cut); atomicAdd(&g_rr_stats[3], (unsigned long long)n);
            atomicAdd(&g_rr_stats[4], (unsigned long long)(reach ? c_cut - need : 0));
        }
#endif
        if (!reach || c_cut <= 48) {
            int rank[4] = {0, 0, 0, 0};
            if (reach && c_cut > need) {
#pragma unroll
                for (int us = 0; us < 4; ++us) {
                    unsigned mm = __ballot_sync(0xffffffffu, us * 32 + lane < n && bin[us] == cut_bin);
                    while (mm) {
                        const int src = __ffs(mm) - 1;
                        mm &= mm - 1;
                        const float sv = __shfl_sync(0xffffffffu, fv[us], src);
#pragma unroll
                        for (int u = 0; u < 4; ++u)
                            rank[u] += (sv < fv[u] || (sv == fv[u] && us * 32 + src < u * 32 + lane)) ? 1 : 0;
                    }
                }
                kept = cb.kprime;
            }
            int base = 0;
            float tmax = -CUDART_INF_F;
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const bool keep = u * 32 + lane < n && (bin[u] < cut_bin || (bin[u] == cut_bin && rank[u] < need));
                const unsigned m = __ballot_sync(0xffffffffu, keep);
                if (keep) {
                    ix[base + __popc(m & ((1u << lane) - 1u))] = (int)kpl[u];
                    tmax = fmaxf(tmax, fv[u]);
                }
                base += __popc(m);
            }
            tmax = sortable_to_float(__reduce_max_sync(0xffffffffu, float_to_sortable(tmax)));
            nc = kept;
            tau_q = reach ? tmax : __ldcg(cb.tau + qi);
        } else {
            uint32_t ks[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) ks[u] = u * 32 + lane < n ? float_to_sortable(fv[u]) : 0xffffffffu;
            sel::sortn(ks, kpl, lane);
            nc = n < cb.kprime ? n : cb.kprime;
            const int e = cb.kprime - 1;                      // kprime <= 64
            const uint32_t ts = __shfl_sync(0xffffffffu, (e >> 5) ? ks[1] : ks[0], e & 31);
            tau_q = n >= cb.kprime ? sortable_to_float(ts) : __ldcg(cb.tau + qi);
#pragma unroll
            for (int u = 0; u < 2; ++u)
                if (u * 32 + lane < nc) ix[u * 32 + lane] = (int)kpl[u];
        }
        __syncwarp();
    } else if (cert.kind != NABO_CERT_NONE) {
        tau_q = cert.tau[qi];
    }
    // The query in shared memory (broadcast reads), then every lane walks the rows of its candidates - slot u of a
    // lane is candidate u * 32 + lane - for all its slots in ONE loop over the dimensions: the loads of different
    // slots are independent, the additions of one slot stay in dimension order (bit-identical to the exact engine).
    double* xw = xs_dims ? smem + (size_t)4 * capp + (size_t)(4 * capp + 1) / 2 + (size_t)warp * xs_dims : nullptr;
    if (xw) {
        for (int kk = lane; kk < g; kk += 32) xw[kk] = x[kk];
        __syncwarp();
    }
    const double* xq = xw ? xw : x;
    int jj[NS];
    int n_slots = 0;
    const bool scramble = (long long)n_ref * ldr * 8 > (96ll << 20);
#pragma unroll
    for (int u = 0; u < NS; ++u) {
        const int c = u * 32 + lane;
        int j = -1;
        if (u * 32 < capp) {
            if (FROM_BUF) {
                // list positions are dealt to the lanes through a fixed bijection of [0, capp): in list order (the
                // order the sweep found them = ascending reference row) the row gathers of a warp run measurably
                // slower once the reference outgrows L2 (2.9 vs 2.3 ms at 227 k x 1.25 M); an L2-resident reference
                // prefers the list order (0.46 vs 0.49 ms at 100 k x 100 k)
                const int cpos = scramble ? ((c * 27 + 5) & (capp - 1)) : c;
                j = (u < 2 && cpos < nc) ? ix[cpos] : -1;
            }
            else j = c < n_cand ? cand[(long long)qi * n_cand + c] : -1;
        }
        if (!(j >= 0 && j < n_ref)) j = -1;
        jj[u] = j;
        if (__any_sync(0xffffffffu, j >= 0)) n_slots = u + 1;
    }
    double accs[NS];
#pragma unroll
    for (int u = 0; u < NS; ++u) accs[u] = 0.0;
    if (METRIC == NABO_MOD_CANBERRA) {
        // the FP64 division sits under a divergent branch: slot by slot, so that a slot with few lanes costs few divisions
#pragma unroll
        for (int u = 0; u < NS; ++u)
            if (u < n_slots) pair_rows<METRIC, 1>(xq, r, ldr, jj + u, g, f, vec2, accs + u);
    } else if (n_slots == 1) pair_rows<METRIC, 1>(xq, r, ldr, jj, g, f, vec2, accs);
    else if (n_slots == 2) pair_rows<METRIC, 2>(xq, r, ldr, jj, g, f, vec2, accs);
    else if (NS > 4 && n_slots > 4) pair_rows<METRIC, NS>(xq, r, ldr, jj, g, f, vec2, accs);
    else if (n_slots > 2) pair_rows<METRIC, 4>(xq, r, ldr, jj, g, f, vec2, accs);
    int n_valid = 0, n_finite = 0;
    int ids[NS];
#pragma unroll
    for (int u = 0; u < NS; ++u) {
        const int j = jj[u];
        double key = CUDART_INF;
        int id = 0x7fffffff;
        if (j >= 0) {
            double nr = 0.0;
            if (METRIC == NABO_COSINE) nr = seq_sqnorm(r + (long long)j * ldr, g);
            double dv = Pair<METRIC>::finish(accs[u], nq, nr);
            if (dv != dv || (mask && mask[j])) dv = CUDART_INF;
            key = dv;
            id = j;
            ++n_valid;
            n_finite += (dv < CUDART_INF);
        }
        accs[u] = key; ids[u] = id;
    }
    // ascending (distance, index) order in registers, then into the warp's shared-memory row for the indexed reads below
    if (capp <= 32) {
        double d1[1] = {accs[0]};
        int i1[1] = {ids[0]};
        warp_bitonic_sort_regs<1>(d1, i1, lane);
        d[lane] = d1[0]; ix[lane] = i1[0];
    } else if (capp <= 64) {
        double d2[2] = {accs[0], accs[1]};
        int i2[2] = {ids[0], ids[1]};
        warp_bitonic_sort_regs<2>(d2, i2, lane);
#pragma unroll
        for (int u = 0; u < 2; ++u) { d[u * 32 + lane] = d2[u]; ix[u * 32 + lane] = i2[u]; }
    } else {
        // every slot of every lane holds a candidate position: capp == 32 * NS (128 for NS = 4, 256 for NS = 8; the
        // launcher picks NS = 8 only for capp > 128)
        NABO_DEV_ASSERT(capp == 32 * NS);
        warp_bitonic_sort_regs<NS>(accs, ids, lane);
#pragma unroll
        for (int u = 0; u < NS; ++u) { d[u * 32 + lane] = accs[u]; ix[u * 32 + lane] = ids[u]; }
    }
    __syncwarp();
    for (int o = 16; o > 0; o >>= 1) {
        n_valid += __shfl_xor_sync(0xffffffffu, n_valid, o);
        n_finite += __shfl_xor_sync(0xffffffffu, n_finite, o);
    }
    __syncwarp();
    const int skip = drop_first ? 1 : 0;
    const int ksel = k + skip;
    for (int t = lane; t < k; t += 32) {
        int src = t + skip;
        int id = -1;
        double dv = CUDART_NAN;
        if (src < n_valid) {
            id = ix[src];
            dv = d[src];
            if (dv == CUDART_INF) dv = CUDART_NAN;
            id += idx_offset;
        }
        oi[t] = id;
        od[t] = dv;
    }
    if (cert.kind != NABO_CERT_NONE && lane == 0) {
        const float tau = tau_q;
        bool fail;
        if (tau == CUDART_INF_F) fail = n_valid < n_ref;          // nothing rejected <=> every reference is a candidate
        else if (n_finite < ksel) fail = true;
        else fail = !(d[ksel - 1] < cert_lower_bound(cert, qi, tau));
        if (fail) fail_rows[atomicAdd(fail_count, 1)] = qi;
    }
}

int nabo_rerank_launch(const double* q, int ldq, const double* r, int ldr, int n_query, int n_ref, int g, int k,
                       int metric, double f, const uint8_t* mask, int drop_first, int idx_offset,
                       const int32_t* cand, int n_cand, const NaboCert& cert, int* fail_rows, int* fail_count,
                       int32_t* out_idx, double* out_dist, const NaboRoute& route, cudaStream_t st,
                       const NaboCandBuf* from_buf, int row0, bool dependent) {
    // up to 128 candidates per query; 256 for Euclidean / cosine (the 256-key tensor-core plan, K' <= 160)
    const int max_cand = metric == NABO_MOD_CANBERRA ? 128 : 256;
    NABO_ARG(n_cand >= 1 && n_cand <= max_cand, "rerank: n_cand=%d unsupported (1..%d)", n_cand, max_cand);
    NABO_ARG(k >= 1 && k + (drop_first ? 1 : 0) <= n_cand, "rerank: k=%d does not fit n_cand=%d", k, n_cand);
    NABO_ARG(row0 >= 0 && row0 <= n_query, "rerank: row0=%d outside [0, %d]", row0, n_query);
    if (n_query - row0 == 0) return 0;
    int capp = nabo_next_pow2(n_cand);
    if (capp < 32) capp = 32;
    size_t smem = (size_t)4 * capp * (sizeof(double) + sizeof(int));
    const int xs_dims = g <= 1024 ? g : 0;                 // the query rides in shared memory when it is short enough
    smem += (size_t)4 * xs_dims * sizeof(double);
    if (from_buf) smem += (size_t)4 * 256 * sizeof(uint32_t);
    const bool vec2 = ((uintptr_t)r & 15) == 0 && (ldr & 1) == 0;
    dim3 grid((n_query - row0 + 3) / 4);
    NaboCandBuf cb;
    cb.buf = nullptr; cb.cnt = nullptr; cb.tau = nullptr; cb.kprime = 0;
    if (from_buf) {
        NABO_ARG(from_buf->kprime >= 1 && from_buf->kprime <= 64 && from_buf->kprime == n_cand,
                 "rerank: buffer mode needs K' = n_cand <= 64");
        cb = *from_buf;
    }
    // dependent launch: the kernel may start as soon as every CTA of the kernel in front of it on the stream has executed
    // griddepcontrol.launch_dependents (it never calls griddepcontrol.wait: what it reads was fenced before the signal)
    // (measured at config 2: letting these blocks share the busy SMs - one fits next to a candidate-kernel CTA - costs
    // that kernel 0.14 ms and hides 0.24 ms; a 16 KB shared-memory request that keeps them on the idle SMs only is
    // slower, the re-rank then outlasts the last wave)
    cudaLaunchConfig_t cfg = {};
    cudaLaunchAttribute attr[1];
    cfg.gridDim = grid; cfg.blockDim = dim3(128); cfg.dynamicSmemBytes = smem; cfg.stream = st;
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = dependent ? 1 : 0;
#define LAUNCH(M)                                                                                              \
    if (from_buf)                                                                                              \
        NABO_CUDA(cudaLaunchKernelEx(&cfg, rerank_kernel<M, true>, q, ldq, r, ldr, n_query, n_ref, g, k, f, mask, \
                                     drop_first, idx_offset, cand, n_cand, capp, cert, fail_rows, fail_count,  \
                                     out_idx, out_dist, route, cb, xs_dims, vec2, row0));                      \
    else                                                                                                       \
        NABO_CUDA(cudaLaunchKernelEx(&cfg, rerank_kernel<M, false>, q, ldq, r, ldr, n_query, n_ref, g, k, f, mask, \
                                     drop_first, idx_offset, cand, n_cand, capp, cert, fail_rows, fail_count,  \
                                     out_idx, out_dist, route, cb, xs_dims, vec2, row0));
#define LAUNCH_WIDE(M)                                                                                         \
    if (capp > 128)                                                                                            \
        NABO_CUDA(cudaLaunchKernelEx(&cfg, rerank_kernel<M, false, 8>, q, ldq, r, ldr, n_query, n_ref, g, k, f,   \
                                     mask, drop_first, idx_offset, cand, n_cand, capp, cert, fail_rows,        \
                                     fail_count, out_idx, out_dist, route, cb, xs_dims, vec2, row0));          \
    else LAUNCH(M)
    if (metric == NABO_EUCLIDEAN) { LAUNCH_WIDE(NABO_EUCLIDEAN) }
    else if (metric == NABO_MOD_CANBERRA) { LAUNCH(NABO_MOD_CANBERRA) }
    else if (metric == NABO_COSINE) { LAUNCH_WIDE(NABO_COSINE) }
    else return nabo_set_error(NABO_EINVAL, "rerank: unknown metric %d", metric);
#undef LAUNCH_WIDE
#undef LAUNCH
    NABO_LAUNCH_CHECK("rerank_kernel");
    return 0;
}

extern "C" int nabo_rerank_exact(const double* q, int ldq, const double* r, int ldr, int n_query, int n_ref,
                                 int g, int k, int metric, double dist_factor, const uint8_t* ref_mask,
                                 int drop_first, int idx_offset, const int32_t* cand, int n_cand,
                                 int32_t* out_idx, double* out_dist, void* stream) {
    NABO_ARG(q && r && cand && out_idx && out_dist, "rerank: null pointer");
    NABO_ARG(ldq >= g && ldr >= g, "rerank: leading dimension smaller than g");
    NABO_ARG(n_cand >= 1 && n_cand <= 128, "rerank: n_cand=%d unsupported (1..128)", n_cand);
    NaboCert none;
    none.kind = NABO_CERT_NONE; none.tau = nullptr; none.qn2 = nullptr; none.scal = nullptr; none.c_acc = 0.0; none.abs_slack = 0.0;
    NaboRoute plain;
    plain.n_parts = 0;
    return nabo_rerank_launch(q, ldq, r, ldr, n_query, n_ref, g, k, metric, dist_factor, ref_mask, drop_first,
                              idx_offset, cand, n_cand, none, nullptr, nullptr, out_idx, out_dist, plain,
                              (cudaStream_t)stream);
}
