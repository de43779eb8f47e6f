// Bit-sliced candidate pass for the modified Canberra metric (nabo/_mapping.py:29-45).
//
// d(x, y) = sum_k term_k with term_k = 1 unless |x_k - y_k| < f|x_k| ("unsaturated"), so
// d >= g - count(x, y), count = number of unsaturated dimensions.  A pair whose bound reaches the
// query's running threshold tau cannot enter the top-K' and needs no arithmetic at all.  This kernel
// evaluates an OVER-estimate of count for 32 references per machine word:
//
//   * every dimension is cut into NBINS value bins (edges = sample quantiles of the reference); a
//     reference word stores, per dimension, the cumulative bit planes P[p] = [bin(y) < p], p = 0..NBINS;
//   * the unsaturated y of a query form the interval (x - f|x|, x + f|x|); with lo / hi the bins of its
//     (outward rounded) end points, P[hi + 1] & ~P[lo] flags every reference whose bin meets the interval -
//     a superset of the unsaturated ones, for 32 references with two shared-memory loads and one LOP3;
//   * the g flag words are summed vertically with a carry-save adder tree (Harley-Seal, 2.25 LOP3 per
//     dimension) into a 6-bit sliced counter (8 bits for g > 56) and compared with need(tau) = min{c : g - c < tau};
//   * the surviving pairs (about 2 % once tau is warm) go through the dense FP32 evaluation
//     (same arithmetic and error bound nabo_cb_eps as canberra_candidates.cu) and the running top-K'
//     selection of select.cuh.
//
// Lanes are queries: a warp owns 32 queries for the whole reference sweep (their bin intervals live in
// registers, their thresholds / counts in a private shared-memory slice); the NW warps of a CTA share the
// reference tiles, which arrive by TMA bulk copies through an mbarrier ring that the warps re-arm
// themselves (last one out of a stage issues the next copy) - no producer warp, no CTA-wide barrier in
// the sweep.  32-query groups are dealt evenly to all CTAs.  Everything rejected has exact distance
// >= tau - eps, which is what the re-rank certificate (NABO_CERT_LINEAR) needs; results are identical to
// the exact engine.  Measured: the kernel time hardly depends on how many of the 12 warps are busy
// (6.6 ms with 2, 8.8 ms with 12, 100 k references): a warp's sweep is a chain of dependent LOP3 / LDS /
// FADD, so throughput is warps x per-warp latency, and both more warps (registers: 167 per thread) and
// more shared memory per warp are exhausted.
#include "common.cuh"
#include "knn_internal.cuh"
#include "ptx.cuh"
#include "select.cuh"

namespace cbs {

#ifdef NABO_CBS_PROF       // development cycle accounting of a busy warp's sweep (tools/probe_cb_prof.py):
                           // [0] tile waits [1] count bound [2] work list [3] FP32 evaluation [4] compaction
                           // [5] stage release [6] round set-up + final selection [7] busy warp-tiles [8] evaluation passes
                           // [9] compactions [10] survivors
__device__ unsigned long long g_cbs_prof[12];
#define CBS_PROF_DECL long long prof_[12] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0}; long long prof_t_ = clock64();
#define CBS_PROF(i) { const long long t1_ = clock64(); prof_[i] += t1_ - prof_t_; prof_t_ = t1_; }
#define CBS_PROF_COUNT(i, n) prof_[i] += (n);
#define CBS_PROF_FLUSH if (lane == 0) { for (int i_ = 0; i_ < 12; ++i_) atomicAdd(&g_cbs_prof[i_], (unsigned long long)prof_[i_]); }
#else
#define CBS_PROF_DECL
#define CBS_PROF(i)
#define CBS_PROF_COUNT(i, n)
#define CBS_PROF_FLUSH
#endif

using namespace sel;   // make_key, compact_select, compact_sort_inline

constexpr int NBINS = 32;                 // value bins per dimension
constexpr int NPL = NBINS + 1;            // cumulative planes per (dimension, word)
constexpr int SLEEP_NS = 400;             // suspend-time hint of the tile waits
constexpr int CAP = sel::CAP;
constexpr int MAX_STAGES = 4;
constexpr int EDGE_SAMPLE = 4096;
constexpr int TRIG_EXTRA = 24;            // keys above kprime that trigger a compaction

// Tile plan, a function of NB = ceil(g / 8) alone (one kernel instance per NB).
//   narrow, g <= 56: 12 warps, 128-reference tiles, 6-bit sliced counters (count <= 63), and the FP32 reference
//                    copy of canberra_candidates.cu ([tile64][k][64]);
//   wide, 57 <= g <= 128: the query bin intervals (4 NB registers) no longer fit 12 warps' register budget (168
//                    per thread), so 8 warps (up to 255); 8-bit counters (count <= 128); the per-warp FP32 query
//                    tiles (1 024 g bytes with 8 warps) leave room for two stages of 64-reference tiles up to
//                    g = 104 (with 448-entry work lists) and of 32-reference tiles up to g = 128.  64-reference tiles
//                    are faster where they fit (g = 100: 44 vs 56 ms per 100 k x 100 k call; DESIGN 4.3).  The FP32
//                    reference copy is this file's own [tile32][k][32] layout (pretile32_kernel), so any multiple of
//                    32 references is one contiguous span.
constexpr bool wide_of(int nb) { return nb >= 8; }
constexpr int nw_of(int nb) { return wide_of(nb) ? 8 : 12; }                        // warps per CTA
constexpr int rt_of(int nb) { return wide_of(nb) ? (nb <= 13 ? 64 : 32) : 128; }    // references per tile
constexpr int lc_of(int nb) { return wide_of(nb) ? 448 : 512; }                     // work-list entries per warp
constexpr int yw_of(int nb) { return wide_of(nb) ? 32 : 64; }                       // references per FP32 copy block
constexpr int cbits_of(int nb) { return wide_of(nb) ? 8 : 6; }                      // bit planes of the sliced counter

static inline int nblocks8(int g) { return (g + 7) / 8; }
// plane rows of one tile, padded to 16 bytes (bulk copies); the narrow tiles (4 x 33 words per dimension) need no pad
static inline size_t plane_tile_bytes(int g, int rt) { return ((size_t)g * (rt / 32) * NPL * 4 + 15) & ~(size_t)15; }
static inline size_t ys_tile_bytes(int g, int rt) { return (size_t)g * rt * 4; }

struct SmemPlan {
    int stages, nw, rt, yw;
    size_t stage_bytes, stage_off, xs_off, hist_off, work_off, tau_off, cnt_off, bar_off, total;
};
static SmemPlan plan_smem(int g) {
    SmemPlan p;
    const int nb = nblocks8(g), NW = nw_of(nb), LC = lc_of(nb);
    p.nw = NW; p.rt = rt_of(nb); p.yw = yw_of(nb);
    p.stage_bytes = plane_tile_bytes(g, p.rt) + ys_tile_bytes(g, p.rt);
    const size_t fixed = (size_t)NW * g * 32 * 4 + (size_t)NW * 256 * 4 + (size_t)NW * LC * 2 + (size_t)NW * 32 * 8 + 128;
    const size_t cap = 227 * 1024;
    p.stages = 0;
    for (int s = MAX_STAGES; s >= 2; --s)
        if (fixed + s * p.stage_bytes <= cap) { p.stages = s; break; }
    size_t o = 0;
    p.stage_off = o; o += (size_t)(p.stages > 0 ? p.stages : 2) * p.stage_bytes;
    p.xs_off = o; o += (size_t)NW * g * 32 * 4;
    p.hist_off = o; o += (size_t)NW * 256 * 4;
    p.work_off = o; o += (size_t)NW * LC * 2;
    p.tau_off = o; o += (size_t)NW * 32 * 4;
    p.cnt_off = o; o += (size_t)NW * 32 * 4;
    p.bar_off = o; o += 128;
    p.total = o;
    return p;
}

// ------------------------------------------------------------------ preparation kernels
// Bin edges of one dimension: NBINS-quantiles of a strided sample of the reference (any edges are valid,
// quantiles just make the bins equally selective).  edges[k][j], j < NBINS - 1, ascending.
__global__ void __launch_bounds__(1024)
edges_kernel(const double* __restrict__ r, int ld, int n_ref, float* __restrict__ edges) {
    __shared__ float v[EDGE_SAMPLE];
    const int k = blockIdx.x;
    const int ns = n_ref < EDGE_SAMPLE ? n_ref : EDGE_SAMPLE;
    for (int i = threadIdx.x; i < EDGE_SAMPLE; i += blockDim.x) {
        float x = CUDART_INF_F;
        if (i < ns) {
            const long long row = (long long)i * n_ref / ns;
            x = (float)r[row * ld + k];
            if (!(x == x)) x = CUDART_INF_F;
        }
        v[i] = x;
    }
    __syncthreads();
    for (int size = 2; size <= EDGE_SAMPLE; size <<= 1)
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int t = threadIdx.x; t < EDGE_SAMPLE / 2; t += blockDim.x) {
                const int lo = 2 * t - (t & (stride - 1)), hi = lo + stride;
                const bool up = (lo & size) == 0;
                const float a = v[lo], b = v[hi];
                if (up ? (b < a) : (a < b)) { v[lo] = b; v[hi] = a; }
            }
            __syncthreads();
        }
    if (threadIdx.x < NBINS - 1) {
        int pos = (int)(((long long)(threadIdx.x + 1) * ns) / NBINS) - 1;
        if (pos < 0) pos = 0;
        edges[k * (NBINS - 1) + threadIdx.x] = v[pos];
    }
}

__device__ __forceinline__ int bin_of(float y, const float* e) {
    int b = 0;
#pragma unroll
    for (int j = 0; j < NBINS - 1; ++j) b += (e[j] <= y) ? 1 : 0;
    return b;
}

// Cumulative planes of one (tile, dimension): word w of dimension k of a tile is at (k * WPT + w) * NPL words
// from the (16-byte aligned) tile start, bit i of it = reference tile * RT + w * 32 + i is live (in range, not
// masked) and bin(y) < p.  rt is the FP32 pre-tiled reference in YW-row blocks ([block][k][YW]).
template <int RT, int YW>
__global__ void __launch_bounds__(RT)
planes_kernel(const float* __restrict__ rt, const float* __restrict__ edges, const uint8_t* __restrict__ mask,
              int n_ref, int g, uint32_t* __restrict__ planes) {
    constexpr int WPT = RT / 32, YSH = YW == 64 ? 6 : 5;
    static_assert(YW == (1 << YSH), "copy block");
    __shared__ float e[NBINS - 1];
    const int tile = blockIdx.x, k = blockIdx.y;
    if (threadIdx.x < NBINS - 1) e[threadIdx.x] = edges[k * (NBINS - 1) + threadIdx.x];
    __syncthreads();
    const int ref = tile * RT + threadIdx.x;
    const bool live = ref < n_ref && !(mask && mask[ref]);
    const float y = live ? rt[((size_t)(ref >> YSH) * g + k) * YW + (ref & (YW - 1))] : 0.f;
    const int b = bin_of(y, e);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const size_t tile_words = (WPT * NPL) % 4 == 0 ? (size_t)g * WPT * NPL : ((size_t)g * WPT * NPL + 3) & ~(size_t)3;
    uint32_t* out = planes + (size_t)tile * tile_words + ((size_t)k * WPT + w) * NPL;
#pragma unroll
    for (int p = 0; p < NPL; ++p) {
        const uint32_t bits = __ballot_sync(0xffffffffu, live && b < p && p <= NBINS);
        if (lane == (p & 31)) out[p] = bits;
    }
}

// Per (query, dimension) plane indices: low byte = lo, high byte = hi + 1, 0 / 0 for an empty
// interval (x = 0 or NaN: nothing is unsaturated).  Two dimensions per 32-bit word, lanes interleaved:
// ctrl[(group32 * nj + j) * 32 + lane].  The interval is widened by 1e-6 relative (FP64 rounding of the
// reference's own test) and its end points are rounded outward to FP32 - the precision the planes were
// binned in; float rounding is monotone, so bin(y) of every unsaturated y lies in [lo, hi].
__global__ void __launch_bounds__(256)
ctrl_kernel(const double* __restrict__ q, int ld, int n_query, int g, int nj, double f,
            const float* __restrict__ edges, uint32_t* __restrict__ ctrl, long long total) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= total) return;
    const int lane = (int)(e & 31);
    const long long gj = e >> 5;
    const int j = (int)(gj % nj);
    const long long row = (gj / nj) * 32 + lane;
    uint32_t word = 0;
    for (int h = 0; h < 2; ++h) {
        const int k = 2 * j + h;
        uint32_t c = 0;
        if (row < n_query && k < g) {
            const double x = q[row * ld + k];
            const double t = f * fabs(x) * (1.0 + 1e-6);
            if (t > 0.0) {
                const float lo_v = __double2float_rd(x - t), hi_v = __double2float_ru(x + t);
                const float* ed = edges + k * (NBINS - 1);
                int lo = 0, hi = 0;
                for (int i = 0; i < NBINS - 1; ++i) {
                    const float ev = ed[i];
                    lo += (ev <= lo_v) ? 1 : 0;
                    hi += (ev <= hi_v) ? 1 : 0;
                }
                if (!(hi_v == hi_v)) hi = NBINS - 1;      // x + t overflowed to NaN / inf: keep everything
                if (!(lo_v == lo_v)) lo = 0;
                c = (uint32_t)lo | ((uint32_t)(hi + 1) << 8);
            }
        }
        word |= c << (16 * h);
    }
    ctrl[e] = word;
}

// FP32 rows, 32 per group, dimension-major: qx[(group32 * g + k) * 32 + lane] (the queries; in the wide plan the
// reference copy too)
__global__ void __launch_bounds__(256)
pretile32_kernel(const double* __restrict__ x, int ld, int n, int g, float* __restrict__ out, long long total) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= total) return;
    const int lane = (int)(e & 31);
    const long long gk = e >> 5;
    const int k = (int)(gk % g);
    const long long row = (gk / g) * 32 + lane;
    out[e] = row < n ? (float)x[row * ld + k] : 0.f;
}

// ------------------------------------------------------------------ the sweep
struct Params {
    const uint32_t* planes;     // [n_tiles][g][WPT][NPL], tiles padded to 16 bytes
    const float* rt;            // [n_yblk][g][YW]
    const float* qx;            // [n_groups][g][32]
    const uint32_t* ctrl;       // [n_groups][nj][32]
    int n_query, n_ref, g, n_tiles, n_yblk, n_groups, kprime, stages, nj, n_split;
    float fm;
    int trig_extra;
    unsigned long long* cand_buf;   // [gridDim][NW * 32][CAP]
    int32_t* cand;              // [n_query][kprime]
    float* tau_out;             // [n_query]
    size_t stage_bytes, stage_off, xs_off, hist_off, work_off, tau_off, cnt_off, bar_off;
};

struct Barriers {
    uint64_t full[MAX_STAGES];
    int done[MAX_STAGES];
};

__device__ __forceinline__ float rcp_approx(float x) {       // MUFU.RCP, 1 ulp: inside the nabo_cb_eps margin
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}

#define NABO_CSA(h, l, a, b, c)                           \
    {                                                     \
        const uint32_t u_ = (a) ^ (b);                    \
        const uint32_t c_ = (c);                          \
        h = ((a) & (b)) | (u_ & c_);                      \
        l = u_ ^ c_;                                      \
    }

// smallest count c with (float)g - c < tau, clamped to [0, NEVER]; NEVER (all counter bits set) exceeds every
// count the counter holds (g <= 63 in 6 bits, g <= 128 in 8), so it rejects everything (tau = -inf, padding queries)
template <int NEVER>
__device__ __forceinline__ int need_of(float tau, int g) {
    if (!(tau > -CUDART_INF_F)) return NEVER;
    if (tau == CUDART_INF_F) return 0;
    int c = (int)floorf((float)g - tau) + 1;
    if (c < 0) c = 0;
    while (c > 0 && (float)(g - (c - 1)) < tau) --c;
    while (c < NEVER && !((float)(g - c) < tau)) ++c;
    return c > NEVER ? NEVER : c;
}

template <int NB, bool SPLIT>      // SPLIT: the CTAs of one query block share out the reference range (n_split > 1)
__global__ void __launch_bounds__(nw_of(NB) * 32, 1)
sliced_kernel(const Params p) {
    constexpr int NW = nw_of(NB), QB = NW * 32;
    constexpr int RT = rt_of(NB), WPT = RT / 32;
    constexpr int YW = yw_of(NB), YSH = YW == 64 ? 6 : 5, TY = RT / YW;    // FP32 copy blocks per tile
    constexpr int CB = cbits_of(NB), NEVER = (1 << CB) - 1;
    constexpr int LC = lc_of(NB);
    static_assert(YW == (1 << YSH) && RT <= 128 && NB * 8 <= NEVER && LC >= 256, "tile plan");
    extern __shared__ __align__(128) unsigned char smem[];
    Barriers* bars = reinterpret_cast<Barriers*>(smem + p.bar_off);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = p.g;

    // Work = 32-query groups, dealt evenly to the CTAs; a CTA sweeps the reference once per round with
    // as many of its warps busy as it has groups left (balanced over the rounds).  Dealing whole
    // NW-group items instead would leave most SMs idle whenever n_query / (32 NW) is not a multiple of the grid.
    // With few groups (a CTA would keep one or two warps busy, and a warp's sweep is latency-bound) the
    // reference range is cut into n_split pieces: CTA b sweeps piece b % n_split for query block b / n_split,
    // each piece yields its own K' list and threshold, the re-rank takes their union / minimum.
    const int n_seg = SPLIT ? p.n_split : 1;
    const int seg = SPLIT ? (int)(blockIdx.x % (unsigned)n_seg) : 0;
    const int qblock = SPLIT ? (int)(blockIdx.x / (unsigned)n_seg) : (int)blockIdx.x;
    const int n_qblocks = SPLIT ? (int)(gridDim.x / (unsigned)n_seg) : (int)gridDim.x;
    const int tile0 = SPLIT ? (int)((long long)p.n_tiles * seg / n_seg) : 0;
    const int n_tiles = SPLIT ? (int)((long long)p.n_tiles * (seg + 1) / n_seg) - tile0 : p.n_tiles;
    const int g_begin = (int)((long long)p.n_groups * qblock / n_qblocks);
    const int n_mine = (int)((long long)p.n_groups * (qblock + 1) / n_qblocks) - g_begin;
    const int rounds = (n_mine + NW - 1) / NW;
    const int wpr = rounds > 0 ? (n_mine + rounds - 1) / rounds : 0;      // busy warps per round
    const uint32_t total_tiles = (uint32_t)rounds * (uint32_t)n_tiles;

    // Reference tiles arrive by TMA bulk copies into a ring of p.stages buffers (full[] mbarriers).  There
    // is no producer warp: every warp counts itself out of a stage when it is done with the tile, and the
    // last one out re-arms the stage with the tile p.stages ahead - the earliest moment it can be issued.
    const uint32_t plane_bytes = (WPT * NPL) % 4 == 0 ? (uint32_t)((size_t)g * WPT * NPL * 4)
                                                      : ((uint32_t)((size_t)g * WPT * NPL * 4) + 15u) & ~15u;
    auto issue_tile = [&](uint32_t tn, uint32_t s) {          // one thread
        const int j = tile0 + (int)(tn % (uint32_t)n_tiles);
        const int ny = min(TY, p.n_yblk - TY * j);
        const uint32_t ys_bytes = (uint32_t)ny * g * YW * 4;
        ptx::mbar_arrive_expect_tx(&bars->full[s], plane_bytes + ys_bytes);
        char* dst = reinterpret_cast<char*>(smem + p.stage_off + (size_t)s * p.stage_bytes);
        const char* src = reinterpret_cast<const char*>(p.planes) + (size_t)j * plane_bytes;
        for (uint32_t o = 0; o < plane_bytes; o += 16384)
            ptx::bulk_g2s(dst + o, src + o, min(16384u, plane_bytes - o), &bars->full[s]);
        dst += plane_bytes;
        src = reinterpret_cast<const char*>(p.rt) + (size_t)j * TY * g * YW * 4;
        for (uint32_t o = 0; o < ys_bytes; o += 16384)
            ptx::bulk_g2s(dst + o, src + o, min(16384u, ys_bytes - o), &bars->full[s]);
    };
    auto release_tile = [&](uint32_t t, uint32_t s) {         // whole warp, after its last read of the stage
        __syncwarp();
        if (lane == 0) {
            __threadfence_block();
            if (atomicAdd(&bars->done[s], 1) == NW - 1) {
                bars->done[s] = 0;
                __threadfence_block();
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                if (t + p.stages < total_tiles) issue_tile(t + p.stages, s);
            }
        }
    };

    if (threadIdx.x == 0) {
        for (int s = 0; s < p.stages; ++s) { ptx::mbar_init(&bars->full[s], 1); bars->done[s] = 0; }
        ptx::fence_barrier_init();
        for (uint32_t tn = 0; tn < (uint32_t)p.stages && tn < total_tiles; ++tn) issue_tile(tn, tn);
    }
    __syncthreads();

    // ===================== consumers: lanes = queries =====================
    float* xs = reinterpret_cast<float*>(smem + p.xs_off) + (size_t)warp * g * 32;
    uint32_t* hist = reinterpret_cast<uint32_t*>(smem + p.hist_off) + (size_t)warp * 256;
    unsigned short* work = reinterpret_cast<unsigned short*>(smem + p.work_off) + (size_t)warp * LC;
    float* s_tau = reinterpret_cast<float*>(smem + p.tau_off) + warp * 32;
    int* s_cnt = reinterpret_cast<int*>(smem + p.cnt_off) + warp * 32;
    unsigned long long* gbuf = p.cand_buf + ((size_t)blockIdx.x * QB + warp * 32) * CAP;
    const float fm = p.fm;
    const int kprime = p.kprime;

    // dense FP32 evaluation of the first n work-list entries of the current tile.  A lane takes TWO entries per pass
    // when more than 32 are left: the two dependency chains (load, rcp, select, add) interleave, and a
    // warp's sweep is latency-bound.  A pass then adds at most 64 keys to one query, so the buffers are kept at or
    // below CAP - 64 (dual passes are used only when kprime + trig_extra allows that).
    CBS_PROF_DECL
    const int trig = min(CAP - 32, kprime + p.trig_extra);
    const bool dual_ok = trig <= CAP - 64;
    auto compact_due = [&]() {
        // compacting earlier than the buffer limit (kprime + trig_extra keys) keeps tau closer to the true running
        // K'-th best score: a stale threshold lets proportionally more pairs through to the dense evaluation
        unsigned need = __ballot_sync(0xffffffffu, s_cnt[lane] > trig);
        if (need) CBS_PROF(3)
        while (need) {
            const int src = __ffs(need) - 1;
            need &= need - 1;
            int nc;
            float nt;
            compact_select<CAP / 32>(gbuf + (size_t)src * CAP, s_cnt[src], lane, kprime, trig - 4 > kprime ? trig - 4 : kprime, hist, nc, nt);
            if (lane == src) { s_cnt[lane] = nc; s_tau[lane] = nt; }
            __syncwarp();
            CBS_PROF_COUNT(9, 1)
            CBS_PROF(4)
        }
    };
    auto evaluate = [&](int n, const float* ys, int ref0) {
        int base = 0;
        CBS_PROF_COUNT(10, n)
        while (base < n) {
            CBS_PROF_COUNT(8, 1)
            if (dual_ok && n - base > 32) {
                const int i0 = base + lane, i1 = base + 32 + lane;
                const bool act1 = i1 < n;
                const int e0 = work[i0], e1 = act1 ? work[i1] : 0;
                const int ql0 = e0 >> 8, rl0 = e0 & 127, ql1 = e1 >> 8, rl1 = e1 & 127;
                const float* xb0 = xs + ql0;
                const float* yb0 = ys + (rl0 >> YSH) * (g * YW) + (rl0 & (YW - 1));
                const float* xb1 = xs + ql1;
                const float* yb1 = ys + (rl1 >> YSH) * (g * YW) + (rl1 & (YW - 1));
                float acc0 = 0.f, acc1 = 0.f;
#pragma unroll 5
                for (int k = 0; k < g; ++k) {
                    const float x0 = xb0[k * 32], y0 = yb0[k * YW];
                    const float x1 = xb1[k * 32], y1 = yb1[k * YW];
                    const float num0 = fabsf(x0 - y0), xa0 = fabsf(x0);
                    const float num1 = fabsf(x1 - y1), xa1 = fabsf(x1);
                    const float term0 = fmaf(num0, rcp_approx(xa0 + (fabsf(y0) + 0.01f)), -1.0f);
                    const float term1 = fmaf(num1, rcp_approx(xa1 + (fabsf(y1) + 0.01f)), -1.0f);
                    if (num0 < fm * xa0) acc0 += term0;           // distance = g + sum over the unsaturated of (term - 1)
                    if (num1 < fm * xa1) acc1 += term1;
                }
                acc0 += (float)g; acc1 += (float)g;
                if (acc0 < s_tau[ql0]) {
                    const int pos = atomicAdd(&s_cnt[ql0], 1);
                    NABO_DEV_ASSERT(pos >= 0 && pos < CAP && ql0 >= 0 && ql0 < 32);
                    gbuf[(size_t)ql0 * CAP + pos] = make_key(acc0, (uint32_t)(ref0 + rl0));
                }
                if (act1 && acc1 < s_tau[ql1]) {
                    const int pos = atomicAdd(&s_cnt[ql1], 1);
                    NABO_DEV_ASSERT(pos >= 0 && pos < CAP && ql1 >= 0 && ql1 < 32);
                    gbuf[(size_t)ql1 * CAP + pos] = make_key(acc1, (uint32_t)(ref0 + rl1));
                }
                base += 64;
            } else {
                const int i = base + lane;
                const bool active = i < n;
                const int e = active ? work[i] : 0;
                const int ql = e >> 8, rl = e & 127;
                const float* xb = xs + ql;
                const float* yb = ys + (rl >> YSH) * (g * YW) + (rl & (YW - 1));
                float acc = 0.f;
#pragma unroll 5
                for (int k = 0; k < g; ++k) {
                    const float x = xb[k * 32], y = yb[k * YW];
                    const float num = fabsf(x - y), xa = fabsf(x);
                    const float term = fmaf(num, rcp_approx(xa + (fabsf(y) + 0.01f)), -1.0f);
                    if (num < fm * xa) acc += term;
                }
                acc += (float)g;
                if (active && acc < s_tau[ql]) {
                    const int pos = atomicAdd(&s_cnt[ql], 1);
                    NABO_DEV_ASSERT(pos >= 0 && pos < CAP && ql >= 0 && ql < 32);
                    gbuf[(size_t)ql * CAP + pos] = make_key(acc, (uint32_t)(ref0 + rl));
                }
                base += 32;
            }
            __syncwarp();
            compact_due();
        }
    };

    uint32_t t = 0;
    for (int round = 0; round < rounds; ++round) {
        const int gi = round * wpr + warp;
        if (warp >= wpr || gi >= n_mine) {
            // no group for this warp in this round: keep the tile ring moving
            for (int j = 0; j < n_tiles; ++j, ++t) {
                const uint32_t s = t % p.stages, use = t / p.stages;
                ptx::mbar_wait_hint(&bars->full[s], use & 1, SLEEP_NS);
                release_tile(t, s);
            }
            continue;
        }
        const int group = g_begin + gi;
        const long long q_mine = (long long)group * 32 + lane;
        uint32_t ctrl[NB * 4];
#pragma unroll
        for (int j = 0; j < NB * 4; ++j) ctrl[j] = p.ctrl[((size_t)group * p.nj + j) * 32 + lane];
        for (int e = lane; e < g * 32; e += 32) xs[e] = p.qx[(size_t)group * g * 32 + e];
        s_tau[lane] = q_mine < p.n_query ? CUDART_INF_F : -CUDART_INF_F;     // padding queries reject everything
        s_cnt[lane] = 0;
        __syncwarp();
        CBS_PROF(6)

        for (int jl = 0; jl < n_tiles; ++jl, ++t) {
            const int j = tile0 + jl;
            const uint32_t s = t % p.stages, use = t / p.stages;
            ptx::mbar_wait_hint(&bars->full[s], use & 1, SLEEP_NS);   // sleep, do not poll: 10 % of the issue slots went here
            CBS_PROF_COUNT(7, 1)
            CBS_PROF(0)
            const unsigned char* stage = smem + p.stage_off + (size_t)s * p.stage_bytes;
            const char* pl = reinterpret_cast<const char*>(stage);
            const float* ys = reinterpret_cast<const float*>(stage + plane_bytes);

            // ---- phase 0: sliced over-estimate of the unsaturated-dimension count, WPT x 32 references per lane
            if constexpr (wide_of(NB)) {
                // the plane offsets derived from ctrl are loop-invariant; hoisted out of the tile loop they would
                // take 2 g registers instead of g / 2 and spill
#pragma unroll
                for (int jj = 0; jj < NB * 4; ++jj) asm volatile("" : "+r"(ctrl[jj]));
            }
            uint32_t c[WPT][CB];
#pragma unroll
            for (int w = 0; w < WPT; ++w)
#pragma unroll
                for (int b = 0; b < CB; ++b) c[w][b] = 0u;
#pragma unroll
            for (int blk = 0; blk < NB; ++blk) {
                uint32_t v[8][WPT];
#pragma unroll
                for (int d = 0; d < 8; ++d) {
                    const int k = blk * 8 + d;
                    if (blk < NB - 1 || k < g) {
                        const uint32_t cw = ctrl[k >> 1];
                        const uint32_t lo4 = ((k & 1) ? ((cw >> 16) & 0xffu) : (cw & 0xffu)) * 4u;
                        const uint32_t hi4 = ((k & 1) ? (cw >> 24) : ((cw >> 8) & 0xffu)) * 4u;
                        const char* base = pl + k * (WPT * NPL * 4);
#pragma unroll
                        for (int w = 0; w < WPT; ++w) {
                            const uint32_t a = *reinterpret_cast<const uint32_t*>(base + w * NPL * 4 + hi4);
                            const uint32_t b = *reinterpret_cast<const uint32_t*>(base + w * NPL * 4 + lo4);
                            v[d][w] = a & ~b;
                        }
                    } else {
#pragma unroll
                        for (int w = 0; w < WPT; ++w) v[d][w] = 0u;
                    }
                }
#pragma unroll
                for (int w = 0; w < WPT; ++w) {
                    uint32_t t2a, t2b, f4a, f4b, e8;
                    NABO_CSA(t2a, c[w][0], c[w][0], v[0][w], v[1][w]);
                    NABO_CSA(t2b, c[w][0], c[w][0], v[2][w], v[3][w]);
                    NABO_CSA(f4a, c[w][1], c[w][1], t2a, t2b);
                    NABO_CSA(t2a, c[w][0], c[w][0], v[4][w], v[5][w]);
                    NABO_CSA(t2b, c[w][0], c[w][0], v[6][w], v[7][w]);
                    NABO_CSA(f4b, c[w][1], c[w][1], t2a, t2b);
                    NABO_CSA(e8, c[w][2], c[w][2], f4a, f4b);
                    const uint32_t k1 = c[w][3] & e8;
                    if constexpr (CB == 8) {      // ripple the carry of weight 16 up to weight 128
                        const uint32_t k2 = c[w][4] & k1, k3 = c[w][5] & k2;
                        c[w][7] ^= c[w][6] & k3;
                        c[w][6] ^= k3;
                        c[w][5] ^= k2;
                    } else {
                        c[w][5] ^= c[w][4] & k1;
                    }
                    c[w][4] ^= k1;
                    c[w][3] ^= e8;
                }
            }
            // count >= need(tau), per lane
            const int need_c = need_of<NEVER>(s_tau[lane], g);
            uint32_t m[WPT];
#pragma unroll
            for (int w = 0; w < WPT; ++w) {
                uint32_t gt = 0u, eq = 0xffffffffu;
#pragma unroll
                for (int b = CB - 1; b >= 0; --b) {
                    const uint32_t nb = 0u - (uint32_t)((need_c >> b) & 1);
                    gt |= eq & c[w][b] & ~nb;
                    eq &= ~(c[w][b] ^ nb);
                }
                const uint32_t live = *reinterpret_cast<const uint32_t*>(pl + (w * NPL + NBINS) * 4);
                m[w] = (gt | eq) & live;
            }

            CBS_PROF(1)
            // ---- survivors -> work list -> phase 2
            int mine = 0;
#pragma unroll
            for (int w = 0; w < WPT; ++w) mine += __popc(m[w]);
            const int total = __reduce_add_sync(0xffffffffu, mine);
            if (total > 0) {
                if (total <= LC) {
                    int incl = mine;
#pragma unroll
                    for (int o = 1; o < 32; o <<= 1) {
                        const int u = __shfl_up_sync(0xffffffffu, incl, o);
                        if (lane >= o) incl += u;
                    }
                    int pos = incl - mine;
#pragma unroll
                    for (int w = 0; w < WPT; ++w) {
                        uint32_t mm = m[w];
                        while (mm) {
                            const int b = __ffs(mm) - 1;
                            mm &= mm - 1;
                            work[pos++] = (unsigned short)((lane << 8) | (w * 32 + b));
                        }
                    }
                    __syncwarp();
                    CBS_PROF(2)
                    evaluate(total, ys, j * RT);
                    CBS_PROF(3)
                } else {
                    // dense tile (cold threshold): one byte column of one word at a time, at most 256 entries
                    for (int w = 0; w < WPT; ++w) {
                        for (int bg = 0; bg < 4; ++bg) {
                            uint32_t mm = 0;
#pragma unroll
                            for (int ww = 0; ww < WPT; ++ww)
                                if (ww == w) mm = m[ww];
                            mm &= 0xffu << (8 * bg);
                            const int cntl = __popc(mm);
                            const int tot = __reduce_add_sync(0xffffffffu, cntl);
                            if (tot == 0) continue;
                            int incl = cntl;
#pragma unroll
                            for (int o = 1; o < 32; o <<= 1) {
                                const int u = __shfl_up_sync(0xffffffffu, incl, o);
                                if (lane >= o) incl += u;
                            }
                            int pos = incl - cntl;
                            while (mm) {
                                const int b = __ffs(mm) - 1;
                                mm &= mm - 1;
                                work[pos++] = (unsigned short)((lane << 8) | (w * 32 + b));
                            }
                            __syncwarp();
                            CBS_PROF(2)
                            evaluate(tot, ys, j * RT);
                            CBS_PROF(3)
                        }
                    }
                }
            }
            CBS_PROF(2)
            release_tile(t, s);
            CBS_PROF(5)
        }

        // ---- round done: exact selection of every query of this warp, emit candidates + threshold
        for (int src = 0; src < 32; ++src) {
            const int n = s_cnt[src];
            const float old_tau = s_tau[src];
            uint32_t ks[4], kpl[4];
            int nc;
            float nt;
            compact_sort_inline(gbuf + (size_t)src * CAP, n, lane, kprime, ks, kpl, nc, nt);
            const long long qg = (long long)group * 32 + src;
            if (qg < p.n_query) {
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int i = u * 32 + lane;
                    if (i < kprime) p.cand[(qg * n_seg + seg) * kprime + i] = i < nc ? (int32_t)kpl[u] : -1;
                }
                if (lane == 0) p.tau_out[(long long)seg * p.n_query + qg] = n >= kprime ? nt : old_tau;
            }
        }
        __syncwarp();
        CBS_PROF(6)
    }
    CBS_PROF_FLUSH
}

}  // namespace cbs

#ifdef NABO_CBS_PROF
extern "C" int nabo_dbg_cbs_prof(unsigned long long* out_host, int reset) {
    cudaDeviceSynchronize();
    cudaMemcpyFromSymbol(out_host, cbs::g_cbs_prof, sizeof(unsigned long long) * 12);
    if (reset) { unsigned long long z[12] = {0}; cudaMemcpyToSymbol(cbs::g_cbs_prof, z, sizeof(z)); }
    return 0;
}
#endif

// ------------------------------------------------------------------ host side
bool nabo_cbs_supported(int g, int k, int drop_first) {
    if (g < 1 || g > 128) return false;
    const int ksel = k + (drop_first ? 1 : 0);
    return cbs::plan_smem(g).stages >= 2 && ksel + 8 <= cbs::CAP - 64;
}

static int cbs_grid(int n_groups) {
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    return n_groups < sms ? n_groups : sms;
}

// planes + bin edges: the reference half of the extra workspace (and of a prepared reference's buffer)
static size_t cbs_ref_extra_bytes(int n_ref, int g) {
    const cbs::SmemPlan pl = cbs::plan_smem(g);
    const size_t n_tiles = (n_ref + pl.rt - 1) / pl.rt;
    return nabo_align_up(n_tiles * cbs::plane_tile_bytes(g, pl.rt), 256) +
           nabo_align_up((size_t)g * (cbs::NBINS - 1) * 4, 256);
}

size_t nabo_cbs_extra_bytes(int n_query, int n_ref, int g, bool with_ref) {
    const cbs::SmemPlan pl = cbs::plan_smem(g);
    const size_t n_groups = (size_t)(n_query + 31) / 32;
    const int nj = cbs::nblocks8(g) * 4;
    size_t b = 0;
    if (with_ref) b += cbs_ref_extra_bytes(n_ref, g);
    b += nabo_align_up(n_groups * nj * 32 * 4, 256);
    b += nabo_align_up(n_groups * g * 32 * 4, 256);
    b += nabo_align_up((size_t)148 * pl.nw * 32 * cbs::CAP * 8, 256);
    return b + 1024;
}

// rt: FP32 copy of the reference (nabo_cb_pretile_floats(n_ref, g) floats: [tile64][k][64], or [tile32][k][32] in
// the wide plan), filled here.
// Pieces the reference range is cut into (see the kernel): only when a CTA would have at most half of its warps
// busy, never below 8 192 references per piece, and the union of the K' lists must fit the re-rank (128).
int nabo_cbs_split(int n_query, int n_ref, int g, int k, int drop_first) {
    const cbs::SmemPlan pl = cbs::plan_smem(g);
    const int n_groups = (n_query + 31) / 32;
    const int n_tiles = (n_ref + pl.rt - 1) / pl.rt;
    const int per_cta = (n_groups + cbs_grid(1 << 30) - 1) / cbs_grid(1 << 30);
    int s = per_cta > 0 ? pl.nw / per_cta : 1;
    if (s > NABO_CBS_MAX_SPLIT) s = NABO_CBS_MAX_SPLIT;
    while (s > 1 && (n_tiles / s < 8192 / pl.rt || s * nabo_cb_kprime(k, drop_first) > 128)) --s;
    return s < 1 ? 1 : s;
}

// The reference half of the sliced pass: the FP32 copy rt (nabo_cb_pretile_floats(n_ref, g) floats), the bin edges
// and the cumulative planes.  None of it depends on the queries or on dist_factor.
static int cbs_ref_launch(const double* r, int ldr, int n_ref, int g, const uint8_t* mask, float* rt, float* edges,
                          uint32_t* planes, cudaStream_t st) {
    const cbs::SmemPlan pl = cbs::plan_smem(g);
    const int n_tiles = (n_ref + pl.rt - 1) / pl.rt;
    const int n_yblk = (n_ref + pl.yw - 1) / pl.yw;
    if (pl.yw == 64) {
        int rc = nabo_cb_pretile_launch(r, ldr, n_ref, g, rt, st);
        if (rc) return rc;
    } else {
        const long long tr = (long long)n_yblk * g * 32;
        cbs::pretile32_kernel<<<(unsigned)((tr + 255) / 256), 256, 0, st>>>(r, ldr, n_ref, g, rt, tr);
    }
    cbs::edges_kernel<<<g, 1024, 0, st>>>(r, ldr, n_ref, edges);
    switch (pl.rt) {
        case 128: cbs::planes_kernel<128, 64><<<dim3(n_tiles, g), 128, 0, st>>>(rt, edges, mask, n_ref, g, planes); break;
        case 64: cbs::planes_kernel<64, 32><<<dim3(n_tiles, g), 64, 0, st>>>(rt, edges, mask, n_ref, g, planes); break;
        default: cbs::planes_kernel<32, 32><<<dim3(n_tiles, g), 32, 0, st>>>(rt, edges, mask, n_ref, g, planes); break;
    }
    return 0;
}

size_t nabo_cbs_prepared_bytes(int n_ref, int g) {
    return nabo_align_up(nabo_cb_pretile_floats(n_ref, g) * 4, 256) + cbs_ref_extra_bytes(n_ref, g);
}

// A prepared reference's sliced operands, in the layout nabo_cbs_candidates builds per call.
int nabo_cbs_prepare_ref(const double* r, int ldr, int n_ref, int g, const uint8_t* mask, void* buffer, NaboCbsRef* out,
                         cudaStream_t st) {
    const cbs::SmemPlan pl = cbs::plan_smem(g);
    const int n_tiles = (n_ref + pl.rt - 1) / pl.rt;
    NaboArena ar(buffer, nabo_cbs_prepared_bytes(n_ref, g));
    float* rt = ar.take<float>(nabo_cb_pretile_floats(n_ref, g));
    uint32_t* planes = (uint32_t*)ar.take<char>((size_t)n_tiles * cbs::plane_tile_bytes(g, pl.rt));
    float* edges = ar.take<float>((size_t)g * (cbs::NBINS - 1));
    if (!ar.ok) return nabo_set_error(NABO_EINVAL, "ref_prepare: buffer layout");
    int rc = cbs_ref_launch(r, ldr, n_ref, g, mask, rt, edges, planes, st);
    if (rc) return rc;
    NABO_LAUNCH_CHECK("cbs reference preparation");
    out->rt = rt;
    out->planes = planes;
    out->edges = edges;
    return 0;
}

// cand: [n_query][n_split][K'], tau: [n_split][n_query].  pre != NULL: rt, planes and edges come from a prepared
// reference (rt, r and mask are not read); extra then needs only the query half (nabo_cbs_extra_bytes(.., false)).
int nabo_cbs_candidates(const double* q, int ldq, const double* r, int ldr, int n_query, int n_ref, int g, int k,
                        double f, const uint8_t* mask, int drop_first, int n_split, float* rt, void* extra,
                        size_t extra_bytes, int32_t* cand, float* tau, cudaStream_t st, const NaboCbsRef* pre) {
    const int kprime = nabo_cb_kprime(k, drop_first);
    if (n_split < 1 || n_split > NABO_CBS_MAX_SPLIT) n_split = 1;
    const cbs::SmemPlan pl = cbs::plan_smem(g);
    const int n_tiles = (n_ref + pl.rt - 1) / pl.rt;
    const int n_yblk = (n_ref + pl.yw - 1) / pl.yw;
    const size_t n_groups = (size_t)(n_query + 31) / 32;
    const int nb = cbs::nblocks8(g), nj = nb * 4;
    int grid = cbs_grid((int)n_groups * n_split);
    if (n_split > 1) grid = grid / n_split * n_split;      // whole query blocks
    if (grid < n_split) n_split = 1, grid = cbs_grid((int)n_groups);

    NaboArena ar(extra, extra_bytes);
    uint32_t* planes = pre ? (uint32_t*)pre->planes : (uint32_t*)ar.take<char>((size_t)n_tiles * cbs::plane_tile_bytes(g, pl.rt));
    float* edges = pre ? (float*)pre->edges : ar.take<float>((size_t)g * (cbs::NBINS - 1));
    uint32_t* ctrl = ar.take<uint32_t>(n_groups * nj * 32);
    float* qx = ar.take<float>(n_groups * g * 32);
    unsigned long long* cbuf = ar.take<unsigned long long>((size_t)grid * pl.nw * 32 * cbs::CAP);
    if (!ar.ok) return nabo_set_error(NABO_EWORKSPACE, "knn: workspace too small for the sliced Canberra pass");
    if (pre) rt = (float*)pre->rt;

    {
        if (!pre) {
            int rc = cbs_ref_launch(r, ldr, n_ref, g, mask, rt, edges, planes, st);
            if (rc) return rc;
        }
        const long long tc = (long long)n_groups * nj * 32;
        cbs::ctrl_kernel<<<(unsigned)((tc + 255) / 256), 256, 0, st>>>(q, ldq, n_query, g, nj, f, edges, ctrl, tc);
        const long long tq = (long long)n_groups * g * 32;
        cbs::pretile32_kernel<<<(unsigned)((tq + 255) / 256), 256, 0, st>>>(q, ldq, n_query, g, qx, tq);
        NABO_LAUNCH_CHECK("cbs preparation kernels");
    }

    cbs::Params p;
    p.planes = planes; p.rt = rt; p.qx = qx; p.ctrl = ctrl;
    p.n_query = n_query; p.n_ref = n_ref; p.g = g; p.n_tiles = n_tiles; p.n_yblk = n_yblk;
    p.n_groups = (int)n_groups; p.kprime = kprime; p.stages = pl.stages; p.nj = nj; p.n_split = n_split;
    const double delta = fmax(1e-5, 4e-7 * (2.0 + f) / f);      // same optimistic margin as canberra_candidates.cu
    p.fm = (float)(f * (1.0 + delta));
    p.cand_buf = cbuf; p.cand = cand; p.tau_out = tau;
    p.trig_extra = cbs::TRIG_EXTRA;
    p.stage_bytes = pl.stage_bytes; p.stage_off = pl.stage_off; p.xs_off = pl.xs_off; p.hist_off = pl.hist_off;
    p.work_off = pl.work_off; p.tau_off = pl.tau_off; p.cnt_off = pl.cnt_off; p.bar_off = pl.bar_off;
    const int threads = pl.nw * 32;
#define NABO_CBS_LAUNCH(NBV)                                                                                       \
    case NBV:                                                                                                      \
        if (n_split > 1) {                                                                                         \
            NABO_CUDA(cudaFuncSetAttribute(cbs::sliced_kernel<NBV, true>,                                          \
                                           cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.total));           \
            cbs::sliced_kernel<NBV, true><<<grid, threads, pl.total, st>>>(p);                                     \
        } else {                                                                                                   \
            NABO_CUDA(cudaFuncSetAttribute(cbs::sliced_kernel<NBV, false>,                                         \
                                           cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.total));           \
            cbs::sliced_kernel<NBV, false><<<grid, threads, pl.total, st>>>(p);                                    \
        }                                                                                                          \
        break;
    switch (nb) {
        NABO_CBS_LAUNCH(1) NABO_CBS_LAUNCH(2) NABO_CBS_LAUNCH(3) NABO_CBS_LAUNCH(4)
        NABO_CBS_LAUNCH(5) NABO_CBS_LAUNCH(6) NABO_CBS_LAUNCH(7) NABO_CBS_LAUNCH(8)
        NABO_CBS_LAUNCH(9) NABO_CBS_LAUNCH(10) NABO_CBS_LAUNCH(11) NABO_CBS_LAUNCH(12)
        NABO_CBS_LAUNCH(13) NABO_CBS_LAUNCH(14) NABO_CBS_LAUNCH(15) NABO_CBS_LAUNCH(16)
        default: return nabo_set_error(NABO_EINVAL, "knn: sliced Canberra pass supports at most 128 dimensions");
    }
#undef NABO_CBS_LAUNCH
    NABO_LAUNCH_CHECK("cbs::sliced_kernel");
    return 0;
}
