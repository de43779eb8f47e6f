// Tensor-core candidate pass for Euclidean / cosine kNN (sm_100a: TMA bulk copies ->
// shared memory -> tcgen05.mma -> TMEM -> fused per-query top-K' filter).
//
//   score(q, r) = ||r~||^2 - 2 q~.r~        (ranking-equivalent to ||q~ - r~||^2)
// with q~ = qh + ql, r~ = rh + rl the two-term FP16 split of the (power-of-two scaled)
// coordinates, evaluated as ONE GEMM with the augmented K dimension
//   A row (query)     = [-2qh | -2qh | -2ql | 1  1  1  | 0..]
//   B row (reference) = [  rh |   rl |   rh | n1 n2 n3 | 0..]      n1+n2+n3 = ||r~||^2
// so the accumulator IS the score and the epilogue is pure selection.  Operands are
// pre-tiled in HBM in the UMMA K-major no-swizzle core-matrix layout (pack kernels below),
// so one tile is one contiguous span and a single cp.async.bulk brings it in.
//
// CTA = 512 threads, persistent over work items of NQ=3 query tiles (384 queries) x one range of
// reference tiles (the whole reference, or a piece of it when there are fewer items than SMs; with more items than SMs
// the items are dealt out on a line of modelled cost, and an item cut at a CTA boundary is swept as a head on one CTA
// and a tail that resumes the head's selection state on the next - see sched_bound):
//   warps 0-11  epilogue: warpgroup w owns query tile w; thread = one query row (TMEM lane)
//   warp 12  TMEM allocator, then TMA producer: A tiles once per item, B (reference) tiles through a ring
//   warp 13  MMA issuer: the three query tiles rotate over FOUR accumulators, so the MMAs of a warpgroup's
//            next tile run while it still reads the current one (warps 14-15 idle)
// Wide plan (53 <= g <= 128, where three query tiles and two whole reference tiles no longer fit in shared memory):
// NQ=2 query tiles (epilogue warps 0-7, each warpgroup double-buffered over the four accumulators) and the reference
// tile streamed through the ring in K-slabs of SLAB K steps - the packed layout is K-chunk-major, so a slab is one
// contiguous span (see plan_smem).
// The epilogue keeps, per query, a running threshold tau (register) and a private
// candidate buffer of CAP keys in L2-resident global memory; a tile chunk is first reduced
// with FMNMX3 and only chunks holding a score < tau take the append path.  When a buffer
// may overflow the warp compacts it (histogram cut in shared memory, select.cuh), keeps at least
// the K' best and tightens tau.  Everything rejected or dropped has score >= final tau, which is
// what the certificate in the re-rank needs.
#include "common.cuh"
#include "knn_internal.cuh"
#include "ptx.cuh"
#include "select.cuh"

#include <cuda_fp16.h>

namespace tc {

constexpr int TILE = 128;           // rows per operand tile (UMMA M and N)
constexpr int NTHREADS = 512;        // epilogue: warps 0 .. 4 NQ - 1 (TMEM lane quarter = warp % 4)
constexpr int MAX_G = 128;           // widest PCA space of the tensor-core pass (certificate constant checked up to here)
constexpr int PRODUCER_WARP = 12;    // highest warp ids on their schedulers: the arbiter favours them,
constexpr int MMA_WARP = 13;         // so the single-thread producer / issuer are never starved
constexpr int TMEM_WARP = 12;
// Candidate buffer entries per query: CAP_SMALL up to K' = MAX_KPRIME, CAP_LARGE above (see plan_k).  256-key buffers
// compact a quarter as often, but measured at 100 k x 100 k, k = 30 the candidate kernel went 3.78 -> 4.51 ms
// (staler thresholds, 2 KB per query in L2) and the final selection 0.17 -> 1.8 ms: they only pay for large K'
// (k = 60: 55 -> 7.4 ms), so they serve only the k the 128-key plan cannot take.
constexpr int CAP_SMALL = 128;
constexpr int CAP_LARGE = 256;
static_assert(CAP_SMALL == sel::CAP, "the fused re-rank (exact.cu) reads the candidate buffers with sel::CAP keys per query");
constexpr int CHUNK = 32;           // columns per tcgen05.ld
constexpr int MAX_KPRIME = 96;      // K' of the 128-key plan (K' lists go to the re-rank, up to 128 per query with splits)
constexpr int MAX_KPRIME_LARGE = 160;   // K' of the 256-key plan (unsplit: the re-rank takes up to 256 per query)
constexpr int MAX_KSEL = 128;       // k + drop_first of the 256-key plan (the exact engine's limit)
constexpr int SLEEP_NS = 2000;      // suspend-time hint of the producer's mbarrier waits
// accumulators in TMEM (128 columns each): the NQ query tiles share four buffers in a fixed rotation
// (job n = tile * NQ + q uses buffer n % 4), so the MMAs of a warpgroup's next tile run while it is still
// reading the current one
constexpr int NACC = 4;
constexpr int MAX_STAGES = 4;        // reference ring stages (b_full / b_empty of Barriers)
constexpr uint32_t KSTEP_BYTES = TILE * 16 * 2;   // one K step (16 columns) of a packed tile: two 16-byte K chunks

__host__ __device__ inline int kp_for(int g) { return (3 * g + 3 + 15) / 16 * 16; }
__host__ __device__ inline size_t tile_bytes(int kp) { return (size_t)TILE * kp * 2; }

// ------------------------------------------------------------------ schedule of the unsplit sweep
// Modelled cost of the first x reference tiles of a work item, in tiles of the warm sweep:
//   F(x) = x + COST_BETA * j0 * ln(1 + x / j0),   j0 = COST_J0 * K' tiles.
// The log term is the cold start of the running selection: a query appends about K' / i of its i-th reference, so the
// appends - and the compactions they trigger - of the first x tiles grow as K' ln(x / K').
// COST_BETA and COST_J0 are fitted to the epilogue cycles per warp-tile by sweep position (-DNABO_TC_STATS,
// tools/probe_tc_stats.py) at 100 k x 100 k, g = 50, k = 30 (K' = 39) on a B200: see DESIGN 4.1.
constexpr double COST_BETA = 16.2, COST_J0 = 1.0 / 20;
__host__ __device__ inline double sweep_cost(int x, int kprime) {
    const double j0 = COST_J0 * kprime;
    return x + COST_BETA * j0 * log1p(x / j0);
}

// McNaughton's wrap-around rule on the cost line: the n_items items lie end to end, CTA ticket c owns [c T, (c + 1) T)
// with T = n_items F(n_rtiles) / grid.  sched_bound(c) is where that segment starts: items < item and reference tiles
// [0, tile) of `item` belong to lower tickets (0 <= tile < n_rtiles; the cut is the first whole tile at or past the
// boundary's cost).  Ticket c therefore runs, in this order,
//   the HEAD of item i1 = tiles [0, x1)         (x1 > 0; (i1, x1) = sched_bound(c + 1))
//   the whole items [i0 or i0 + 1, i1)
//   the TAIL of item i0 = tiles [x0, n_rtiles)  (x0 > 0; (i0, x0) = sched_bound(c)), resuming the head ticket c - 1 left.
// A head is the first piece of its CTA and waits on nothing; a tail waits only on the next lower ticket.  In model cost
// a head ends no later than its tail starts: head + tail = one item < T, and a CTA without whole items runs the head of
// item i0 + 1 first, cut at a larger cost offset than its tail's (T > F(n_rtiles) when grid < n_items).  With
// grid = n_items every boundary falls on an item: one whole item per CTA.
__host__ __device__ inline void sched_bound(int b, int n_items, int n_rtiles, int grid, int kprime, int& item, int& tile) {
    const long long pos = (long long)b * n_items;           // boundary in units of items: pos / grid
    item = (int)(pos / grid);
    const int rem = (int)(pos - (long long)item * grid);
    tile = 0;
    if (rem == 0) return;
    const double o = sweep_cost(n_rtiles, kprime) * rem / grid;      // cost into `item`, 0 < o < F(n_rtiles)
    // smallest x with F(x) >= o: F(lo) < o <= F(hi)
    int lo = 0, hi = n_rtiles;
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (sweep_cost(mid, kprime) >= o) hi = mid; else lo = mid;
    }
    tile = hi;
    if (tile == n_rtiles) { ++item; tile = 0; }
}

// The tile plan of a PCA width g - the one place that decides it:
//   g <= 52       NQ = 3 query tiles, whole reference tiles per ring stage (2 - 4 stages)
//   53 <= g <= 128  NQ = 2 query tiles, reference slabs of 4 or 2 K steps (16 / 8 KB) per stage: the slab width with
//                 the most bytes in flight (at most MAX_STAGES stages, at least 2), the wider one on a tie.  Slabs of
//                 1 K step would never win up to g = 128 (g = 128 leaves 17.5 KB: 2 x 8 KB).
// stages = 0: no plan fits (g > 128).
struct SmemPlan {
    int nq;              // query tiles per work item
    int slab;            // K steps per reference slab, 0 = whole tiles
    int stages;
    size_t stage_bytes;
    size_t a_off, b_off, sort_off, bar_off, total;
};
inline SmemPlan plan_smem(int g) {
    const int kp = kp_for(g);
    const size_t bars = 512;
    const size_t budget = 227 * 1024 - 1024;   // keep 1 KB for alignment slack
    auto room = [&](int nq) {                  // what nq query tiles, their warps' histograms and the barriers leave
        const size_t used = nq * tile_bytes(kp) + (size_t)4 * nq * 256 * 4 + bars;
        return budget > used ? budget - used : (size_t)0;
    };
    SmemPlan p;
    p.nq = 3;
    p.slab = 0;
    p.stage_bytes = tile_bytes(kp);
    p.stages = (int)(room(3) / p.stage_bytes);
    if (p.stages > MAX_STAGES) p.stages = MAX_STAGES;
    if (p.stages < 2) {
        p.nq = 2;
        p.stages = 0;
        for (int slab = 4; slab >= 2 && g <= MAX_G; slab /= 2) {
            const size_t sb = (size_t)slab * KSTEP_BYTES;
            int st = (int)(room(2) / sb);
            if (st > MAX_STAGES) st = MAX_STAGES;
            if (st >= 2 && st * sb > p.stages * p.stage_bytes) { p.slab = slab; p.stages = st; p.stage_bytes = sb; }
        }
    }
    const size_t a = p.nq * tile_bytes(kp);
    p.a_off = 0;
    p.b_off = a;
    p.sort_off = a + (size_t)p.stages * p.stage_bytes;
    p.bar_off = p.sort_off + (size_t)4 * p.nq * 256 * 4;     // per-warp histogram
    p.total = p.bar_off + bars;
    return p;
}

// The candidate-buffer plan of ksel = k + drop_first - the one place that decides it.  K' = ksel + max(ksel / 4, 8)
// (the extra ranks are the certificate margin, see nabo_tc_kprime), capped by the plan:
//   ksel + 8 <= MAX_KPRIME   128-key buffers, K' <= 96 (every k the pass took before the 256-key plan existed)
//   89 <= ksel <= 128        256-key buffers, K' = 111 .. 160
// ksel > 128 has no plan; workspace sizing still gets the 256-key one (supported() decides what runs).
struct KPlan {
    int cap;
    int kprime;
};
inline int kprime_for(int ksel, int cap_kprime) {
    const int kprime = ksel + (ksel / 4 > 8 ? ksel / 4 : 8);
    return kprime < cap_kprime ? kprime : cap_kprime;
}
inline KPlan plan_k(int ksel) {
    KPlan kp;
    const bool small = ksel + 8 <= MAX_KPRIME;
    kp.cap = small ? CAP_SMALL : CAP_LARGE;
    kp.kprime = kprime_for(ksel, small ? MAX_KPRIME : MAX_KPRIME_LARGE);
    return kp;
}

// ------------------------------------------------------------------ operand packing
// norms2[row] = ||x||^2 (FP64, exact coordinates); maxn2 = max finite norm^2 (as float bits)
__global__ void __launch_bounds__(256)
norms_kernel(const double* __restrict__ x, int ld, int n, int g, double* __restrict__ norms2,
             unsigned int* __restrict__ maxn2_bits) {
    int row = blockIdx.x * blockDim.x + threadIdx.x;
    float mine = 0.f;
    if (row < n) {
        const double* p = x + (long long)row * ld;
        double s = 0.0;
        for (int k = 0; k < g; ++k) s = fma(p[k], p[k], s);
        norms2[row] = s;
        if (isfinite(s)) mine = __double2float_ru(s);
    }
    for (int o = 16; o > 0; o >>= 1) mine = fmaxf(mine, __shfl_xor_sync(0xffffffffu, mine, o));
    if ((threadIdx.x & 31) == 0 && mine > 0.f) atomicMax(maxn2_bits, __float_as_uint(mine));
}

// scal[0] = sc (power of two), scal[1] = 1/sc, scal[2] = max scaled reference norm, scal[3] = cosine flag
__global__ void scale_kernel(const unsigned int* __restrict__ maxq_bits, const unsigned int* __restrict__ maxr_bits,
                             int cosine, double* __restrict__ scal) {
    double sc = 1.0, rmax;
    if (cosine) {
        sc = 32.0;               // unit vectors
        rmax = 32.0 * (1.0 + 1e-6);
    } else {
        float mq = __uint_as_float(*maxq_bits), mr = __uint_as_float(*maxr_bits);
        double mx = sqrt((double)fmaxf(mq, mr));
        if (mx > 0.0 && isfinite(mx)) {
            int e;
            frexp(mx, &e);        // mx = f * 2^e, f in [0.5, 1)  ->  mx * 2^(6-e) in [32, 64)
            sc = ldexp(1.0, 6 - e);
        }
        rmax = sqrt((double)__uint_as_float(*maxr_bits)) * sc * (1.0 + 1e-6);
    }
    scal[0] = sc;
    scal[1] = 1.0 / sc;
    scal[2] = rmax;
    scal[3] = cosine ? 1.0 : 0.0;
}

// PACK_SPLIT threads per row (thread c takes the 16-byte chunks kc = c, c + PACK_SPLIT, ...); chunk kc of row r of
// tile t lands at
//   t * TILE*kp*2 + kc * (TILE*16) + (r>>3)*128 + (r&7)*16
// (core matrices of 8 rows x 16 B, K-chunk-major: SBO = 128 B, LBO = TILE*16 B).  The chunks that hold the norm
// columns 3g .. 3g+2 of a reference row need the whole ||r~||^2: they are written after the partial sums of the
// row's threads have met in shared memory (fixed order: deterministic).
constexpr int PACK_SPLIT = 4;
template <bool IS_QUERY>
__global__ void __launch_bounds__(TILE * PACK_SPLIT)
pack_kernel(const double* __restrict__ x, int ld, int n, int g, int kp, const double* __restrict__ norms2,
            const double* __restrict__ scal, const uint8_t* __restrict__ mask, __half* __restrict__ out,
            double* __restrict__ qn2_out) {
    __shared__ double part[PACK_SPLIT][TILE];
    const int r = threadIdx.x & (TILE - 1);
    const int c = threadIdx.x / TILE;                 // warp-uniform
    const long long row = (long long)blockIdx.x * TILE + r;
    __half* tile = out + (size_t)blockIdx.x * TILE * kp;
    const bool live = row < n;
    const double sc = scal[0];
    const bool cosine = scal[3] != 0.0;
    double mul = sc;
    bool dead = false;          // reference that can never be a neighbour (masked / zero norm under cosine)
    if (live && cosine) {
        double nn = sqrt(norms2[row]);
        if (nn > 0.0 && isfinite(nn)) mul = sc / nn; else { mul = 0.0; dead = true; }
    }
    if (live && !IS_QUERY && mask && mask[row]) dead = true;
    if (!live && !IS_QUERY) dead = true;        // padding rows of the last reference tile: score 60000, like a masked
                                                // cell, so the epilogue needs no column-limit test
    const double* p = x + (live ? row : 0) * (long long)ld;
    const int nchunks = kp / 8;
    // chunk kc of this row; n2 (in/out): ||x~||^2 of the split value actually fed to the tensor core (scaled units),
    // summed over the segment-0 columns of the chunk; n2_row: the whole row's sum, for the norm columns
    auto chunk = [&](int kc, double& n2, double n2_row) {
        __align__(16) __half h[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const int col = kc * 8 + e;
            __half v = __float2half(0.f);
            if (live && col < 3 * g) {
                const int seg = col / g, k = col - seg * g;
                const double xv = p[k] * mul;
                const __half hi = __double2half(xv);
                const __half lo = __double2half(xv - (double)__half2float(hi));
                if (seg == 0) { const double t = (double)__half2float(hi) + (double)__half2float(lo); n2 = fma(t, t, n2); }
                if (IS_QUERY) {
                    const __half src = seg == 2 ? lo : hi;
                    v = __float2half(-2.0f * __half2float(src));      // exact: power-of-two scaling
                    if (__hisinf(v)) {
                        // a query far outside the scale of a prepared reference (|x~| >= 32 760): its operand would
                        // overflow FP16.  The row is fed zeros and its |q~|^2 becomes NaN, which fails the certificate
                        // and sends it to the exact fallback.  (With the joint scale of the one-shot path |x~| < 64.)
                        v = __float2half(0.f);
                        n2 = CUDART_NAN;
                    }
                } else {
                    v = seg == 1 ? lo : hi;
                }
            } else if (live && col < 3 * g + 3) {
                if (IS_QUERY) v = __float2half(1.0f);
            }
            h[e] = v;
        }
        if (!IS_QUERY && (live || dead) && 3 * g + 3 > kc * 8 && 3 * g < kc * 8 + 8) {
            // norm pieces n1 + n2 + n3 = ||r~||^2
            double rem = dead ? 60000.0 : n2_row;
            for (int t = 0; t < 3; ++t) {
                const int col = 3 * g + t;
                const __half piece = __double2half(rem);
                rem -= (double)__half2float(piece);
                if (dead && t > 0) { if (col >= kc * 8 && col < kc * 8 + 8) h[col - kc * 8] = __float2half(0.f); continue; }
                if (col >= kc * 8 && col < kc * 8 + 8) h[col - kc * 8] = piece;
            }
        }
        *reinterpret_cast<uint4*>(reinterpret_cast<char*>(tile) + (size_t)kc * (TILE * 16) + (r >> 3) * 128 + (r & 7) * 16) =
            *reinterpret_cast<const uint4*>(h);
    };
    const int norm_lo = (3 * g) / 8, norm_hi = (3 * g + 2) / 8;        // chunks that hold the norm columns
    double n2 = 0.0;
    for (int kc = c; kc < nchunks; kc += PACK_SPLIT) {
        if (!IS_QUERY && kc >= norm_lo && kc <= norm_hi) continue;
        chunk(kc, n2, 0.0);
    }
    if (!IS_QUERY) {
        // segment-0 columns inside the deferred chunks (only when 3g < 8, i.e. g <= 2) still belong to the sum
        for (int kc = norm_lo + c; kc <= norm_hi && kc < nchunks; kc += PACK_SPLIT)
            for (int e = 0; e < 8; ++e) {
                const int col = kc * 8 + e;
                if (live && col < g) {
                    const double xv = p[col] * mul;
                    const __half hi = __double2half(xv);
                    const __half lo = __double2half(xv - (double)__half2float(hi));
                    const double t = (double)__half2float(hi) + (double)__half2float(lo);
                    n2 = fma(t, t, n2);
                }
            }
    }
    part[c][r] = n2;
    __syncthreads();
    double n2_row = part[0][r];
#pragma unroll
    for (int i = 1; i < PACK_SPLIT; ++i) n2_row += part[i][r];
    if (!IS_QUERY) {
        for (int kc = norm_lo + c; kc <= norm_hi && kc < nchunks; kc += PACK_SPLIT) {
            double unused = 0.0;
            chunk(kc, unused, n2_row);
        }
    }
    if (IS_QUERY && c == 0 && live && qn2_out) qn2_out[row] = n2_row;
}

// ------------------------------------------------------------------ the candidate kernel
struct Params {
    const __half* qa;       // packed queries  [n_qtiles_padded][TILE*kp]
    const __half* rb;       // packed references [n_rtiles][TILE*kp]
    int n_query, n_ref, kp, n_items, n_rtiles, stages, kprime, kc_out, soft;
    int n_split;            // reference ranges per query item (work item = n_items x n_split, see nabo_tc_split)
    int cut;                // n_split = 1: 1 = the cost-line schedule of sched_bound, 0 = items c, c + grid, ... per CTA c
    int signal_round;       // > 0 = every CTA signals the dependent launch after its signal_round-th item (0 = never;
                            // only without cuts and with n_split = 1)
    unsigned int* ticket;   // n_split = 1: CTA ticket counter, then one flag per item: its head is in global memory
                            // (zeroed before every launch)
    unsigned long long* cand_buf;   // [work item][NQ*TILE][CAP]: every (query, reference range) owns CAP keys (plan_k)
    int* cand_cnt;          // [work item][NQ*TILE] live keys of each buffer when its sweep ended
    float* cand_tau;        // [work item][NQ*TILE] running threshold when its sweep ended
    int32_t* cand_idx;      // [n_query][n_split][kc_out]      (written by emit_kernel)
    float* cert_tau;        // [n_split][n_query]              (written by emit_kernel)
    size_t a_off, b_off, sort_off, bar_off;
};

struct Barriers {
    uint64_t a_full, a_empty;
    uint64_t b_full[MAX_STAGES], b_empty[MAX_STAGES];
    uint64_t acc_full[NACC], acc_empty[NACC];
    uint32_t tmem_base;
    int ticket;             // n_split = 1: this CTA's ticket c
    int sched[4];           // n_split = 1: sched_bound of c and of c + 1 (i0, x0, i1, x1)
};

using namespace sel;   // make_key, compact_sort_inline, compact_select (select.cuh)

#ifdef NABO_TC_STATS       // development counters (tools/probe_tc_stats.py): [0] warp chunks, [1] warp chunks with a hit,
                           // [2] lanes with a hit, [3] keys appended, [4] running compactions, cycles per warp:
                           // [5] compaction, [6] filter_chunk, [7] wait for the accumulator, [8] tcgen05.ld + wait,
                           // [9] final emit, [10] whole item loop; [TC_HIST + b] epilogue cycles of the warp-tiles at
                           // sweep position 2^b - 1 <= j < 2^(b+1) - 1 of an item, [TC_HIST + 32 + b] their count;
                           // [TC_TIME + 2 c], [TC_TIME + 2 c + 1] %globaltimer at the start and end of CTA (ticket) c
constexpr int TC_HIST = 12, TC_TIME = TC_HIST + 64, TC_NSTATS = TC_TIME + 2 * 1024;
__device__ unsigned long long g_tc_stats[TC_NSTATS];
__device__ __forceinline__ unsigned long long globaltimer() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
// accumulated in per-thread registers (tc_loc), flushed with one atomic per counter at the end of an item
#define TC_STAT(i, v) (tc_loc[i] += (unsigned long long)(v))
#define TC_CLK(var) const long long var = clock64()
#define TC_CLK_ADD(i, t0) (tc_loc[i] += (unsigned long long)(clock64() - (t0)))
#define TC_DECL unsigned long long tc_loc[12] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0}
#define TC_FLUSH do { if ((threadIdx.x & 31) == 0) for (int i_ = 0; i_ < 12; ++i_) { if (tc_loc[i_]) atomicAdd(&g_tc_stats[i_], tc_loc[i_]); tc_loc[i_] = 0; } } while (0)
#define TC_ARG , unsigned long long (&tc_loc)[12]
#define TC_PASS , tc_loc
#else
#define TC_STAT(i, v)
#define TC_CLK(var)
#define TC_CLK_ADD(i, t0)
#define TC_DECL
#define TC_FLUSH
#define TC_ARG
#define TC_PASS
#endif

// 32 freshly loaded scores of one query: reduce with FMNMX3 and append the ones below tau
template <int CAP>
__device__ __forceinline__ void filter_chunk(const uint32_t (&vr)[32], uint32_t col0, float tau,
                                             unsigned long long* mybuf, int& cnt TC_ARG) {
    float v[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(vr[i]);
    float g4[4];
#pragma unroll
    for (int gi = 0; gi < 4; ++gi) {
        const float a = ptx::min3(v[8 * gi], v[8 * gi + 1], v[8 * gi + 2]);
        const float b = ptx::min3(v[8 * gi + 3], v[8 * gi + 4], v[8 * gi + 5]);
        g4[gi] = ptx::min3(a, b, fminf(v[8 * gi + 6], v[8 * gi + 7]));
    }
    const float m = fminf(fminf(g4[0], g4[1]), fminf(g4[2], g4[3]));
#ifdef NABO_TC_STATS
    {
        const unsigned hb = __ballot_sync(0xffffffffu, m < tau);
        if ((threadIdx.x & 31) == 0) { TC_STAT(0, 1); if (hb) { TC_STAT(1, 1); TC_STAT(2, __popc(hb)); } }
        int na = 0;
        for (int i = 0; i < 32; ++i) na += v[i] < tau;
        for (int o = 16; o > 0; o >>= 1) na += __shfl_xor_sync(0xffffffffu, na, o);
        if ((threadIdx.x & 31) == 0) TC_STAT(3, na);
    }
#endif
    if (m < tau) {
#pragma unroll
        for (int gi = 0; gi < 4; ++gi) {
            if (g4[gi] < tau) {
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    if (v[8 * gi + i] < tau) {
                        NABO_DEV_ASSERT(cnt >= 0 && cnt < CAP);
                        mybuf[cnt] = make_key(v[8 * gi + i], col0 + 8 * gi + i);
                        ++cnt;
                    }
                }
            }
        }
    }
}

// Work enumeration (the r-th piece of this CTA; false when there is none).  SPLIT: the reference range of every query
// item is cut into n_split equal pieces, each a work item with its own buffer `slot`, K' list and threshold; the re-rank
// takes the union of the lists and the smallest threshold; CTA c takes the slots c, c + grid, c + 2 grid, ...
// SPLIT is a template parameter: one general form for both measured 3.59 -> 3.72 ms in the unsplit kernel at
// 100 k x 100 k, k = 30 (B200, 1 000 W power limit).
// SPLIT = false: CTA ticket c runs the pieces of sched_bound (head, whole items, tail; sched = {i0, x0, i1, x1}), or,
// without cuts (sched[0] = -1 - c), the whole items c, c + grid, c + 2 grid, ...
template <bool SPLIT>
__device__ __forceinline__ bool work_piece(const Params& p, const int (&sched)[4], int r, int& slot, int& qitem, int& j0,
                                           int& j1) {
    if (!SPLIT) {
        const int i0 = sched[0], x0 = sched[1], i1 = sched[2], x1 = sched[3];
        if (i0 < 0) {
            slot = qitem = -1 - i0 + r * (int)gridDim.x;
            j0 = 0; j1 = p.n_rtiles;
            return slot < p.n_items;
        }
        if (x1 > 0 && r-- == 0) {                          // head
            slot = qitem = i1; j0 = 0; j1 = x1;
            return true;
        }
        const int first = x0 > 0 ? i0 + 1 : i0;
        j1 = p.n_rtiles;
        if (r < i1 - first) {                              // whole items
            slot = qitem = first + r; j0 = 0;
            return true;
        }
        if (x0 > 0 && r == i1 - first) {                   // tail
            slot = qitem = i0; j0 = x0;
            return true;
        }
        return false;
    }
    slot = (int)blockIdx.x + r * (int)gridDim.x;
    if (slot >= p.n_items * p.n_split) return false;
    qitem = slot / p.n_split;
    const int seg = slot - qitem * p.n_split;
    j0 = (int)((long long)p.n_rtiles * seg / p.n_split);
    j1 = (int)((long long)p.n_rtiles * (seg + 1) / p.n_split);
    return true;
}

// KSTEPS: K steps of 16 known at compile time (0 = runtime loop); SPLIT: see work_piece; NQ: query tiles per work item;
// SLAB: K steps per reference slab (0 = whole reference tiles).  The tile plan (plan_smem) picks NQ and SLAB.
// CAP: keys per candidate buffer (plan_k); the 256-key plan only runs unsplit.
template <int KSTEPS, bool SPLIT, int NQ = 3, int SLAB = 0, int CAP = CAP_SMALL>
__global__ void __launch_bounds__(NTHREADS, 1) candidates_kernel(const Params p) {
    static_assert(NQ * 4 <= PRODUCER_WARP && (SLAB == 0 || KSTEPS == 0), "tile plan");
    static_assert(CAP == CAP_SMALL || (CAP == CAP_LARGE && !SPLIT), "buffer plan");
    constexpr int N_EPI_WARPS = 4 * NQ;
    extern __shared__ __align__(1024) uint8_t smem[];
    Barriers* bars = reinterpret_cast<Barriers*>(smem + p.bar_off);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int ksteps = p.kp / 16;
    const uint32_t a_tile_bytes = (uint32_t)tile_bytes(p.kp);
    const int nslab = SLAB ? (ksteps + SLAB - 1) / SLAB : 1;       // ring stages per reference tile
    const uint32_t stage_bytes = SLAB ? SLAB * KSTEP_BYTES : a_tile_bytes;

    if (threadIdx.x == 0) {
        ptx::mbar_init(&bars->a_full, 1);
        ptx::mbar_init(&bars->a_empty, 1);
        for (int s = 0; s < MAX_STAGES; ++s) { ptx::mbar_init(&bars->b_full[s], 1); ptx::mbar_init(&bars->b_empty[s], 1); }
        for (int q = 0; q < NACC; ++q) { ptx::mbar_init(&bars->acc_full[q], 1); ptx::mbar_init(&bars->acc_empty[q], 4); }
        ptx::fence_barrier_init();
        if (!SPLIT) {
            // the ticket, not blockIdx.x, orders the CTAs: a lower ticket belongs to a CTA that has already started, so
            // a tail's wait for its head (ticket c - 1) ends even when only some CTAs of the grid are resident
            const int c = (int)atomicAdd(p.ticket, 1u);
            bars->ticket = c;
            if (p.cut) {
                sched_bound(c, p.n_items, p.n_rtiles, (int)gridDim.x, p.kprime, bars->sched[0], bars->sched[1]);
                sched_bound(c + 1, p.n_items, p.n_rtiles, (int)gridDim.x, p.kprime, bars->sched[2], bars->sched[3]);
            } else {
                bars->sched[0] = -1 - c;             // items c, c + grid, c + 2 grid, ... (see work_piece)
                bars->sched[1] = bars->sched[2] = bars->sched[3] = 0;
            }
#ifdef NABO_TC_STATS
            if (c < 1024) g_tc_stats[TC_TIME + 2 * c] = globaltimer();
#endif
        }
    }
    if (warp == TMEM_WARP) ptx::tmem_alloc(&bars->tmem_base, 512);
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem_base = bars->tmem_base;
    const int sched[4] = {bars->sched[0], bars->sched[1], bars->sched[2], bars->sched[3]};

    if (warp == PRODUCER_WARP) {
        // ===================== TMA producer =====================
        if (lane == 0) {
            uint32_t t = 0, it = 0;
            for (int wr = 0;; ++wr, ++it) {
                int w, item, j0, j1;
                if (!work_piece<SPLIT>(p, sched, wr, w, item, j0, j1)) break;
                ptx::mbar_wait_hint(&bars->a_empty, (it & 1) ^ 1, SLEEP_NS);
                ptx::mbar_arrive_expect_tx(&bars->a_full, NQ * a_tile_bytes);
                for (int q = 0; q < NQ; ++q) {
                    const char* src = reinterpret_cast<const char*>(p.qa) + (size_t)(item * NQ + q) * a_tile_bytes;
                    char* dst = reinterpret_cast<char*>(smem + p.a_off) + (size_t)q * a_tile_bytes;
                    for (uint32_t o = 0; o < a_tile_bytes; o += 8192)
                        ptx::bulk_g2s(dst + o, src + o, min(8192u, a_tile_bytes - o), &bars->a_full);
                }
                for (int j = j0; j < j1; ++j)
                    for (int sl = 0; sl < nslab; ++sl, ++t) {
                        // slab sl: K chunks [2 SLAB sl, 2 SLAB (sl + 1)) of tile j, one contiguous span (the last may be shorter)
                        const uint32_t s = t % p.stages, use = t / p.stages;
                        const uint32_t off = sl * stage_bytes, bytes = min(stage_bytes, a_tile_bytes - off);
                        ptx::mbar_wait_hint(&bars->b_empty[s], (use & 1) ^ 1, SLEEP_NS);   // far ahead of the consumers
                        ptx::mbar_arrive_expect_tx(&bars->b_full[s], bytes);
                        const char* src = reinterpret_cast<const char*>(p.rb) + (size_t)j * a_tile_bytes + off;
                        char* dst = reinterpret_cast<char*>(smem + p.b_off) + (size_t)s * stage_bytes;
                        for (uint32_t o = 0; o < bytes; o += 8192)
                            ptx::bulk_g2s(dst + o, src + o, min(8192u, bytes - o), &bars->b_full[s]);
                    }
            }
        }
    } else if (warp == MMA_WARP) {
        // ===================== MMA issuer: one warp, jobs in a fixed rotation =====================
        // Job n = (reference tile, query tile q = n % NQ) accumulates into buffer n % 4.  With one buffer more
        // than there are warpgroups, the MMAs of job n start as soon as the warpgroup of job n - 4 (the
        // PREVIOUS query tile, one reference tile back) has read its accumulator - about a third of a period
        // before warpgroup q finishes its current tile - so they complete while q is still filtering.  With NQ = 2
        // job n - 4 is the SAME query tile two reference tiles back: each warpgroup has a full double buffer.
        // The whole warp runs the loop (descriptor arithmetic in the uniform datapath); only the elected
        // lane issues tcgen05.mma / commit.
        {
            const uint32_t idesc = ptx::make_idesc_f16(TILE, TILE);
            const uint32_t lbo = TILE * 16, sbo = 128;
            const uint64_t ad0 = ptx::make_smem_desc(ptx::smem_u32(smem + p.a_off), lbo, sbo);
            const uint64_t bd0 = ptx::make_smem_desc(ptx::smem_u32(smem + p.b_off), lbo, sbo);
            uint32_t t = 0, it = 0, n = 0;
            for (int wr = 0;; ++wr, ++it) {
                int w, item, j0, j1;
                if (!work_piece<SPLIT>(p, sched, wr, w, item, j0, j1)) break;
                ptx::mbar_wait(&bars->a_full, it & 1);
                for (int j = j0; j < j1; ++j, n += NQ, ++t)
                    for (int sl = 0; sl < nslab; ++sl) {
                        // slab sl of reference tile j against every query tile; with slabs the NQ accumulators of tile j
                        // are all open until its last slab
                        const uint32_t u = t * nslab + sl, s = u % p.stages, use = u / p.stages;
                        ptx::mbar_wait(&bars->b_full[s], use & 1);
                        // descriptors differ only in the start-address field (16-byte units): one K step = 2 * LBO
                        const uint64_t bd1 = bd0 + (uint64_t)((s * stage_bytes) >> 4);
                        const int k0 = sl * SLAB;
#pragma unroll
                        for (int q = 0; q < NQ; ++q) {
                            const uint32_t job = n + q, buf = job & 3;
                            if (sl == 0) {
                                ptx::mbar_wait(&bars->acc_empty[buf], ((job >> 2) & 1) ^ 1);
                                ptx::tc_fence_after();
                            }
                            const uint32_t d_tmem = tmem_base + buf * TILE;
                            const uint64_t ad1 = ad0 + (uint64_t)((q * a_tile_bytes + k0 * KSTEP_BYTES) >> 4);
                            if (ptx::elect_one()) {
                                if (SLAB > 0) {
#pragma unroll
                                    for (int ks = 0; ks < SLAB; ++ks)
                                        if (k0 + ks < ksteps)
                                            ptx::mma_f16_ss(d_tmem, ad1 + ks * ((2 * lbo) >> 4), bd1 + ks * ((2 * lbo) >> 4),
                                                            idesc, k0 + ks > 0 ? 1u : 0u);
                                } else if (KSTEPS > 0) {
#pragma unroll
                                    for (int ks = 0; ks < KSTEPS; ++ks)
                                        ptx::mma_f16_ss(d_tmem, ad1 + ks * ((2 * lbo) >> 4), bd1 + ks * ((2 * lbo) >> 4), idesc,
                                                        ks > 0 ? 1u : 0u);
                                } else {
                                    for (int ks = 0; ks < ksteps; ++ks)
                                        ptx::mma_f16_ss(d_tmem, ad1 + ks * ((2 * lbo) >> 4), bd1 + ks * ((2 * lbo) >> 4), idesc,
                                                        ks > 0 ? 1u : 0u);
                                }
                                if (sl == nslab - 1) ptx::mma_commit(&bars->acc_full[buf]);
                                if (q == NQ - 1) {
                                    ptx::mma_commit(&bars->b_empty[s]);
                                    if (j == j1 - 1 && sl == nslab - 1) ptx::mma_commit(&bars->a_empty);
                                }
                            }
                            __syncwarp();
                        }
                    }
            }
        }
    } else if (warp < N_EPI_WARPS) {
        // ===================== epilogue: fused top-K' selection =====================
        const int q = warp >> 2;                           // query tile of this warpgroup
        const int quarter = warp & 3;                      // TMEM lane quarter this warp may read
        const int row = quarter * 32 + lane;
        const int slot = q * TILE + row;                   // this thread's query inside a work item
        const uint32_t tlane0 = tmem_base + ((uint32_t)(quarter * 32) << 16);
        uint32_t t = 0;
        uint32_t* hist = reinterpret_cast<uint32_t*>(smem + p.sort_off) + (size_t)warp * 256;
        TC_DECL;
        for (int wr = 0;; ++wr) {
            int w, item, j0, j1;
            if (!work_piece<SPLIT>(p, sched, wr, w, item, j0, j1)) break;
            unsigned long long* mybuf = p.cand_buf + ((size_t)w * NQ * TILE + slot) * CAP;
            float tau = CUDART_INF_F;
            int cnt = 0;
            if (!SPLIT && j0 > 0) {
                // tail: resume the selection state (buffer, count, tau) the head left in global memory.  One thread
                // waits for the head's flag (acquire), the epilogue warps meet on the named barrier, then read.
                if (threadIdx.x == 0) {
                    unsigned int ns = 32, done;
#ifdef NABO_CHECK
                    unsigned int spins = 0;
#endif
                    while (true) {
                        asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(done) : "l"(p.ticket + 1 + item) : "memory");
                        if (done) break;
                        __nanosleep(ns);
                        if (ns < 1024) ns *= 2;
                        NABO_DEV_ASSERT(++spins < (1u << 24));      // ~17 s: a schedule bug, not a slow head
                    }
                }
                asm volatile("bar.sync 1, %0;" ::"n"(N_EPI_WARPS * 32) : "memory");
                cnt = __ldcg(p.cand_cnt + (size_t)w * NQ * TILE + slot);
                tau = __ldcg(p.cand_tau + (size_t)w * NQ * TILE + slot);
            }
            TC_CLK(t_item);
#ifdef NABO_TC_STATS
            int hb = -1;                       // log2 bucket of the sweep position, its cycles and warp-tiles so far
            unsigned long long hcyc = 0, hcnt = 0;
#endif
            for (int j = j0; j < j1; ++j, ++t) {
#ifdef NABO_TC_STATS
                const long long t_tile = clock64();
                const int pos = SPLIT ? j - j0 : j;          // tiles since this selection state started cold
                const int b = 31 - __clz(pos + 1);
                if (b != hb) {
                    if (lane == 0 && hcnt) { atomicAdd(&g_tc_stats[TC_HIST + hb], hcyc); atomicAdd(&g_tc_stats[TC_HIST + 32 + hb], hcnt); }
                    hb = b; hcyc = 0; hcnt = 0;
                }
#endif
                const uint32_t job = t * NQ + q, buf = job & 3, acc_par = (job >> 2) & 1;
                const uint32_t taddr0 = tlane0 + buf * TILE;
                TC_CLK(t_w);
                ptx::mbar_wait(&bars->acc_full[buf], acc_par);
                ptx::tc_fence_after();
                TC_CLK_ADD(7, t_w);
                NABO_DEV_ASSERT(j >= 0 && j < p.n_rtiles);
                // the compaction of every lane whose buffer passed `lim` (soft limit once per tile, after the
                // accumulator has been handed back; hard limit otherwise: the next chunk may append 32 more)
                auto compact_over = [&](int lim) {
                    unsigned need = __ballot_sync(0xffffffffu, cnt > lim);
                    TC_CLK(t_c);
                    while (need) {
                        const int src = __ffs(need) - 1;
                        need &= need - 1;
                        unsigned long long* gb = reinterpret_cast<unsigned long long*>(
                            __shfl_sync(0xffffffffu, (unsigned long long)mybuf, src));
                        const int n = __shfl_sync(0xffffffffu, cnt, src);
                        int nc;
                        float nt;
                        compact_select<CAP / 32>(gb, n, lane, p.kprime, p.soft - 8, hist, nc, nt);
                        if (lane == src) { cnt = nc; tau = nt; }
                        if (lane == 0) TC_STAT(4, 1);
                    }
                    TC_CLK_ADD(5, t_c);
                };
#pragma unroll 1
                for (int c = 0; c < TILE / CHUNK; ++c) {
                    uint32_t vr[32];
                    TC_CLK(t_l);
                    ptx::tmem_ld_32x32(taddr0 + c * CHUNK, vr);
                    ptx::tmem_ld_wait();
                    TC_CLK_ADD(8, t_l);
                    if (c == TILE / CHUNK - 1) {        // accumulator fully read: hand it back to the MMA warp
                        ptx::tc_fence_before();
                        __syncwarp();
                        if (lane == 0) ptx::mbar_arrive(&bars->acc_empty[buf]);
                    }
                    TC_CLK(t_f);
                    filter_chunk<CAP>(vr, (uint32_t)(j * TILE + c * CHUNK), tau, mybuf, cnt TC_PASS);
                    TC_CLK_ADD(6, t_f);
                    compact_over(c == TILE / CHUNK - 1 ? p.soft : CAP - CHUNK);
                }
#ifdef NABO_TC_STATS
                hcyc += (unsigned long long)(clock64() - t_tile);
                ++hcnt;
#endif
            }
#ifdef NABO_TC_STATS
            if (lane == 0 && hcnt) { atomicAdd(&g_tc_stats[TC_HIST + hb], hcyc); atomicAdd(&g_tc_stats[TC_HIST + 32 + hb], hcnt); }
#endif
            // item done: leave the buffer as it is; emit_kernel makes the final selection of every (query, range)
            // at full occupancy instead of 32 serial sorts per warp here, with the tensor pipe idle meanwhile
            TC_CLK(t_e);
            p.cand_cnt[(size_t)w * NQ * TILE + slot] = cnt;
            p.cand_tau[(size_t)w * NQ * TILE + slot] = tau;
            TC_CLK_ADD(9, t_e);
            TC_CLK_ADD(10, t_item);
            TC_FLUSH;
            if (!SPLIT && p.signal_round == wr + 1) {
                // the full waves are done on this CTA: its buffers, counts and thresholds are in global memory
                // (fence), the epilogue warps meet on a named barrier, one thread lets the dependent grid - the
                // re-rank of those queries - start while the last, partly filled wave is still running
                __threadfence();
                asm volatile("bar.sync 1, %0;" ::"n"(N_EPI_WARPS * 32) : "memory");
                if (threadIdx.x == 0) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
            }
            if (!SPLIT && j1 < p.n_rtiles) {
                // head: its buffers, counts and thresholds are in global memory (fence), the epilogue warps meet on
                // the named barrier, one thread publishes the item's flag for the tail on the next ticket
                __threadfence();
                asm volatile("bar.sync 1, %0;" ::"n"(N_EPI_WARPS * 32) : "memory");
                if (threadIdx.x == 0)
                    asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p.ticket + 1 + item), "r"(1u) : "memory");
            }
        }
    }
    ptx::tc_fence_before();
    __syncthreads();
#ifdef NABO_TC_STATS
    if (!SPLIT && threadIdx.x == 0 && bars->ticket < 1024) g_tc_stats[TC_TIME + 2 * bars->ticket + 1] = globaltimer();
#endif
    if (warp == TMEM_WARP) ptx::tmem_dealloc(tmem_base, 512);
}

// Final selection: one warp per (query, reference range).  Sorts the buffer the sweep left behind, emits the K'
// best reference rows and the threshold every other reference of the range is at or above.
template <int NQ, int CAP = CAP_SMALL>
__global__ void __launch_bounds__(256)
emit_kernel(const Params p) {
    constexpr int KPL = CAP / 32;
    const int lane = threadIdx.x & 31;
    const long long wq = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);          // (buffer slot, query of the item)
    if (wq >= (long long)p.n_items * p.n_split * NQ * TILE) return;
    const int w = (int)(wq / (NQ * TILE)), slot = (int)(wq - (long long)w * NQ * TILE);
    const int item = w / p.n_split, seg = w - item * p.n_split;
    const long long qg = (long long)item * NQ * TILE + slot;                       // query row
    if (qg >= p.n_query) return;
    const int n = p.cand_cnt[wq];
    const float old_tau = p.cand_tau[wq];
    NABO_DEV_ASSERT(n >= 0 && n <= CAP);
    uint32_t ks[KPL], kpl[KPL];
    int nc;
    float nt;
    compact_sort_inline(p.cand_buf + (size_t)wq * CAP, n, lane, p.kprime, ks, kpl, nc, nt);
#pragma unroll
    for (int u = 0; u < KPL; ++u) {               // kc_out <= K' <= CAP
        const int i = u * 32 + lane;
        if (i < p.kc_out) {
            int32_t id = -1;
            if (i < nc && kpl[u] < (uint32_t)p.n_ref) id = (int32_t)kpl[u];
            p.cand_idx[(qg * p.n_split + seg) * p.kc_out + i] = id;
        }
    }
    if (lane == 0) p.cert_tau[(long long)seg * p.n_query + qg] = n >= p.kprime ? nt : old_tau;
}

}  // namespace tc

// ------------------------------------------------------------------ host side
static bool tc_plan_fits(int g) { return g >= 1 && g <= tc::MAX_G && tc::plan_smem(g).stages >= 2; }

bool nabo_tc_supported(int g, int k, int drop_first) {
    const int ksel = k + (drop_first ? 1 : 0);
    return tc_plan_fits(g) && ksel <= tc::MAX_KSEL;
}

int nabo_tc_kprime(int k, int drop_first) {
    // Extra ranks = certificate margin.  A row fails when ranks ksel..K' lie closer together than the
    // (provable, 2^-16) score error bound; measured at 100k x 100k / 200k x 1.25M, k = 30: +4 ranks ->
    // 76 / 944 uncertified rows, +6 -> 0 / 12, +8 -> 0 / 0, while the kernel time barely moves.
    return tc::plan_k(k + (drop_first ? 1 : 0)).kprime;
}

static int tc_grid(int n_items) {
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    return n_items < sms ? n_items : sms;
}

static size_t l2_bytes() {
    int dev = 0, l2 = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&l2, cudaDevAttrL2CacheSize, dev);
    return (size_t)l2;
}

// With fewer query items than SMs the reference range of every item is cut into up to NABO_TC_MAX_SPLIT
// pieces, each a work item of its own with its own K' candidates and threshold: a 20 000-query call keeps
// 106 SMs busy instead of 53.  The re-rank sees the union of the candidate lists and the smallest threshold
// (everything a piece rejected scored >= that piece's threshold >= the minimum), so nothing else changes.
int nabo_tc_split(int n_query, int n_ref, int g) {
    const int nq = tc::plan_smem(g).nq;
    const int n_items = (n_query + nq * tc::TILE - 1) / (nq * tc::TILE);
    const int n_rtiles = (n_ref + tc::TILE - 1) / tc::TILE;
    int s = n_items > 0 ? tc_grid(1 << 30) / n_items : 1;
    if (s > NABO_TC_MAX_SPLIT) s = NABO_TC_MAX_SPLIT;
    while (s > 1 && n_rtiles / s < 32) --s;              // keep >= 4096 references per piece
    return s < 1 ? 1 : s;
}

__global__ void tau_min_kernel(float* __restrict__ tau, int n_query, int n_split) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_query) return;
    float t = tau[i];
    for (int s = 1; s < n_split; ++s) t = fminf(t, tau[(size_t)s * n_query + i]);
    tau[i] = t;
}

int nabo_tau_min_launch(float* tau, int n_query, int n_split, cudaStream_t st) {
    tau_min_kernel<<<(n_query + 255) / 256, 256, 0, st>>>(tau, n_query, n_split);
    NABO_LAUNCH_CHECK("tau_min_kernel");
    return 0;
}

size_t nabo_tc_workspace_bytes(int n_query, int n_ref, int g, int k, int drop_first, bool with_ref) {
    const int kp = tc::kp_for(g);
    const size_t tb = tc::tile_bytes(kp);
    const int nq = tc::plan_smem(g).nq;
    const int n_items = (n_query + nq * tc::TILE - 1) / (nq * tc::TILE);
    const tc::KPlan kpl = tc::plan_k(k + (drop_first ? 1 : 0));
    const int kprime = kpl.kprime;
    const int max_split = kpl.cap == tc::CAP_SMALL ? NABO_TC_MAX_SPLIT : 1;
    size_t b = 0;
    b += nabo_align_up((size_t)n_items * nq * tb, 256);          // packed queries
    if (with_ref) b += nabo_tc_ref_bytes(n_ref, g);                   // packed references, r norms, scale
    b += nabo_align_up((size_t)n_query * 8, 256) * 2;                 // q norms, qn2
    b += nabo_align_up((size_t)n_items * max_split * nq * tc::TILE * ((size_t)kpl.cap * 8 + 8), 256) + 512;   // candidate buffers, counts, thresholds
    b += nabo_align_up((size_t)n_query * kprime * 4 * NABO_TC_MAX_SPLIT, 256);   // candidate indices (per reference range)
    b += nabo_align_up((size_t)n_query * 4 * NABO_TC_MAX_SPLIT, 256) + nabo_align_up((size_t)n_query * 4, 256);   // cert tau, fail rows
    b += nabo_align_up((size_t)(3 + n_items) * 4, 256);              // norm maxima, CTA ticket, head flags
    b += 4096;
    return b;
}

// ------------------------------------------------------------------ reference half of the operands
// Packed reference tiles and their norms: what the workspace holds for one call, and the first part of a prepared
// reference's buffer (which adds the scale and the norm maximum, kTcRefTail bytes).
size_t nabo_tc_ref_bytes(int n_ref, int g) {
    const size_t tb = tc::tile_bytes(tc::kp_for(g));
    const int n_rtiles = (n_ref + tc::TILE - 1) / tc::TILE;
    return nabo_align_up((size_t)n_rtiles * tb, 256) + nabo_align_up((size_t)n_ref * 8, 256);
}
static const size_t kTcRefTail = 512;      // scal[4] and the reference's norm maximum, 256-aligned pieces each

static void tc_ref_norms(const double* r, int ldr, int n_ref, int g, double* rnorm, unsigned int* maxr_bits, cudaStream_t st) {
    tc::norms_kernel<<<(n_ref + 255) / 256, 256, 0, st>>>(r, ldr, n_ref, g, rnorm, maxr_bits);
}

static void tc_ref_pack(const double* r, int ldr, int n_ref, int g, const double* rnorm, const double* scal,
                        const uint8_t* mask, __half* rb, cudaStream_t st) {
    const int n_rtiles = (n_ref + tc::TILE - 1) / tc::TILE;
    tc::pack_kernel<false><<<n_rtiles, tc::TILE * tc::PACK_SPLIT, 0, st>>>(r, ldr, n_ref, g, tc::kp_for(g), rnorm, scal, mask,
                                                                          rb, nullptr);
}

size_t nabo_tc_prepared_bytes(int n_ref, int g) { return nabo_tc_ref_bytes(n_ref, g) + kTcRefTail; }

// A prepared reference's operands: the same norms and packing as a one-shot call, but the scale comes from the
// reference's largest norm alone (cosine: 32), so that any later query batch can use the tiles.
int nabo_tc_prepare_ref(const double* r, int ldr, int n_ref, int g, int metric, const uint8_t* mask, void* buffer,
                        NaboTcRef* out, cudaStream_t st) {
    const int n_rtiles = (n_ref + tc::TILE - 1) / tc::TILE;
    NaboArena ar(buffer, nabo_tc_prepared_bytes(n_ref, g));
    __half* rb = (__half*)ar.take<char>((size_t)n_rtiles * tc::tile_bytes(tc::kp_for(g)));
    double* rnorm = ar.take<double>(n_ref);
    double* scal = ar.take<double>(4);
    unsigned int* maxr = ar.take<unsigned int>(1);
    if (!ar.ok) return nabo_set_error(NABO_EINVAL, "ref_prepare: buffer layout");
    NABO_CUDA(cudaMemsetAsync(maxr, 0, sizeof(unsigned int), st));
    tc_ref_norms(r, ldr, n_ref, g, rnorm, maxr, st);
    tc::scale_kernel<<<1, 1, 0, st>>>(maxr, maxr, metric == NABO_COSINE ? 1 : 0, scal);
    tc_ref_pack(r, ldr, n_ref, g, rnorm, scal, mask, rb, st);
    NABO_LAUNCH_CHECK("tc reference preparation");
    out->rb = rb;
    out->scal = scal;
    return 0;
}

// Runs norms -> scale -> pack -> candidate kernel.  Outputs (device, inside the arena):
// cand_idx [n_query][kprime], cert_tau [n_query], qn2 [n_query], scal[4].  pre != NULL: the reference half comes
// from a prepared reference (nabo_tc_prepare_ref) and only the queries are packed, with its scale.
int nabo_tc_candidates(const double* q, int ldq, const double* r, int ldr, int n_query, int n_ref, int g, int k,
                       int metric, const uint8_t* mask, int drop_first, int* n_split_io, NaboArena& ar, int32_t** cand_idx_out,
                       int* kprime_out, float** cert_tau_out, double** qn2_out, double** scal_out, int* launches,
                       NaboStageTimer& tm, cudaStream_t st, NaboCandBuf* raw_out, NaboTailSplit* tail, const NaboTcRef* pre) {
    // raw_out != NULL: when every query has ONE buffer (no reference split, K' <= 64) the final selection is left to
    // the re-rank kernel: raw_out is filled and no emit kernel runs.
    // *n_split_io in: reference pieces per item when there are few items (nabo_tc_split), or 0 = one piece (the
    // public candidate entry point: one K' list per query); out: K' lists per query
    int n_split = *n_split_io;
    const int kp = tc::kp_for(g);
    const tc::SmemPlan pl = tc::plan_smem(g);
    const size_t tb = tc::tile_bytes(kp);
    const int n_items = (n_query + pl.nq * tc::TILE - 1) / (pl.nq * tc::TILE);
    const int n_qtiles = n_items * pl.nq;
    const int n_rtiles = (n_ref + tc::TILE - 1) / tc::TILE;
    const tc::KPlan kpl = tc::plan_k(k + (drop_first ? 1 : 0));
    const int kprime = kpl.kprime;
    if (n_split < 1 || n_split > NABO_TC_MAX_SPLIT || kpl.cap != tc::CAP_SMALL) n_split = 1;   // 256 keys: unsplit only
    const int grid = tc_grid(n_items * n_split);

    __half* qa = (__half*)ar.take<char>((size_t)n_qtiles * tb);
    __half* rb = pre ? (__half*)pre->rb : (__half*)ar.take<char>((size_t)n_rtiles * tb);
    double* qnorm = ar.take<double>(n_query);
    double* qn2 = ar.take<double>(n_query);
    double* rnorm = pre ? nullptr : ar.take<double>(n_ref);
    const size_t n_slots = (size_t)n_items * n_split * pl.nq * tc::TILE;
    unsigned long long* cbuf = ar.take<unsigned long long>(n_slots * kpl.cap);
    int* ccnt = ar.take<int>(n_slots);
    float* ctau = ar.take<float>(n_slots);
    int32_t* cand = ar.take<int32_t>((size_t)n_query * kprime * n_split);
    float* tau = ar.take<float>((size_t)n_query * n_split);
    double* scal = pre ? (double*)pre->scal : ar.take<double>(4);
    unsigned int* maxbits = ar.take<unsigned int>(3 + (size_t)n_items);    // 2 norm maxima, CTA ticket, head flags
    if (!ar.ok) return nabo_set_error(NABO_EWORKSPACE, "knn: workspace too small for the tensor-core pass");

    NABO_CUDA(cudaMemsetAsync(maxbits, 0, (3 + (size_t)n_items) * sizeof(unsigned int), st));
    tc::norms_kernel<<<(n_query + 255) / 256, 256, 0, st>>>(q, ldq, n_query, g, qnorm, maxbits);
    if (!pre) {
        tc_ref_norms(r, ldr, n_ref, g, rnorm, maxbits + 1, st);
        tc::scale_kernel<<<1, 1, 0, st>>>(maxbits, maxbits + 1, metric == NABO_COSINE ? 1 : 0, scal);
    }
    tc::pack_kernel<true><<<n_qtiles, tc::TILE * tc::PACK_SPLIT, 0, st>>>(q, ldq, n_query, g, kp, qnorm, scal, nullptr, qa, qn2);
    if (!pre) tc_ref_pack(r, ldr, n_ref, g, rnorm, scal, mask, rb, st);
    NABO_LAUNCH_CHECK("tc pack kernels");
    tm.end(3);

    tc::Params p;
    p.qa = qa; p.rb = rb;
    p.n_query = n_query; p.n_ref = n_ref; p.kp = kp; p.n_items = n_items; p.n_rtiles = n_rtiles;
    p.stages = pl.stages; p.kprime = kprime; p.kc_out = kprime; p.n_split = n_split;
    p.cand_buf = cbuf; p.cand_cnt = ccnt; p.cand_tau = ctau; p.cand_idx = cand; p.cert_tau = tau; p.ticket = maxbits + 2;
    p.a_off = pl.a_off; p.b_off = pl.b_off; p.sort_off = pl.sort_off; p.bar_off = pl.bar_off;
    p.soft = kpl.cap - tc::CHUNK - 16 > kprime ? kpl.cap - tc::CHUNK - 16 : kprime;
    // Cut items at CTA boundaries only when the last wave would be partly filled and the packed reference fits in half of
    // L2 (the running items' candidate buffers take 57 MB at g <= 52 with 128 keys; with 256 keys they take 116 MB, 78 MB
    // in the wide plan, and reference + buffers exceed L2 - yet the cuts still pay there: 100 k queries at k = 100,
    // g = 50, candidate kernel 5.36 -> 4.80 ms against 100 k references (31 MB packed) and 7.68 -> 6.81 ms against 190 k
    // (61 MB), B200 at a 1 000 W power limit, so both plans keep this rule).  The cuts put the CTAs'
    // sweeps out of step by up to an item.  Measured on a B200 (1 000 W power limit) at the two ends only: at 100 k x 100 k,
    // g = 50 (31 MB packed) the cuts take the candidate kernel from 3.62 to 3.25 ms; at 500 k x 2 M cosine, g = 50 (625 MB
    // packed) they took the kNN from 3.9e12 to 3.3e12 pairs/s (-18 %; the SM clock under the power cap fell from 1.52 to
    // 1.30 GHz: the CTAs no longer share the reference tiles they read from HBM).  Between about 63 and 625 MB the half-L2
    // line is a reasoned choice, not a measured one.  Without cuts every CTA c sweeps the items c, c + grid, ... (contiguous
    // blocks of whole items measured 2 % slower at 500 k x 2 M), as it does for a whole number of waves.
    p.cut = n_items % grid != 0 && (size_t)n_rtiles * tb <= l2_bytes() / 2 ? 1 : 0;
    // Without cuts the last wave is partly filled (see NaboTailSplit): every CTA signals after its last full-wave item
    // when the caller can use the gap - the fused re-rank path only, at least two waves, at least 16 SMs idle in the last
    // one.  At 500 k x 2 M cosine (1 303 items) dropping this overlap cost 2.5 % of the kNN stage.
    const bool fused = raw_out && n_split == 1 && kprime <= 64;
    const int rem_items = n_items % grid;
    const bool tail_applies = tail && fused && !p.cut && n_items > grid && rem_items > 0 && grid - rem_items >= 16;
    const bool overlap = tail_applies && !tail->dry;
    p.signal_round = overlap ? n_items / grid : 0;
    if (tail) {
        tail->applies = tail_applies ? 1 : 0;
        tail->rows_full = overlap ? (n_items - rem_items) * pl.nq * tc::TILE : 0;
    }
#define NABO_TC_LAUNCH1(KS, SPLIT, NQ, SLAB, CAP)                                                                  \
    do {                                                                                                           \
        NABO_CUDA(cudaFuncSetAttribute(tc::candidates_kernel<KS, SPLIT, NQ, SLAB, CAP>,                            \
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.total));               \
        tc::candidates_kernel<KS, SPLIT, NQ, SLAB, CAP><<<grid, tc::NTHREADS, pl.total, st>>>(p);                  \
    } while (0)
#define NABO_TC_LAUNCH(KS, NQ, SLAB)                                                                               \
    do {                                                                                                           \
        if (kpl.cap == tc::CAP_LARGE) NABO_TC_LAUNCH1(KS, false, NQ, SLAB, tc::CAP_LARGE);                         \
        else if (n_split > 1) NABO_TC_LAUNCH1(KS, true, NQ, SLAB, tc::CAP_SMALL);                                  \
        else NABO_TC_LAUNCH1(KS, false, NQ, SLAB, tc::CAP_SMALL);                                                  \
    } while (0)
    if (pl.stages < 2) return nabo_set_error(NABO_EUNSUPPORTED, "knn: g=%d outside the tensor-core tile plans", g);
    if (pl.nq == 2) {                             // 53 <= g <= 128 (wide plan): slabs of 4 or 2 K steps
        if (pl.slab == 4) NABO_TC_LAUNCH(0, 2, 4);
        else NABO_TC_LAUNCH(0, 2, 2);
    } else if (kp == 160) NABO_TC_LAUNCH(10, 3, 0);    // g = 50 (BASELINE configs 2-5)
    else if (kp == 80) NABO_TC_LAUNCH(5, 3, 0);        // g = 25 (config 1)
    else NABO_TC_LAUNCH(0, 3, 0);
#undef NABO_TC_LAUNCH1
#undef NABO_TC_LAUNCH
    NABO_LAUNCH_CHECK("candidates_kernel");
    if (!overlap) tm.end(0);       // the final selection below is timed with the re-rank stage; with a dependent launch the
                                   // caller ends the stage after that launch (nothing may sit between the two kernels)
    if (fused) {
        raw_out->buf = cbuf; raw_out->cnt = ccnt; raw_out->tau = ctau; raw_out->kprime = kprime;
        *cand_idx_out = cand; *kprime_out = kprime; *cert_tau_out = tau; *qn2_out = qn2; *scal_out = scal;
        *launches += pre ? 3 : 6;
        *n_split_io = 1;
        return 0;
    }
    if (raw_out) raw_out->buf = nullptr;
    const unsigned emit_blocks = (unsigned)((n_slots + 7) / 8);
    if (kpl.cap == tc::CAP_LARGE) {
        if (pl.nq == 2) tc::emit_kernel<2, tc::CAP_LARGE><<<emit_blocks, 256, 0, st>>>(p);
        else tc::emit_kernel<3, tc::CAP_LARGE><<<emit_blocks, 256, 0, st>>>(p);
    } else if (pl.nq == 2) tc::emit_kernel<2><<<emit_blocks, 256, 0, st>>>(p);
    else tc::emit_kernel<3><<<emit_blocks, 256, 0, st>>>(p);
    NABO_LAUNCH_CHECK("emit_kernel");
    *launches += 1;
    if (n_split > 1) {
        int rc = nabo_tau_min_launch(tau, n_query, n_split, st);
        if (rc) return rc;
        *launches += 1;
    }
    *n_split_io = n_split;
    *cand_idx_out = cand; *kprime_out = kprime; *cert_tau_out = tau; *qn2_out = qn2; *scal_out = scal;
    *launches += pre ? 3 : 6;
    return 0;
}

#ifdef NABO_TC_STATS
extern "C" int nabo_dbg_tc_stats(unsigned long long* out_host, int reset) {
    cudaDeviceSynchronize();
    cudaMemcpyFromSymbol(out_host, tc::g_tc_stats, sizeof(unsigned long long) * tc::TC_NSTATS);
    if (reset) { static unsigned long long z[tc::TC_NSTATS]; cudaMemcpyToSymbol(tc::g_tc_stats, z, sizeof(z)); }
    return 0;
}
#endif

// The unsplit schedule as the kernel computes it (tests/test_tc_schedule_cpu.py): out[2 b], out[2 b + 1] =
// sched_bound(b) for b = 0 .. grid; the modelled cost F(x) of the first x reference tiles of an item.
extern "C" int nabo_dbg_tc_sched_bounds(int n_items, int n_rtiles, int grid, int kprime, int* out) {
    for (int b = 0; b <= grid; ++b) tc::sched_bound(b, n_items, n_rtiles, grid, kprime, out[2 * b], out[2 * b + 1]);
    return 0;
}
extern "C" double nabo_dbg_tc_sweep_cost(int x, int kprime) { return tc::sweep_cost(x, kprime); }

// ------------------------------------------------------------------ public candidate-pass entry points
// The public candidate pass keeps the 128-key plan only (k + drop_first + 8 <= 96): its K' never exceeds 96.
static bool candidates_supported(int g, int k, int drop_first) {
    return tc_plan_fits(g) && k + (drop_first ? 1 : 0) + 8 <= tc::MAX_KPRIME;
}

extern "C" int nabo_knn_candidates_width(int k, int drop_first) {
    return tc::kprime_for(k + (drop_first ? 1 : 0), tc::MAX_KPRIME);
}

extern "C" size_t nabo_knn_candidates_workspace_bytes(int n_query, int n_ref, int g, int k, int drop_first) {
    return nabo_tc_workspace_bytes(n_query, n_ref, g, k, drop_first);
}

extern "C" int nabo_knn_candidates(const double* q, int ldq, const double* r, int ldr, int n_query, int n_ref, int g,
                                   int k, int metric, const uint8_t* ref_mask, int drop_first, int32_t* out_cand,
                                   float* out_tau, double* out_qn2, double* out_scal, void* workspace,
                                   size_t workspace_bytes, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    NABO_ARG(metric == NABO_EUCLIDEAN || metric == NABO_COSINE, "candidates: metric %d has no tensor-core pass", metric);
    NABO_ARG(n_query >= 1 && n_ref >= 1 && ldq >= g && ldr >= g, "candidates: bad sizes");
    NABO_ARG(q && r && out_cand && out_tau, "candidates: null pointer");
    if (!candidates_supported(g, k, drop_first))
        return nabo_set_error(NABO_EUNSUPPORTED, "candidates: g=%d k=%d outside the tensor-core tile plan", g, k);
    NaboArena ar(workspace, workspace_bytes);
    NaboStageTimer tm(false, st);
    int32_t* cand = nullptr;
    float* tau = nullptr;
    double *qn2 = nullptr, *scal = nullptr;
    int kprime = 0, launches = 0;
    int one_list = 0;
    int rc = nabo_tc_candidates(q, ldq, r, ldr, n_query, n_ref, g, k, metric, ref_mask, drop_first, &one_list, ar, &cand,
                                &kprime, &tau, &qn2, &scal, &launches, tm, st);
    if (rc) return rc;
    NABO_CUDA(cudaMemcpyAsync(out_cand, cand, sizeof(int32_t) * (size_t)n_query * kprime, cudaMemcpyDeviceToDevice, st));
    NABO_CUDA(cudaMemcpyAsync(out_tau, tau, sizeof(float) * (size_t)n_query, cudaMemcpyDeviceToDevice, st));
    if (out_qn2) NABO_CUDA(cudaMemcpyAsync(out_qn2, qn2, sizeof(double) * (size_t)n_query, cudaMemcpyDeviceToDevice, st));
    if (out_scal) NABO_CUDA(cudaMemcpyAsync(out_scal, scal, sizeof(double) * 4, cudaMemcpyDeviceToDevice, st));
    return 0;
}
