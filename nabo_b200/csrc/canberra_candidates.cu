// FP32 CUDA-core candidate pass for the modified Canberra metric (nabo/_mapping.py:29-45).
//
// The metric is not a contraction (per dimension: compare, divide, select), so tensor cores do not
// apply; the bound is the FP32 / SFU pipes.  Two phases per 64 x 64 tile of (query, reference) pairs:
//
//   phase 1  no division: count the dimensions where |x - y| < f|x| (the only ones whose term is
//            below 1).  d(x, y) >= g - count, so a pair whose bound already reaches the query's
//            running threshold tau is rejected.  The count runs in packed FP16 (HADD2 / HSET2 / HADD2 per
//            two pair-dimensions) on per-dimension power-of-two scaled copies; the threshold f|x| is
//            widened by the FP16 rounding bound so the count can only OVER-estimate (see fm16 below).
//   phase 2  the survivors (a few per cent once tau is warm) go to a shared-memory work list and
//            are evaluated densely, one pair per thread: term = |x - y| * rcp(|x| + |y| + 0.01).
//
// Both phases evaluate the predicate with an optimistic margin (f|x|(1 + delta)), so the FP32
// score is a LOWER bound of the exact FP64 distance up to eps = nabo_cb_eps(g).  Per-query top-K' lives in
// shared memory (packed sortable keys, warp bitonic compaction).  The exact FP64 re-rank and the
// certificate D_k < tau - eps (rerank_kernel, NABO_CERT_LINEAR) make the final result identical to
// the exact engine; uncertified rows fall back to it.
#include "common.cuh"
#include "knn_internal.cuh"

#include <cuda_fp16.h>

namespace cb {

constexpr int TQ = 64, TR = 64, NT = 512;
constexpr int CAP = 128;                // candidate keys per query in shared memory

struct Smem {
    float *xs, *xt, *xa;                // [g][TQ]  x, f|x|(1+delta), |x|
    float *ys0, *ys1;                   // [g][TR]  y, double-buffered (cp.async prefetch of the next tile)
    __half2* xh2;                       // [g][TQ][2]  (x,x) and (t,t) in FP16, per-dimension scaled
    __half *yh0, *yh1;                  // [g][TR]  FP16 scaled y, double-buffered
    unsigned long long* keys;           // [TQ][CAP]
    float* tau;                         // [TQ]
    int* cnt;                           // [TQ]
    unsigned short* work;               // [TQ*TR] packed (q << 8 | r)
    int* nwork;
};

__device__ __forceinline__ Smem carve(unsigned char* base, int g) {
    Smem s;
    s.keys = reinterpret_cast<unsigned long long*>(base);
    float* f = reinterpret_cast<float*>(s.keys + (size_t)TQ * CAP);
    s.xs = f; f += (size_t)g * TQ;
    s.xt = f; f += (size_t)g * TQ;
    s.xa = f; f += (size_t)g * TQ;
    s.ys0 = f; f += (size_t)g * TR;
    s.ys1 = f; f += (size_t)g * TR;
    s.xh2 = reinterpret_cast<__half2*>(f); f += (size_t)g * TQ * 2;
    s.yh0 = reinterpret_cast<__half*>(f); f += (size_t)g * TR / 2;
    s.yh1 = reinterpret_cast<__half*>(f); f += (size_t)g * TR / 2;
    s.tau = f; f += TQ;
    s.cnt = reinterpret_cast<int*>(f);
    s.nwork = s.cnt + TQ;
    s.work = reinterpret_cast<unsigned short*>(s.nwork + 4);
    return s;
}
static size_t smem_bytes(int g) {
    return (size_t)TQ * CAP * 8 + ((size_t)g * (3 * TQ + 2 * TR + 2 * TQ + TR) + TQ) * 4 + (TQ + 4) * 4 + (size_t)TQ * TR * 2;
}

// FP32 copy of a row-major FP64 matrix, pre-tiled k-major: out[(tile * g + k) * 64 + row_in_tile].
// A tile of the main kernel is then a straight, coalesced float4 copy.
__global__ void __launch_bounds__(256)
pretile_kernel(const double* __restrict__ x, int ld, int n, int g, float* __restrict__ out) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long total = (long long)((n + 63) / 64) * g * 64;
    if (e >= total) return;
    const int rl = (int)(e & 63);
    const long long tk = e >> 6;
    const int k = (int)(tk % g);
    const long long tile = tk / g;
    const long long row = tile * 64 + rl;
    out[e] = row < n ? (float)x[row * ld + k] : 0.f;
}

// max |value| per dimension over the finite entries (float bits are monotone for non-negative values)
__global__ void __launch_bounds__(256)
dimmax_kernel(const double* __restrict__ x, int ld, int n, int g, unsigned* __restrict__ maxbits) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (long long)n * g) return;
    const int k = (int)(e % g);
    const float v = fabsf((float)x[(e / g) * ld + k]);
    if (isfinite(v) && v > 0.f) atomicMax(maxbits + k, __float_as_uint(v));
}

// per-dimension power-of-two scale that brings the largest magnitude into [2^12, 2^13): no FP16 overflow,
// 29 binades of headroom below; the saturation predicate |x-y| < f|x| is scale-invariant
__global__ void dimscale_kernel(const unsigned* __restrict__ maxbits, int g, float* __restrict__ scale) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= g) return;
    const float mx = __uint_as_float(maxbits[k]);
    float sc = 1.f;
    if (mx > 0.f) { int e; frexpf(mx, &e); sc = ldexpf(1.f, 13 - e); }
    scale[k] = sc;
}

__global__ void __launch_bounds__(256)
pretile_half_kernel(const double* __restrict__ x, int ld, int n, int g, const float* __restrict__ scale,
                    __half* __restrict__ out) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long total = (long long)((n + 63) / 64) * g * 64;
    if (e >= total) return;
    const int rl = (int)(e & 63);
    const long long tk = e >> 6;
    const int k = (int)(tk % g);
    const long long row = (tk / g) * 64 + rl;
    out[e] = row < n ? __double2half(x[row * ld + k] * (double)scale[k]) : __float2half(0.f);
}

__device__ __forceinline__ void compact(const Smem& s, int q, int kprime, int lane) {
    unsigned long long* k = s.keys + (size_t)q * CAP;
    const int n = s.cnt[q];
    for (int i = n + lane; i < CAP; i += 32) k[i] = ~0ull;
    __syncwarp();
    warp_bitonic_sort_u64(k, CAP, lane);
    if (lane == 0 && n >= kprime) {
        s.cnt[q] = kprime;
        s.tau[q] = sortable_to_float((uint32_t)(k[kprime - 1] >> 32));
    }
    __syncwarp();
}

__global__ void __launch_bounds__(NT, 1)
candidates_kernel(const float* __restrict__ qt, const float* __restrict__ rt, const __half* __restrict__ rh,
                  const float* __restrict__ scale, int n_query, int n_ref, int g, float fm, float fm16, float a16,
                  const uint8_t* __restrict__ mask, int kprime, int32_t* __restrict__ cand,
                  float* __restrict__ tau_out) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const Smem s = carve(smem_raw, g);
    const int q0 = blockIdx.x * TQ;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int tr = threadIdx.x & 15, tq = threadIdx.x >> 4;      // 16 reference groups of 4, 32 query groups of 2
    const int nvec = g * TQ / 4;

    {
        const float4* src = reinterpret_cast<const float4*>(qt + (size_t)blockIdx.x * g * TQ);
        for (int e = threadIdx.x; e < nvec; e += NT) {
            const float4 x = src[e];
            reinterpret_cast<float4*>(s.xs)[e] = x;
            reinterpret_cast<float4*>(s.xa)[e] = make_float4(fabsf(x.x), fabsf(x.y), fabsf(x.z), fabsf(x.w));
            // NaN x -> NaN threshold -> predicate false -> term 1 (as the reference)
            reinterpret_cast<float4*>(s.xt)[e] = make_float4(fm * fabsf(x.x), fm * fabsf(x.y), fm * fabsf(x.z), fm * fabsf(x.w));
            // FP16 copies for phase 1: x_h = fl16(x * s_k); t_h = round-up(fm16 * |x_h| + a16) >= every |d_h| the
            // exact predicate can produce (derivation at fm16 in nabo_cb_candidates)
            const float sc = scale[(e * 4) / TQ];
            const float xv[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const __half xh = __float2half(xv[u] * sc);
                const __half th = __float2half_ru(fm16 * fabsf(__half2float(xh)) + a16);
                s.xh2[(e * 4 + u) * 2] = __half2half2(xh);
                s.xh2[(e * 4 + u) * 2 + 1] = __half2half2(th);
            }
        }
    }
    if (threadIdx.x < TQ) { s.cnt[threadIdx.x] = 0; s.tau[threadIdx.x] = CUDART_INF_F; }
    if (threadIdx.x < 2) s.nwork[threadIdx.x] = 0;

    // reference tiles are double-buffered: tile j+1 streams in with cp.async while tile j is processed
    auto prefetch = [&](int tile, float* dst, __half* dsth) {
        const float4* src = reinterpret_cast<const float4*>(rt + (size_t)tile * g * TR);
        for (int e = threadIdx.x; e < nvec; e += NT) {
            const unsigned sa = (unsigned)__cvta_generic_to_shared(reinterpret_cast<float4*>(dst) + e);
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sa), "l"(src + e) : "memory");
        }
        const uint4* srch = reinterpret_cast<const uint4*>(rh + (size_t)tile * g * TR);
        for (int e = threadIdx.x; e < nvec / 2; e += NT) {
            const unsigned sa = (unsigned)__cvta_generic_to_shared(reinterpret_cast<uint4*>(dsth) + e);
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sa), "l"(srch + e) : "memory");
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    const int n_tiles = (n_ref + TR - 1) / TR;
    prefetch(0, s.ys0, s.yh0);
    for (int tile = 0; tile < n_tiles; ++tile) {
        const int r0 = tile * TR;
        float* ys = (tile & 1) ? s.ys1 : s.ys0;
        const __half* yh = (tile & 1) ? s.yh1 : s.yh0;
        int* nwork = s.nwork + (tile & 1);                 // work-list counters alternate between tiles
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncthreads();                                   // tile landed; phase 2 of the previous tile finished
        if (tile + 1 < n_tiles) prefetch(tile + 1, (tile & 1) ? s.ys0 : s.ys1, (tile & 1) ? s.yh0 : s.yh1);
        // compaction of the previous tile's appends rides inside the phase-1 region (no extra barrier):
        // phase 1 only reads tau, and a slightly stale tau is still a valid threshold
        for (int ql = warp; ql < TQ; ql += NT / 32)
            if (s.cnt[ql] > CAP - TR) compact(s, ql, kprime, lane);
        // ---- phase 1: unsaturated-dimension counts of a 2 x 4 micro tile, two references per HFMA2-class op
        __half2 ch[2][2];
#pragma unroll
        for (int a = 0; a < 2; ++a)
#pragma unroll
            for (int b = 0; b < 2; ++b) ch[a][b] = __float2half2_rn(0.f);
#pragma unroll 4
        for (int k = 0; k < g; ++k) {
            const uint4 xt = *reinterpret_cast<const uint4*>(s.xh2 + (size_t)(k * TQ + tq * 2) * 2);   // (x,x)(t,t) x 2 queries
            const uint2 yv = *reinterpret_cast<const uint2*>(yh + k * TR + tr * 4);                     // 4 references
            const __half2 x2[2] = {*reinterpret_cast<const __half2*>(&xt.x), *reinterpret_cast<const __half2*>(&xt.z)};
            const __half2 t2[2] = {*reinterpret_cast<const __half2*>(&xt.y), *reinterpret_cast<const __half2*>(&xt.w)};
            const __half2 y2[2] = {*reinterpret_cast<const __half2*>(&yv.x), *reinterpret_cast<const __half2*>(&yv.y)};
#pragma unroll
            for (int a = 0; a < 2; ++a)
#pragma unroll
                for (int b = 0; b < 2; ++b)
                    ch[a][b] = __hadd2(ch[a][b], __hle2(__habs2(__hsub2(x2[a], y2[b])), t2[a]));
        }
        float c[2][4];
#pragma unroll
        for (int a = 0; a < 2; ++a)
#pragma unroll
            for (int b = 0; b < 2; ++b) {
                c[a][2 * b] = __low2float(ch[a][b]);
                c[a][2 * b + 1] = __high2float(ch[a][b]);
            }
#pragma unroll
        for (int a = 0; a < 2; ++a) {
            const int ql = tq * 2 + a;
            if (q0 + ql >= n_query) continue;
            const float tau = s.tau[ql];
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                const int rl = tr * 4 + b, j = r0 + rl;
                if (j >= n_ref || (mask && mask[j])) continue;
                if ((float)g - c[a][b] < tau) {                   // d >= g - count: bound still below tau
                    const int pos = atomicAdd(nwork, 1);
                    s.work[pos] = (unsigned short)((ql << 8) | rl);
                }
            }
        }
        __syncthreads();
        // ---- phase 2: dense evaluation of the survivors
        const int nw = *nwork;
        if (threadIdx.x == 0) s.nwork[(tile + 1) & 1] = 0;       // nobody touches the other counter until the next tile
        // four lanes per surviving pair (dimensions k = part, part + 4, ...), partial sums combined with two
        // shuffles: the work list is short once tau is warm, and one thread per pair left most of the block
        // idle at the next barrier.  (FP32 partial sums in a different order stay within nabo_cb_eps.)
        for (int base = 0; base < nw * 4; base += NT) {
            const int w4 = base + threadIdx.x;
            const bool active = w4 < nw * 4;
            const int w = active ? (w4 >> 2) : 0, part = w4 & 3;
            const int ql = s.work[w] >> 8, rl = s.work[w] & 255;
            float acc = 0.f;
            if (active) {
                for (int k = part; k < g; k += 4) {
                    const float x = s.xs[k * TQ + ql], y = ys[k * TR + rl];
                    const float num = fabsf(x - y);
                    const float term = __fdividef(num, s.xa[k * TQ + ql] + (fabsf(y) + 0.01f));
                    acc += (num < s.xt[k * TQ + ql]) ? term : 1.0f;
                }
            }
            acc += __shfl_xor_sync(0xffffffffu, acc, 1);
            acc += __shfl_xor_sync(0xffffffffu, acc, 2);
            if (active && part == 0 && acc < s.tau[ql]) {
                const int pos = atomicAdd(&s.cnt[ql], 1);
                s.keys[(size_t)ql * CAP + pos] =
                    ((unsigned long long)float_to_sortable(acc) << 32) | (unsigned)(r0 + rl);
            }
        }
    }
    __syncthreads();
    for (int ql = warp; ql < TQ; ql += NT / 32) {
        const int qi = q0 + ql;
        if (qi >= n_query) continue;
        const int n = s.cnt[ql];
        const float old_tau = s.tau[ql];
        compact(s, ql, kprime, lane);
        const unsigned long long* k = s.keys + (size_t)ql * CAP;
        const int nc = n < kprime ? n : kprime;
        for (int i = lane; i < kprime; i += 32) cand[(long long)qi * kprime + i] = i < nc ? (int32_t)(uint32_t)k[i] : -1;
        if (lane == 0) tau_out[qi] = n >= kprime ? s.tau[ql] : old_tau;
    }
}

}  // namespace cb

bool nabo_cb_supported(int g, int k, int drop_first) {
    const int ksel = k + (drop_first ? 1 : 0);
    return cb::smem_bytes(g) <= 227 * 1024 && ksel + 8 <= cb::CAP - cb::TR;
}

int nabo_cb_kprime(int k, int drop_first) {
    const int ksel = k + (drop_first ? 1 : 0);
    int kp = ksel + (ksel / 4 > 8 ? ksel / 4 : 8);
    if (kp > cb::CAP - cb::TR) kp = cb::CAP - cb::TR;
    return kp;
}

size_t nabo_cb_pretile_floats(int n, int g) { return (size_t)((n + 63) / 64) * g * 64; }
int nabo_cb_pretile_launch(const double* x, int ld, int n, int g, float* out, cudaStream_t st) {
    const size_t t = nabo_cb_pretile_floats(n, g);
    cb::pretile_kernel<<<(unsigned)((t + 255) / 256), 256, 0, st>>>(x, ld, n, g, out);
    NABO_LAUNCH_CHECK("cb::pretile_kernel");
    return 0;
}

void nabo_cb_carve(NaboArena& ar, int n_query, int n_ref, int g, const NaboFastPlan& p, NaboCbWork* w) {
    w->cand = ar.take<int32_t>((size_t)n_query * p.kprime);
    w->tau = ar.take<float>(n_query);
    w->qt = ar.take<float>(nabo_cb_pretile_floats(n_query, g));
    w->rt = ar.take<float>(nabo_cb_pretile_floats(n_ref, g));
    w->rh = ar.take<char>(nabo_cb_pretile_floats(n_ref, g) * 2);      // FP16 tiles of the reference
    w->maxbits = ar.take<unsigned>(g);                                // per-dimension maximum and scale
    w->scale = ar.take<float>(g);
}

// What either modified-Canberra pass hands to the re-rank: its score is a lower bound of the distance up to
// nabo_cb_eps(g).
void nabo_cb_result(const int32_t* cand, const float* tau, int n_cand, int g, int launches, NaboCandidates* out) {
    out->cand = cand; out->n_cand = n_cand; out->raw.buf = nullptr; out->rows_full = 0; out->launches = launches;
    out->cert.kind = NABO_CERT_LINEAR; out->cert.tau = tau; out->cert.qn2 = nullptr; out->cert.scal = nullptr;
    out->cert.c_acc = nabo_cb_eps(g); out->cert.abs_slack = 0.0;
}

int nabo_cb_candidates(const double* q, int ldq, const double* r, int ldr, int n_query, int n_ref, int g, double f,
                       const uint8_t* mask, const NaboFastPlan& p, const NaboCbWork& w, cudaStream_t st,
                       NaboCandidates* out) {
    const int kprime = p.kprime;
    __half* rh = (__half*)w.rh;
    {
        const size_t tq = nabo_cb_pretile_floats(n_query, g), tr = nabo_cb_pretile_floats(n_ref, g);
        NABO_CUDA(cudaMemsetAsync(w.maxbits, 0, sizeof(unsigned) * g, st));
        cb::dimmax_kernel<<<(unsigned)(((size_t)n_query * g + 255) / 256), 256, 0, st>>>(q, ldq, n_query, g, w.maxbits);
        cb::dimmax_kernel<<<(unsigned)(((size_t)n_ref * g + 255) / 256), 256, 0, st>>>(r, ldr, n_ref, g, w.maxbits);
        cb::dimscale_kernel<<<(g + 63) / 64, 64, 0, st>>>(w.maxbits, g, w.scale);
        cb::pretile_kernel<<<(unsigned)((tq + 255) / 256), 256, 0, st>>>(q, ldq, n_query, g, w.qt);
        cb::pretile_kernel<<<(unsigned)((tr + 255) / 256), 256, 0, st>>>(r, ldr, n_ref, g, w.rt);
        cb::pretile_half_kernel<<<(unsigned)((tr + 255) / 256), 256, 0, st>>>(r, ldr, n_ref, g, w.scale, rh);
        NABO_LAUNCH_CHECK("cb::pretile kernels");
    }
    const size_t smem = cb::smem_bytes(g);
    NABO_CUDA(cudaFuncSetAttribute(cb::candidates_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    // Optimistic margin of the saturation predicate: whenever the exact FP64 test |x-y| < f|x| holds, the
    // FP32 test on the rounded inputs must hold too.  Near the threshold |y| <= (1+f)|x|, so the FP32
    // difference is off by at most ~1.2e-7 (2+f)|x|; delta covers it with a 3x reserve.
    const double delta = fmax(1e-5, 4e-7 * (2.0 + f) / f);
    const float fm = (float)(f * (1.0 + delta));
    // FP16 phase 1.  With X = x s_k, Y = y s_k (exact), u = 2^-11 and eta = 2^-25 (subnormal step / 2):
    //   x_h = fl(X), y_h = fl(Y), d_h = fl(x_h - y_h):  |d_h| <= (1+u)(|X-Y| + u(|X|+|Y|) + 2 eta) + eta.
    // If |X-Y| < f|X| then |Y| < (1+f)|X| and |X| <= (|x_h| + eta)/(1-u), hence
    //   |d_h| < fm0 |x_h| + (fm0 + 4) eta,   fm0 = (1+u)(f + u(2+f))/(1-u).
    // t_h = round-up(fm16 |x_h| + a16) with fm16 = fm0 (1 + 1e-4), a16 = (fm0 + 4) eta therefore makes the
    // FP16 test |d_h| <= t_h true whenever the exact test is: the count can only over-estimate.
    const double u = 1.0 / 2048.0, eta = 1.0 / 33554432.0;
    const double fm0 = (1.0 + u) * (f + u * (2.0 + f)) / (1.0 - u);
    const float fm16 = (float)(fm0 * (1.0 + 1e-4));
    const float a16 = (float)((fm0 + 4.0) * eta);
    cb::candidates_kernel<<<(n_query + cb::TQ - 1) / cb::TQ, cb::NT, smem, st>>>(w.qt, w.rt, rh, w.scale, n_query, n_ref, g,
                                                                              fm, fm16, a16, mask, kprime, w.cand, w.tau);
    NABO_LAUNCH_CHECK("cb::candidates_kernel");
    nabo_cb_result(w.cand, w.tau, kprime, g, 7, out);
    return 0;
}

// |FP32 score - (a lower bound of) the exact distance|: sequential FP32 sum of g terms <= 1 plus the
// per-term rounding of the difference, the denominator and the approximate division.
double nabo_cb_eps(int g) { return 1.2e-7 * (double)g * g + 2e-6 * g + 4e-7 * g; }
