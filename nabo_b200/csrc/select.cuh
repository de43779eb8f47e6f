// Per-query running top-K' selection over a CAP-entry key buffer in global memory (L2 resident):
// shared by the tensor-core candidate kernel (tc_candidates.cu) and the bit-sliced Canberra kernel
// (canberra_sliced.cu).  All routines are warp-cooperative; `lane` is the caller's lane id.
#pragma once
#include "common.cuh"

namespace sel {

// A buffer holds 32 * KPL keys (KPL keys per lane: element i = u * 32 + lane sits in slot u of its lane); KPL is a
// template parameter of every routine below.  CAP: the 128-key buffers of the Canberra pass, the fused re-rank
// (exact.cu) and the tensor-core pass up to K' = 96; the tensor-core pass for K' > 96 uses 256 keys (tc_candidates.cu).
constexpr int CAP = 128;

// buffer key = raw float bits of the score (high word) | local reference index (low word);
// the compaction routines convert to an order-preserving integer when they load a key
__device__ __forceinline__ unsigned long long make_key(float score, uint32_t col) {
    return ((unsigned long long)__float_as_uint(score) << 32) | col;
}

// ---- warp-cooperative compaction entirely in registers -----------------------------------
// The 32 * KPL keys of one query are spread KPL per lane (element i = u*32 + lane) and sorted by
// score with a bitonic network: strides >= 32 are register-to-register, smaller strides are
// shuffles.  Only the score is compared (ties keep an arbitrary member; everything dropped
// still has score >= the new threshold, which is all the certificate needs).
__device__ __forceinline__ void cex(uint32_t& s0, uint32_t& p0, uint32_t& s1, uint32_t& p1, bool up) {
    // after: (s0 <= s1) if up else (s0 >= s1)
    const bool sw = up ? (s1 < s0) : (s0 < s1);
    if (sw) { uint32_t t = s0; s0 = s1; s1 = t; t = p0; p0 = p1; p1 = t; }
}

template <int KPL>
__device__ __forceinline__ void sortn(uint32_t (&s)[KPL], uint32_t (&pl)[KPL], int lane) {
#pragma unroll
    for (int size = 2; size <= 32 * KPL; size <<= 1) {
#pragma unroll
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            if (stride >= 32) {
                const int du = stride >> 5;
#pragma unroll
                for (int u = 0; u < KPL; ++u) {
                    if ((u & du) == 0) {
                        const bool up = (((u * 32) & size) == 0);      // lane bits never reach `size` >= 64
                        cex(s[u], pl[u], s[u | du], pl[u | du], up);
                    }
                }
            } else {
#pragma unroll
                for (int u = 0; u < KPL; ++u) {
                    const int i = u * 32 + lane;
                    const uint32_t os = __shfl_xor_sync(0xffffffffu, s[u], stride);
                    const uint32_t op = __shfl_xor_sync(0xffffffffu, pl[u], stride);
                    const bool up = ((i & size) == 0);
                    const bool lower = ((lane & stride) == 0);
                    const bool take_min = (up == lower);
                    const bool other = take_min ? (os < s[u]) : (s[u] < os);
                    if (other) { s[u] = os; pl[u] = op; }
                }
            }
        }
    }
}

// Exact compaction: sort lane `src`'s buffer (n live keys), keep the kprime best at the front of the
// buffer.  New count / threshold come back through nc / nt (valid on every lane); s / pl hold the sorted
// keys.  Force-inlined where the caller consumes s / pl (the per-item final emit) so that the arrays
// stay in registers; compact_select uses the out-of-line wrapper below as its rare fallback.
template <int KPL>
__device__ __forceinline__ void compact_sort_inline(unsigned long long* gbuf, int n, int lane, int kprime,
                                                    uint32_t (&s)[KPL], uint32_t (&pl)[KPL], int& nc, float& nt) {
    __syncwarp();            // the owner's appends (plain global stores) are ordered before our loads
#pragma unroll
    for (int u = 0; u < KPL; ++u) {
        const int i = u * 32 + lane;
        const unsigned long long kv = i < n ? __ldcg(gbuf + i) : 0ull;     // through L2: never a stale L1 line
        s[u] = i < n ? float_to_sortable(__uint_as_float((uint32_t)(kv >> 32))) : 0xffffffffu;
        pl[u] = (uint32_t)kv;
    }
    sortn(s, pl, lane);
    nc = n < kprime ? n : kprime;
#pragma unroll
    for (int u = 0; u < KPL; ++u) {
        const int i = u * 32 + lane;
        if (i < nc) gbuf[i] = ((unsigned long long)__float_as_uint(sortable_to_float(s[u])) << 32) | pl[u];
    }
    // threshold = score of element kprime-1 (only meaningful when n >= kprime)
    const int e = kprime - 1;
    uint32_t ts = s[0];
#pragma unroll
    for (int u = 1; u < KPL; ++u)
        if ((e >> 5) == u) ts = s[u];
    ts = __shfl_sync(0xffffffffu, ts, e & 31);
    nt = n >= kprime ? sortable_to_float(ts) : CUDART_INF_F;
    __syncwarp();
}

template <int KPL>
static __device__ __noinline__ void compact_sort(unsigned long long* gbuf, int n, int lane, int kprime, int& nc, float& nt) {
    uint32_t s[KPL], pl[KPL];
    compact_sort_inline(gbuf, n, lane, kprime, s, pl, nc, nt);
}

// Cheap running compaction: one 256-bin histogram pass over the scores of the buffer finds a
// cut with at least kprime keys at or below it; those keys are kept (a few more than kprime),
// the rest is dropped, and the new threshold is the largest kept score.  Every dropped key
// lies in a higher bin, i.e. has a strictly larger score, so the certificate invariant
// ("everything rejected or dropped has score >= tau") holds without an exact selection.
// If the cut keeps more than max_keep keys (ties, duplicates) the exact sort takes over.
// hist: 256 counters of this warp in shared memory.
template <int KPL>
static __device__ __noinline__ void compact_select(unsigned long long* gbuf, int n, int lane, int kprime, int max_keep,
                                            uint32_t* hist, int& nc, float& nt) {
    __syncwarp();
    float fv[KPL];
    uint32_t pl[KPL];
    float flo = CUDART_INF_F, fhi = -CUDART_INF_F;
#pragma unroll
    for (int u = 0; u < KPL; ++u) {
        const int i = u * 32 + lane;
        const unsigned long long kv = i < n ? __ldcg(gbuf + i) : 0ull;
        fv[u] = __uint_as_float((uint32_t)(kv >> 32));
        pl[u] = (uint32_t)kv;
        if (i < n) { flo = fminf(flo, fv[u]); fhi = fmaxf(fhi, fv[u]); }
    }
    flo = sortable_to_float(__reduce_min_sync(0xffffffffu, float_to_sortable(flo)));
    fhi = sortable_to_float(__reduce_max_sync(0xffffffffu, float_to_sortable(fhi)));
    // zero the histogram (8 bins per lane)
    reinterpret_cast<uint4*>(hist)[lane * 2] = make_uint4(0, 0, 0, 0);
    reinterpret_cast<uint4*>(hist)[lane * 2 + 1] = make_uint4(0, 0, 0, 0);
    __syncwarp();
    const float range = fhi - flo;
    const float scale = range > 0.f ? 255.999f / range : 0.f;       // monotone map of [flo, fhi] onto bins 0..255
    int bin[KPL];
#pragma unroll
    for (int u = 0; u < KPL; ++u) {
        const int i = u * 32 + lane;
        bin[u] = max(0, min(255, (int)((fv[u] - flo) * scale)));
        if (i < n) atomicAdd(&hist[bin[u]], 1u);
    }
    __syncwarp();
    // prefix over the 256 bins: each lane owns 8 consecutive bins
    const uint4 h0 = reinterpret_cast<const uint4*>(hist)[lane * 2];
    const uint4 h1 = reinterpret_cast<const uint4*>(hist)[lane * 2 + 1];
    const uint32_t c[8] = {h0.x, h0.y, h0.z, h0.w, h1.x, h1.y, h1.z, h1.w};
    uint32_t mine = 0;
#pragma unroll
    for (int e = 0; e < 8; ++e) mine += c[e];
    uint32_t incl = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += v;
    }
    // first lane whose inclusive prefix reaches kprime holds the cut bin
    const unsigned reach = __ballot_sync(0xffffffffu, incl >= (uint32_t)kprime);
    int cut_bin = 255;
    uint32_t kept = (uint32_t)n;
    if (reach) {
        const int owner = __ffs(reach) - 1;
        uint32_t run = incl - mine;
        int b = 7;
        uint32_t k_at = 0;
        bool found = false;
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            run += c[e];
            if (!found && run >= (uint32_t)kprime) { found = true; b = e; k_at = run; }
        }
        cut_bin = __shfl_sync(0xffffffffu, lane * 8 + b, owner);
        kept = __shfl_sync(0xffffffffu, k_at, owner);
    }
    if ((int)kept > max_keep) {
        compact_sort<KPL>(gbuf, n, lane, kprime, nc, nt);
        return;
    }
    // stream-compact the kept keys to the front (all keys are in registers: in-place is safe)
    uint32_t base = 0;
    float tmax = -CUDART_INF_F;
#pragma unroll
    for (int u = 0; u < KPL; ++u) {
        const int i = u * 32 + lane;
        const bool keep = i < n && bin[u] <= cut_bin;
        const unsigned m = __ballot_sync(0xffffffffu, keep);
        if (keep) {
            gbuf[base + __popc(m & ((1u << lane) - 1u))] = ((unsigned long long)__float_as_uint(fv[u]) << 32) | pl[u];
            tmax = fmaxf(tmax, fv[u]);
        }
        base += __popc(m);
    }
    tmax = sortable_to_float(__reduce_max_sync(0xffffffffu, float_to_sortable(tmax)));
    nc = (int)kept;
    nt = reach ? tmax : CUDART_INF_F;
    __syncwarp();
}

// The histogram cut of compact_select on keys already in registers: bin[u] of every live key and the cut bin with
// at least kprime keys at or below it (kept = how many).  reach = false when n < kprime (keep everything).
// fv[u] of element i = u * 32 + lane, live iff i < n.  hist: 256 counters of this warp in shared memory.
template <int KPL>
__device__ __forceinline__ void histogram_cut(const float (&fv)[KPL], int n, int lane, int kprime, uint32_t* hist,
                                              int (&bin)[KPL], int& cut_bin, int& kept, bool& reach_out) {
    float flo = CUDART_INF_F, fhi = -CUDART_INF_F;
#pragma unroll
    for (int u = 0; u < KPL; ++u)
        if (u * 32 + lane < n) { flo = fminf(flo, fv[u]); fhi = fmaxf(fhi, fv[u]); }
    flo = sortable_to_float(__reduce_min_sync(0xffffffffu, float_to_sortable(flo)));
    fhi = sortable_to_float(__reduce_max_sync(0xffffffffu, float_to_sortable(fhi)));
    reinterpret_cast<uint4*>(hist)[lane * 2] = make_uint4(0, 0, 0, 0);
    reinterpret_cast<uint4*>(hist)[lane * 2 + 1] = make_uint4(0, 0, 0, 0);
    __syncwarp();
    const float range = fhi - flo;
    const float scale = range > 0.f ? 255.999f / range : 0.f;
#pragma unroll
    for (int u = 0; u < KPL; ++u) {
        bin[u] = max(0, min(255, (int)((fv[u] - flo) * scale)));
        if (u * 32 + lane < n) atomicAdd(&hist[bin[u]], 1u);
    }
    __syncwarp();
    const uint4 h0 = reinterpret_cast<const uint4*>(hist)[lane * 2];
    const uint4 h1 = reinterpret_cast<const uint4*>(hist)[lane * 2 + 1];
    const uint32_t c[8] = {h0.x, h0.y, h0.z, h0.w, h1.x, h1.y, h1.z, h1.w};
    uint32_t mine = 0;
#pragma unroll
    for (int e = 0; e < 8; ++e) mine += c[e];
    uint32_t incl = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += v;
    }
    const unsigned reach = __ballot_sync(0xffffffffu, incl >= (uint32_t)kprime);
    cut_bin = 255;
    kept = n;
    reach_out = reach != 0;
    if (reach) {
        const int owner = __ffs(reach) - 1;
        uint32_t run = incl - mine;
        int b = 7;
        uint32_t k_at = 0;
        bool found = false;
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            run += c[e];
            if (!found && run >= (uint32_t)kprime) { found = true; b = e; k_at = run; }
        }
        cut_bin = __shfl_sync(0xffffffffu, lane * 8 + b, owner);
        kept = (int)__shfl_sync(0xffffffffu, k_at, owner);
    }
    __syncwarp();
}

}  // namespace sel
