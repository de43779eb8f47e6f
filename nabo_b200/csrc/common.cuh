// Shared helpers for the nabo_b200 CUDA library (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdint.h>
#include <math_constants.h>

#include "../../include/nabo_b200.h"

// ---- error channel: no exceptions cross the C ABI (SURVEY.md 8b) ------------------
int nabo_set_error(int code, const char* fmt, ...);

#define NABO_ARG(cond, ...)                                        \
    do {                                                           \
        if (!(cond)) return nabo_set_error(NABO_EINVAL, __VA_ARGS__); \
    } while (0)

#define NABO_CUDA(call)                                                                  \
    do {                                                                                 \
        cudaError_t e__ = (call);                                                        \
        if (e__ != cudaSuccess)                                                          \
            return nabo_set_error((int)e__, "%s failed: %s", #call, cudaGetErrorString(e__)); \
    } while (0)

#define NABO_LAUNCH_CHECK(name)                                                          \
    do {                                                                                 \
        cudaError_t e__ = cudaGetLastError();                                            \
        if (e__ != cudaSuccess)                                                          \
            return nabo_set_error((int)e__, "launch of %s failed: %s", name, cudaGetErrorString(e__)); \
    } while (0)

// -DNABO_CHECK: device-side bounds assertions in the hand-rolled pipelines (candidate-buffer appends, emit, tile
// indices).  compute-sanitizer is closed on the GPU pool this was developed on, so the test suite is run once
// against a library built with this switch instead (tools/build_variant.py check -DNABO_CHECK; profiles/).
#ifdef NABO_CHECK
#define NABO_DEV_ASSERT(cond) do { if (!(cond)) { printf("NABO_CHECK failed: %s (%s:%d)\n", #cond, __FILE__, __LINE__); __trap(); } } while (0)
#else
#define NABO_DEV_ASSERT(cond)
#endif

static inline size_t nabo_align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// Bump allocator over a caller-owned workspace.  A measuring arena (no memory) only counts: running a carve on it
// and reading `off` gives the bytes the same carve takes from a real workspace.
struct NaboArena {
    char* base;
    size_t off, cap;
    bool ok;
    NaboArena(void* p, size_t bytes) : base((char*)p), off(0), cap(bytes), ok(true) {}
    static NaboArena measure() { return NaboArena(nullptr, 0); }
    template <typename T>
    T* take(size_t n) {
        off = nabo_align_up(off, 256);
        size_t need = n * sizeof(T);
        if (base == nullptr || off + need > cap) { ok = false; off += need; return nullptr; }
        T* r = (T*)(base + off);
        off += need;
        return r;
    }
};

// ---- (distance, index) ordering used everywhere --------------------------------
// Order: ascending distance, ties by ascending index; NaN / masked are mapped to +inf
// by the producers so that they sort last (numpy.ma.argsort semantics, _mapping.py:140).
__device__ __forceinline__ bool nabo_less(double da, int ia, double db, int ib) {
    return (da < db) || (da == db && ia < ib);
}

// Warp-cooperative bitonic sort of n = power-of-two (d, i) pairs in shared memory.
__device__ __forceinline__ void warp_bitonic_sort(double* d, int* idx, int n, int lane) {
    for (int size = 2; size <= n; size <<= 1) {
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int t = lane; t < (n >> 1); t += 32) {
                int lo = 2 * t - (t & (stride - 1));
                int hi = lo + stride;
                bool up = ((lo & size) == 0);
                double dl = d[lo], dh = d[hi];
                int il = idx[lo], ih = idx[hi];
                bool sw = up ? nabo_less(dh, ih, dl, il) : nabo_less(dl, il, dh, ih);
                if (sw) {
                    d[lo] = dh; d[hi] = dl;
                    idx[lo] = ih; idx[hi] = il;
                }
            }
            __syncwarp();
        }
    }
}

// The same order for NU * 32 pairs held in registers: position u * 32 + lane is slot u of lane `lane`.  Strides below
// 32 exchange through shuffles, strides of 32 and more are register swaps inside the lane; no shared memory.
template <int NU>
__device__ __forceinline__ void warp_bitonic_sort_regs(double (&d)[NU], int (&ix)[NU], int lane) {
#pragma unroll
    for (int size = 2; size <= NU * 32; size <<= 1) {
#pragma unroll
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            if (stride >= 32) {
                const int su = stride >> 5;
#pragma unroll
                for (int u = 0; u < NU; ++u) {
                    if (u & su) continue;
                    const bool up = (((u << 5) | lane) & size) == 0;
                    const int v = u | su;
                    const bool sw = up ? nabo_less(d[v], ix[v], d[u], ix[u]) : nabo_less(d[u], ix[u], d[v], ix[v]);
                    const double dl = d[u], dh = d[v];
                    const int il = ix[u], ih = ix[v];
                    d[u] = sw ? dh : dl; d[v] = sw ? dl : dh;
                    ix[u] = sw ? ih : il; ix[v] = sw ? il : ih;
                }
            } else {
#pragma unroll
                for (int u = 0; u < NU; ++u) {
                    const bool up = (((u << 5) | lane) & size) == 0;
                    const bool want_min = ((lane & stride) == 0) == up;
                    const double pd = __shfl_xor_sync(0xffffffffu, d[u], stride);
                    const int pi = __shfl_xor_sync(0xffffffffu, ix[u], stride);
                    const bool take = want_min ? nabo_less(pd, pi, d[u], ix[u]) : nabo_less(d[u], ix[u], pd, pi);
                    d[u] = take ? pd : d[u];
                    ix[u] = take ? pi : ix[u];
                }
            }
        }
    }
}

// Same for packed 64-bit keys (sortable-float << 32 | index).
__device__ __forceinline__ void warp_bitonic_sort_u64(unsigned long long* a, int n, int lane) {
    for (int size = 2; size <= n; size <<= 1) {
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int t = lane; t < (n >> 1); t += 32) {
                int lo = 2 * t - (t & (stride - 1));
                int hi = lo + stride;
                bool up = ((lo & size) == 0);
                unsigned long long x = a[lo], y = a[hi];
                if (up ? (y < x) : (x < y)) { a[lo] = y; a[hi] = x; }
            }
            __syncwarp();
        }
    }
}

__device__ __forceinline__ uint32_t float_to_sortable(float f) {
    uint32_t b = __float_as_uint(f);
    return b ^ ((b >> 31) ? 0xFFFFFFFFu : 0x80000000u);
}
__device__ __forceinline__ float sortable_to_float(uint32_t u) {
    uint32_t b = u ^ ((u >> 31) ? 0x80000000u : 0xFFFFFFFFu);
    return __uint_as_float(b);
}

// SMs of the current device; 148 (B200) when no device answers, so that the workspace-size functions run without one.
static inline int nabo_sm_count() {
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    return sms;
}

static inline int nabo_next_pow2(int x) {
    int p = 1;
    while (p < x) p <<= 1;
    return p;
}
