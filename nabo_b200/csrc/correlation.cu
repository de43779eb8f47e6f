// Row centring of the correlation metric (include/nabo_b200.h, NABO_CORRELATION): out[i][k] = x[i][k] - mu_i with
// mu_i = (x[i][0] + ... + x[i][g-1]) / g, the sum sequential in ascending k.  The kNN entry points centre the queries
// and the reference once per call and run the cosine engines on the copies (knn.cu).
#include "knn_internal.cuh"

namespace {

constexpr int CENTRE_NT = 256;   // 8 rows per block, one warp each

// Lanes load 32 consecutive coordinates of the row at a time (coalesced) and every lane adds them in ascending k from
// shuffles, so each lane holds the same sequential sum and no broadcast is needed.
__global__ void __launch_bounds__(CENTRE_NT)
centre_rows_kernel(const double* __restrict__ x, int ld, int n, int g, double* __restrict__ out) {
    const long long row = (long long)blockIdx.x * (CENTRE_NT / 32) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= n) return;                                   // warp-uniform
    const double* p = x + row * ld;
    double s = 0.0;
    for (int k0 = 0; k0 < g; k0 += 32) {
        const double v = k0 + lane < g ? p[k0 + lane] : 0.0;
        const int nk = min(32, g - k0);
        for (int j = 0; j < nk; ++j) s = __dadd_rn(s, __shfl_sync(0xffffffffu, v, j));
    }
    const double mu = __ddiv_rn(s, (double)g);
    double* o = out + row * g;
    for (int k = lane; k < g; k += 32) o[k] = __dsub_rn(p[k], mu);
}

}  // namespace

int nabo_centre_rows(const double* x, int ld, int n, int g, double* out, cudaStream_t st) {
    if (n == 0) return 0;
    const int rows = CENTRE_NT / 32;
    centre_rows_kernel<<<(unsigned)((n + rows - 1) / rows), CENTRE_NT, 0, st>>>(x, ld, n, g, out);
    NABO_LAUNCH_CHECK("centre_rows_kernel");
    return 0;
}
