// mnf_moments.cu -- reduction over Monte-Carlo samples for MNFFeedForward.predict:
//   sums[0, b, n] += sum_s f(y)[s * B + b, n],   sums[1, b, n] += sum_s f(y)[s * B + b, n]^2
// with f = identity or a per-row softmax (mean class probabilities and their spread).  Rows are sample-major, as
// forward_mc lays them out.  Every output element is owned by one thread that walks s in order, in fp64 (the variance is
// finished as E[y^2] - E[y]^2, which fp32 would lose to cancellation), so the sums do not depend on the launch geometry
// and need no atomics.  A call forms its sums from zero and adds them to the buffer once: sums split at chunk boundaries
// then add up to the same bits as one call over all samples.  With softmax the kernel can also sum each sample row's
// entropy H(softmax(y)) into entropy_sums[b] (mnf_mc_class_moments), under the same ordering and add-once rules.
#include <math.h>

#include "common.cuh"

namespace mnf {

__global__ void __launch_bounds__(256) mc_moments_kernel(const float *__restrict__ y, long long n_elems, long long n_samples,
                                                         double *__restrict__ sums) {
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < n_elems; e += (long long)gridDim.x * blockDim.x) {
        double s1 = 0.0, s2 = 0.0;
        const float *p = y + e;
#pragma unroll 4
        for (long long s = 0; s < n_samples; ++s) {
            const double v = (double)__ldg(p + s * n_elems);
            s1 += v;
            s2 = fma(v, v, s2);
        }
        sums[e] += s1;
        sums[n_elems + e] += s2;
    }
}

// softmax rows: one warp per (unique row b, block of kSoftmaxCols columns).  The row's max and normaliser come from a
// lane-strided pass over all its columns and a butterfly reduction, which leaves the same bits in every lane; each lane
// then accumulates its own kSoftmaxCols / 32 columns.  entropy_sums (nullable): the warp of column block 0 also forms
//   H_s = log z - (1 / z) sum_c e_c (y_c - m),   e_c = expf(y_c - m),  z = sum_c e_c
// in fp64 over all columns (terms with e_c == 0 skipped: 0 log 0 = 0, and a -inf column adds nothing), sums it over the
// samples in order and adds it to entropy_sums[b] once.  The sums path is the same code with or without it.
constexpr int kSoftmaxCols = 128;

__global__ void __launch_bounds__(256) mc_moments_softmax_kernel(const float *__restrict__ y, long long n_unique,
                                                                 long long n_samples, int n_cols, double *__restrict__ sums,
                                                                 double *__restrict__ entropy_sums) {
    constexpr int CPL = kSoftmaxCols / 32;
    const int lane = threadIdx.x & 31;
    const int n_blk = (n_cols + kSoftmaxCols - 1) / kSoftmaxCols;
    const long long n_items = n_unique * n_blk, warps = (long long)gridDim.x * (blockDim.x >> 5);
    for (long long it = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; it < n_items; it += warps) {
        const long long b = it / n_blk;
        const int c0 = (int)(it % n_blk) * kSoftmaxCols;
        const bool entropy = entropy_sums != nullptr && c0 == 0;  // warp-uniform
        double s1[CPL], s2[CPL], h = 0.0;
#pragma unroll
        for (int k = 0; k < CPL; ++k) s1[k] = 0.0, s2[k] = 0.0;
        for (long long s = 0; s < n_samples; ++s) {
            const float *row = y + (s * n_unique + b) * n_cols;
            float m = -INFINITY;
            for (int n = lane; n < n_cols; n += 32) m = fmaxf(m, __ldg(row + n));
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
            float z = 0.f;
            for (int n = lane; n < n_cols; n += 32) z += expf(__ldg(row + n) - m);
            z = warp_sum(z);
            const double inv = 1.0 / (double)z;
#pragma unroll
            for (int k = 0; k < CPL; ++k) {
                const int n = c0 + lane + 32 * k;
                if (n < n_cols) {
                    const double p = (double)expf(__ldg(row + n) - m) * inv;
                    s1[k] += p;
                    s2[k] = fma(p, p, s2[k]);
                }
            }
            if (entropy) {
                double t = 0.0;
                for (int n = lane; n < n_cols; n += 32) {
                    const float d = __ldg(row + n) - m, e = expf(d);
                    if (e != 0.f) t = fma((double)e, (double)d, t);
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
                h += log((double)z) - inv * t;
            }
        }
        if (entropy && lane == 0) entropy_sums[b] += h;
        const long long plane = n_unique * n_cols;
#pragma unroll
        for (int k = 0; k < CPL; ++k) {
            const int n = c0 + lane + 32 * k;
            if (n < n_cols) {
                sums[b * n_cols + n] += s1[k];
                sums[plane + b * n_cols + n] += s2[k];
            }
        }
    }
}

}  // namespace mnf

using namespace mnf;

namespace {

int mc_moments(const float *y, int64_t n_unique, int64_t n_samples, int n_cols, int softmax, double *sums,
               double *entropy_sums, void *stream) {
    MNF_REQUIRE(softmax == 0 || softmax == 1, MNF_E_ARG, "softmax must be 0 or 1 (got %d)", softmax);
    MNF_REQUIRE(n_unique >= 1 && n_samples >= 0 && n_cols >= 1, MNF_E_SHAPE,
                "bad shape: n_unique=%lld n_samples=%lld n_cols=%d", (long long)n_unique, (long long)n_samples, n_cols);
    MNF_REQUIRE(n_unique <= (INT64_MAX / n_cols) / (n_samples > 0 ? n_samples : 1), MNF_E_SHAPE, "too many elements");
    if (n_samples == 0) return 0;
    const DeviceProps *dp = device_props();
    MNF_REQUIRE(dp != nullptr, MNF_E_DEVICE, "no CUDA device");
    const long long cap = (long long)dp->sm_count * 16;
    cudaStream_t st = (cudaStream_t)stream;
    if (softmax) {
        const long long warps = n_unique * ((n_cols + kSoftmaxCols - 1) / kSoftmaxCols);
        long long blocks = (warps + 7) / 8;
        mc_moments_softmax_kernel<<<(unsigned)(blocks < cap ? blocks : cap), 256, 0, st>>>(y, n_unique, n_samples, n_cols,
                                                                                             sums, entropy_sums);
        return launch_status("mc_moments_softmax_kernel");
    }
    const long long n_elems = n_unique * n_cols;
    long long blocks = (n_elems + 255) / 256;
    mc_moments_kernel<<<(unsigned)(blocks < cap ? blocks : cap), 256, 0, st>>>(y, n_elems, n_samples, sums);
    return launch_status("mc_moments_kernel");
}

}  // namespace

extern "C" {

int mnf_mc_moments(const float *y, int64_t n_unique, int64_t n_samples, int n_cols, int softmax, double *sums,
                   void *stream) {
    MNF_REQUIRE(y && sums, MNF_E_ARG, "NULL pointer");
    return mc_moments(y, n_unique, n_samples, n_cols, softmax, sums, nullptr, stream);
}

int mnf_mc_class_moments(const float *y, int64_t n_unique, int64_t n_samples, int n_cols, double *sums,
                         double *entropy_sums, void *stream) {
    MNF_REQUIRE(y && sums && entropy_sums, MNF_E_ARG, "NULL pointer");
    return mc_moments(y, n_unique, n_samples, n_cols, 1, sums, entropy_sums, stream);
}

}  // extern "C"
