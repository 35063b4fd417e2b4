// mnf_functions.cu -- posterior function samples of an MNFLinear (exact fp32, arbitrary shapes):
//   * the weight draw: W[s] = W_mean * z[s] + exp(0.5 W_log_var) * E[s],  b[s] = b_mean + exp(0.5 b_log_var) * e[s],
//     one image [S, n_out, n_in] + [S, n_out] per chunk of samples
//   * the function GEMM: out[s, m] = A_s[m] @ W[s]^T + b[s] (+ ReLU, + folded eval-mode BatchNorm1d), the samples on
//     grid dimension z of the SIMT skeleton in mnf_common.cuh
// Unlike MNFLinear.forward's local reparameterisation, every input row of sample s sees the same W[s], b[s]: the
// outputs of one sample are one network evaluated at several inputs.
#include "mnf_common.cuh"

namespace mnf {

struct FnWeightArgs {
    const float *Wm, *Wlv, *bm, *blv;  // [n_out, n_in], [n_out]
    const float *z;                    // [S, n_in]
    NoiseSrc E, e;                     // injected [S, n_out, n_in] / [S, n_out], or Philox (row_offset unused)
    uint64_t sample_offset;
    float *W, *b;  // [S, n_out, n_in], [S, n_out]
    long long S;
    int n_in, n_out;
};

// the four normals of Philox block q: the element -> word mapping of philox_normal, so element 4q + u draws n4[u]
__device__ __forceinline__ void quad_normals(const Philox &rng, uint64_t q, uint32_t stream, float (&n4)[4]) {
    const uint4 r = rng(q, stream);
    const float2 a = box_muller(r.x, r.y), c = box_muller(r.z, r.w);
    n4[0] = a.x, n4[1] = a.y, n4[2] = c.x, n4[3] = c.y;
}

// A thread owns one aligned quad of GLOBAL element indices (one Philox block) of an image whose local element l has
// global index base + l; `row` elements share a parameter row (n_out * n_in for W, n_out for b), `inner` is the
// length of the innermost axis (n_in for W, n_out for b).  The quad's first element is decoded once and the others
// follow by increments, so the loop carries no 64-bit division per element.
template <bool W_IMAGE>
__device__ __forceinline__ void draw_weights(const FnWeightArgs &a) {
    const NoiseSrc src = W_IMAGE ? a.E : a.e;
    const long long row = W_IMAGE ? (long long)a.n_out * a.n_in : a.n_out, total = a.S * row;
    const int inner = W_IMAGE ? a.n_in : a.n_out;
    const uint64_t base = a.sample_offset * (uint64_t)row;
    const Philox rng(src.seed);
    const uint64_t q_end = (base + (uint64_t)total + 3) >> 2;
    for (uint64_t q = (base >> 2) + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; q < q_end;
         q += (uint64_t)gridDim.x * blockDim.x) {
        const long long l0 = (long long)(4 * q - base);  // -3 .. -1 for a first quad that starts before the image
        const long long ls = l0 < 0 ? 0 : l0;
        float n4[4] = {0.f, 0.f, 0.f, 0.f};
        if (!src.ptr) quad_normals(rng, q, src.stream, n4);
        long long s = ls / row, rem = ls - s * row;
        int i = (int)(rem % inner);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const long long l = l0 + u;
            if (l < 0) continue;
            if (l >= total) break;
            const float nv = src.ptr ? src.ptr[l] : n4[u];
            if constexpr (W_IMAGE)
                a.W[l] = fmaf(expf(0.5f * a.Wlv[rem]), nv, a.Wm[rem] * a.z[s * a.n_in + i]);
            else
                a.b[l] = fmaf(expf(0.5f * a.blv[rem]), nv, a.bm[rem]);
            if (++i == inner) i = 0;
            if (++rem == row) rem = 0, ++s;
        }
    }
}

__global__ void __launch_bounds__(256) function_weights_kernel(const FnWeightArgs a) {
    draw_weights<true>(a);
    draw_weights<false>(a);
}

// out[s, m, n] = A_s[m] . W[s, n] + b[s, n], then ReLU, then col_scale[n] * v + col_shift[n]; sample s = blockIdx.z.
// A_s = A + s * a_stride: a_stride 0 shares x [M, K] among the samples, M * K walks h [S, M, K].
struct MnfFunctionProb {
    int M, N, K;  // batch rows, n_out, n_in
    const float *A;
    long long a_stride;
    const float *W, *b;  // [S, N, K], [S, N]
    float *out;          // [S, M, N]
    int relu;
    const float *col_scale, *col_shift;  // NULL = none
    static constexpr bool kRowReduce = false;
    using RowCtx = size_t;
    __device__ RowCtx row_ctx(int m) const { return (size_t)blockIdx.z * a_stride + (size_t)m * K; }
    __device__ void load_a(const RowCtx &r, int, int k, float (&a)[1]) const { a[0] = A[r + k]; }
    __device__ void load_b(int n, int k, float (&v)[1]) const { v[0] = W[((size_t)blockIdx.z * N + n) * K + k]; }
    __device__ void epilogue4(int m0, int n, const float (&acc)[1][4], float (&)[4]) const {
        const size_t s = blockIdx.z;
        const float bn = b[s * N + n];
        const float sc = col_scale ? col_scale[n] : 1.f, sh = col_scale ? col_shift[n] : 0.f;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int m = m0 + i;
            if (m >= M) continue;
            const float v = acc[0][i] + bn;
            const float r = relu ? fmaxf(v, 0.f) : v;
            out[(s * M + m) * N + n] = col_scale ? fmaf(sc, r, sh) : r;
        }
    }
    __device__ void row_out(int, float) const {}
};

}  // namespace mnf

using namespace mnf;

extern "C" {

int mnf_linear_sample_weights(const float *W_mean, const float *W_log_var, const float *b_mean, const float *b_log_var,
                              const float *z, const float *eps_w, const float *eps_b, uint64_t seed,
                              uint32_t w_noise_stream, uint32_t b_noise_stream, uint64_t sample_offset, float *W_out,
                              float *b_out, int64_t n_samples, int n_in, int n_out, void *stream) {
    MNF_REQUIRE(W_mean && W_log_var && b_mean && b_log_var && z && W_out && b_out, MNF_E_ARG, "NULL pointer");
    MNF_REQUIRE(n_samples >= 0 && n_in >= 1 && n_out >= 1, MNF_E_ARG, "bad shape");
    const long long NK = (long long)n_out * n_in;
    MNF_REQUIRE(n_samples <= (1LL << 62) / NK, MNF_E_SHAPE, "weight image of %lld samples x %lld floats too large",
                (long long)n_samples, NK);
    MNF_REQUIRE(sample_offset <= (1ull << 63) / (uint64_t)NK - (uint64_t)n_samples, MNF_E_SHAPE,
                "sample_offset %llu overflows the 64-bit element index", (unsigned long long)sample_offset);
    if (n_samples == 0) return 0;
    const long long quads = (n_samples * NK) / 4 + 2;
    long long blocks = (quads + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    const FnWeightArgs a{W_mean, W_log_var, b_mean, b_log_var, z, NoiseSrc{eps_w, seed, w_noise_stream, 0},
                         NoiseSrc{eps_b, seed, b_noise_stream, 0}, sample_offset, W_out, b_out, (long long)n_samples,
                         n_in, n_out};
    function_weights_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(a);
    return launch_status("function_weights_kernel");
}

int mnf_linear_function_forward(const float *x, int x_per_sample, const float *W, const float *b, float *out,
                                int64_t n_samples, int64_t batch, int n_in, int n_out, int relu, const float *col_scale,
                                const float *col_shift, void *stream) {
    MNF_REQUIRE(x && W && b && out, MNF_E_ARG, "NULL pointer");
    MNF_REQUIRE((col_scale == nullptr) == (col_shift == nullptr), MNF_E_ARG,
                "col_scale and col_shift must both be given or both be NULL");
    MNF_REQUIRE(x_per_sample == 0 || x_per_sample == 1, MNF_E_ARG, "x_per_sample must be 0 or 1, got %d", x_per_sample);
    MNF_REQUIRE(n_samples >= 0 && batch >= 0 && n_in >= 1 && n_out >= 1, MNF_E_ARG, "bad shape");
    MNF_REQUIRE(n_samples <= 65535, MNF_E_SHAPE, "%lld samples in one call: at most 65535 (grid dimension z)",
                (long long)n_samples);
    MNF_REQUIRE(batch <= 0x7fffffff - 64, MNF_E_SHAPE, "batch of %lld rows too large for one call", (long long)batch);
    if (n_samples == 0 || batch == 0) return 0;
    const MnfFunctionProb p{(int)batch, n_out, n_in, x, x_per_sample ? (long long)batch * n_in : 0, W, b, out, relu,
                            col_scale, col_shift};
    // the tiled form for every batch size: a row's sum runs in the same order whatever else is in the batch
    return launch_simt_gemm<MnfFunctionProb, 1>(p, (cudaStream_t)stream, "mnf_linear_function_forward",
                                                (int)n_samples, false);
}

}  // extern "C"
