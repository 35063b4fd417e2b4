// mnf_layers.cu -- MNF layer kernels, exact-fp32 path (arbitrary shapes):
//   * z0 = q0_mean + sqrt(exp(q0_log_var)) * eps                      (mnf_linear.py:59-62)
//   * RNVP forward with injected or Philox masks                       (rnvp.py:25-39)
//   * MNFLinear.forward: dual GEMM sharing the x tile + noise epilogue (mnf_linear.py:46-56)
//   * MNFConv2d.forward as an implicit GEMM, optional fused ReLU + 2x2 max-pool epilogue
//                                                                      (mnf_conv.py:67-78)
// All GEMM-shaped work goes through the functor skeleton in mnf_common.cuh.
#include <cooperative_groups.h>

#include <cuda_fp16.h>

#include <type_traits>

#include "mnf_common.cuh"

namespace mnf {

// ---------------------------------------------------------------------------------------
__global__ void sample_z0_kernel(const float *__restrict__ q0_mean, const float *__restrict__ q0_log_var,
                                 NoiseSrc eps, float *__restrict__ z, long long n_rows, int dim) {
    const long long total = n_rows * dim;
    const Philox rng(eps.seed);
    // four consecutive elements per step: one Philox block yields exactly their four normals
    // (same element -> number mapping as philox_normal)
    for (long long e0 = 4 * ((long long)blockIdx.x * blockDim.x + threadIdx.x); e0 < total;
         e0 += 4LL * gridDim.x * blockDim.x) {
        float n4[4];
        if (eps.ptr == nullptr) {
            const uint4 q = rng((uint64_t)((long long)eps.row_offset * dim + e0) >> 2, eps.stream);
            const float2 a = box_muller(q.x, q.y), b = box_muller(q.z, q.w);
            n4[0] = a.x, n4[1] = a.y, n4[2] = b.x, n4[3] = b.y;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const long long e = e0 + u;
            if (e >= total) break;
            const int d = (int)(e % dim);
            const float std = sqrtf(expf(q0_log_var[d]));  // .exp().sqrt(), mnf_linear.py:59
            // (row_offset * dim) % 4 == 0 is required for the block alignment; otherwise fall back per element
            const float nz = eps.ptr ? eps.ptr[e]
                                     : ((((long long)eps.row_offset * dim) & 3) == 0
                                            ? n4[u]
                                            : philox_normal(rng, (uint64_t)((long long)eps.row_offset * dim + e), eps.stream));
            z[e] = q0_mean[d] + std * nz;
        }
    }
}

// ---------------------------------------------------------------------------------------
// plain Linear (+ optional LeakyReLU 0.2): extra conditioner layers when h_sizes has > 1 entry
struct LinearProb {
    int M, N, K;
    const float *A, *W, *b;
    float *C;
    int leaky;
    static constexpr bool kRowReduce = false;
    using RowCtx = size_t;
    __device__ RowCtx row_ctx(int m) const { return (size_t)m * K; }
    __device__ void load_a(const RowCtx &r, int, int k, float (&a)[1]) const { a[0] = A[r + k]; }
    __device__ void load_b(int n, int k, float (&v)[1]) const { v[0] = W[(size_t)n * K + k]; }
    __device__ void epilogue4(int m0, int n, const float (&acc)[1][4], float (&)[4]) const {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            if (m0 + i >= M) continue;
            float v = acc[0][i] + b[n];
            if (leaky) v = fmaxf(v, 0.2f * v);
            C[(size_t)(m0 + i) * N + n] = v;
        }
    }
    __device__ void row_out(int, float) const {}
};

// RNVP stage 1: y = (mask * z) @ Wn^T + bn        (rnvp.py:30-31)
struct RnvpHiddenProb {
    int M, N, K;  // rows, hidden, dim
    const float *z, *Wn, *bn;
    float *y;
    NoiseSrc mask;
    int leaky;
    static constexpr bool kRowReduce = false;
    using RowCtx = long long;
    __device__ RowCtx row_ctx(int m) const { return (long long)m * K; }
    __device__ void load_a(const RowCtx &r, int, int k, float (&a)[1]) const {
        const long long e = r + k;
        a[0] = noise_bernoulli(mask, e, (long long)mask.row_offset * K + e) * z[e];
    }
    __device__ void load_b(int n, int k, float (&v)[1]) const { v[0] = Wn[(size_t)n * K + k]; }
    __device__ void epilogue4(int m0, int n, const float (&acc)[1][4], float (&)[4]) const {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            if (m0 + i >= M) continue;
            float v = acc[0][i] + bn[n];
            if (leaky) v = fmaxf(v, 0.2f * v);
            y[(size_t)(m0 + i) * N + n] = v;
        }
    }
    __device__ void row_out(int, float) const {}
};

// RNVP stage 2: shift = y Wt^T + bt, scale = y Ws^T + bs, gated update + log-det (rnvp.py:32-39)
struct RnvpOutProb {
    int M, N, K;  // rows, dim, hidden
    const float *y, *Wt, *bt, *Ws, *bs;
    float *z;       // in/out [M, N]
    float *logdet;  // [M], accumulated with atomics over column tiles (zeroed by the caller)
    NoiseSrc mask;
    static constexpr bool kRowReduce = true;
    using RowCtx = size_t;
    __device__ RowCtx row_ctx(int m) const { return (size_t)m * K; }
    __device__ void load_a(const RowCtx &r, int, int k, float (&a)[2]) const { a[0] = a[1] = y[r + k]; }
    __device__ void load_b(int n, int k, float (&v)[2]) const {
        v[0] = Wt[(size_t)n * K + k];
        v[1] = Ws[(size_t)n * K + k];
    }
    __device__ void epilogue4(int m0, int n, const float (&acc)[2][4], float (&rowsum)[4]) const {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int m = m0 + i;
            if (m >= M) continue;
            const long long e = (long long)m * N + n;
            const float mk = noise_bernoulli(mask, e, (long long)mask.row_offset * N + e);
            const float shift = acc[0][i] + bt[n], scale = acc[1][i] + bs[n];
            const float gate = 1.f / (1.f + expf(-scale));  // torch.sigmoid
            const float zz = z[e];
            const float z1 = (1.f - mk) * zz, z2 = mk * zz;
            z[e] = (z1 * gate + (1.f - gate) * shift) + z2;  // rnvp.py:37 (shift reaches kept dims too)
            rowsum[i] += (1.f - mk) * logf(gate);           // rnvp.py:36
        }
    }
    __device__ void row_out(int m, float sum) const { atomicAdd(&logdet[m], sum); }
};

// MNFLinear.forward: mean = (x*z) Wm^T + bm ; var = x^2 exp(Wlv)^T + exp(blv) ; out = mean + sqrt(var) eps
struct MnfLinearProb {
    int M, N, K;  // rows, n_out, n_in
    const float *x;
    int x_rows;      // row m reads x[m % x_rows] (MC replication without materialising x.repeat)
    const float *z;  // [M, K]
    const float *Wm, *Wlv, *bm, *blv;
    float *out;
    NoiseSrc eps;
    int relu;
    // optional per-column affine map after the noise and ReLU, out = col_scale[n] * v + col_shift[n]: an eval-mode
    // BatchNorm1d folded to its inference coefficients (MNFFeedForward's hidden blocks); NULL = none
    const float *col_scale, *col_shift;
    static constexpr bool kRowReduce = false;
    struct RowCtx {
        size_t xo, zo;
    };
    __device__ RowCtx row_ctx(int m) const { return RowCtx{(size_t)(m % x_rows) * K, (size_t)m * K}; }
    __device__ void load_a(const RowCtx &r, int, int k, float (&a)[2]) const {
        const float xv = x[r.xo + k];
        a[0] = xv * z[r.zo + k];
        a[1] = xv * xv;
    }
    __device__ void load_b(int n, int k, float (&v)[2]) const {
        v[0] = Wm[(size_t)n * K + k];
        v[1] = expf(Wlv[(size_t)n * K + k]);
    }
    __device__ void epilogue4(int m0, int n, const float (&acc)[2][4], float (&)[4]) const {
        const float b0 = bm[n], b1 = expf(blv[n]);
        const float sc = col_scale ? col_scale[n] : 1.f, sh = col_scale ? col_shift[n] : 0.f;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int m = m0 + i;
            if (m >= M) continue;
            const long long e = (long long)m * N + n;
            const float mean = acc[0][i] + b0, var = acc[1][i] + b1;
            const float v = mean + sqrtf(var) * noise_normal(eps, e, (long long)eps.row_offset * N + e);
            const float a = relu ? fmaxf(v, 0.f) : v;
            out[e] = col_scale ? fmaf(sc, a, sh) : a;
        }
    }
    __device__ void row_out(int, float) const {}
};

// MNFConv2d.forward as an implicit GEMM: rows = output pixels, cols = output channels,
// K = n_in*k*k.  With `pool` the row index is pool-major (4 consecutive rows = one 2x2 window)
// and the epilogue applies ReLU + max over the window (the nn.ReLU / nn.MaxPool2d(2) that
// follow every MNFConv2d in MNFLeNet, mnf_lenet.py:16-21).
// GEOM: zero padding `pad`, stride `stride`, dilation `dil` and channel groups.  Output pixel (oy, ox) reads the window
// whose origin is (oy*stride - pad, ox*stride - pad), tap (ky, kx) at (ky*dil, kx*dil) from it; a tap outside the
// image loads 0, so it adds to neither moment.  With groups, the launch carries one problem per group on grid
// dimension z: N and K are the group's (n_out / groups columns, cg * ks * ks taps), group g reads input channels
// g*cg .. g*cg + cg - 1 and writes output channels g*N .. g*N + N - 1.  Without GEOM (pad 0, stride 1, dilation 1,
// one group) every tap is inside the image and the loads carry no bounds test.
template <bool GEOM>
struct MnfConvProb {
    int M, N, K;
    const float *x;  // [R, C, H, W]
    int x_imgs;      // image r reads x[r % x_imgs]
    int C, H, W, ks, OH, OW;
    const float *Wm, *Wlv, *blv;  // [N, C, ks, ks], [N] (GEOM: [N * groups, cg, ks, ks], [N * groups])
    const float *z;               // [N] multiplicative noise, shared by the batch (mnf_conv.py:72)
    float *out;                   // [R, N, OH, OW] or pooled [R, N, OH/2, OW/2]
    NoiseSrc eps;                 // indexed like the un-pooled output [R, N, OH, OW]
    int pool;
    float *sd_out;                // moments mode: out <- mean, sd_out <- sqrt(var), no noise
    static constexpr bool kRowReduce = false;
    __device__ __forceinline__ void decode(int m, int &r, int &oy, int &ox) const {
        if (pool) {
            const int q = m & 3, w = m >> 2;
            const int PW = OW >> 1, PH = OH >> 1;
            const int px = w % PW, py = (w / PW) % PH;
            r = w / (PW * PH);
            oy = 2 * py + (q >> 1);
            ox = 2 * px + (q & 1);
        } else {
            ox = m % OW;
            oy = (m / OW) % OH;
            r = m / (OW * OH);
        }
    }
    // offset of filter tap k inside an image, (ci*H + ky)*W + kx, tabulated on the host for the first kMaxTaps taps
    // (the table travels as a kernel parameter); wider filters compute the remaining offsets arithmetically
    static constexpr int kMaxTaps = 1600;
    int koff[kMaxTaps];
    int pad, stride;                 // GEOM only
    int kyx[GEOM ? kMaxTaps : 1];    // GEOM: (ky*dil << 16) | kx*dil of tap k, for the bounds test
    int dil, cg;                     // GEOM only: dilation, input channels per group
    __device__ __forceinline__ int tap_offset(int k) const {
        if (k < kMaxTaps) return koff[k];
        if constexpr (GEOM) {
            const int kx = (k % ks) * dil, ky = ((k / ks) % ks) * dil, ci = k / (ks * ks);
            return (ci * H + ky) * W + kx;
        } else {
            const int kx = k % ks, ky = (k / ks) % ks, ci = k / (ks * ks);
            return (ci * H + ky) * W + kx;
        }
    }
    // GEOM: global output channel of the group's column n, and the layer's channel count
    __device__ __forceinline__ int gcol(int n) const {
        if constexpr (GEOM) return (int)blockIdx.z * N + n;
        else return n;
    }
    __device__ __forceinline__ int n_total() const {
        if constexpr (GEOM) return N * (int)gridDim.z;
        else return N;
    }
    // GEOM: offset of the receptive-field origin in x (negative or past a row when it lies in the padding) and
    // the origin's coordinates; otherwise the offset alone
    struct GeomRow {
        long long o;
        int iy, ix;
    };
    using RowCtx = std::conditional_t<GEOM, GeomRow, size_t>;
    __device__ RowCtx row_ctx(int m) const {
        int r, oy, ox;
        decode(m, r, oy, ox);
        if constexpr (GEOM) {
            const int iy = oy * stride - pad, ix = ox * stride - pad;
            return GeomRow{(((long long)(r % x_imgs) * C + (long long)blockIdx.z * cg) * H + iy) * W + ix, iy, ix};
        } else {
            return ((size_t)(r % x_imgs) * C * H + oy) * W + ox;
        }
    }
    __device__ void load_a(const RowCtx &r, int, int k, float (&a)[2]) const {
        float xv;
        if constexpr (GEOM) {
            int ky, kx;
            if (k < kMaxTaps) {
                ky = kyx[k] >> 16, kx = kyx[k] & 0xffff;
            } else {
                kx = (k % ks) * dil, ky = ((k / ks) % ks) * dil;
            }
            const bool in = (unsigned)(r.iy + ky) < (unsigned)H && (unsigned)(r.ix + kx) < (unsigned)W;
            xv = in ? x[r.o + tap_offset(k)] : 0.f;
        } else {
            xv = x[r + tap_offset(k)];
        }
        a[0] = xv;
        a[1] = xv * xv;
    }
    __device__ void load_b(int gn, int k, float (&v)[2]) const {
        const int n = gcol(gn);
        v[0] = Wm[(size_t)n * K + k] * (z ? z[n] : 1.f);  // z == NULL: unit scale (per-sample z applied later)
        v[1] = expf(Wlv[(size_t)n * K + k]);
    }
    __device__ void epilogue4(int m0, int gn, const float (&acc)[2][4], float (&)[4]) const {
        const int n = gcol(gn), NT = n_total();
        const float bvar = expf(blv[n]);
        float best = 0.f;  // ReLU floor
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int m = m0 + i;
            if (m >= M) continue;
            int r, oy, ox;
            decode(m, r, oy, ox);
            const long long e = (((long long)r * NT + n) * OH + oy) * OW + ox;
            const long long ge = ((((long long)r + (long long)eps.row_offset) * NT + n) * OH + oy) * OW + ox;
            if (sd_out) {
                out[e] = acc[0][i];
                sd_out[e] = sqrtf(acc[1][i] + bvar);
                continue;
            }
            const float v = acc[0][i] + sqrtf(acc[1][i] + bvar) * noise_normal(eps, e, ge);  // b_mean == 0
            if (pool)
                best = fmaxf(best, v);
            else
                out[e] = v;
        }
        if (pool && m0 < M) {
            int r, oy, ox;
            decode(m0, r, oy, ox);
            out[(((size_t)r * NT + n) * (OH >> 1) + (oy >> 1)) * (OW >> 1) + (ox >> 1)] = best;
        }
    }
    __device__ void row_out(int, float) const {}
};

// out[r, c, py, px] = max over the 2x2 window of relu(mean[b] + sd[b] * eps[r]),  b = r % n_unique:
// the noise / ReLU / MaxPool2d(2) tail of an MNFConv2d whose mean and variance do not depend on the sample
// (z is shared by the whole call, mnf_conv.py:72, so under MC replication they are per-IMAGE quantities).
// zs (optional): per-sample channel scales [n_z, C] -- the per-sample conv-z option of the MC predict entry point
// (SURVEY 8f-4): z scales OUTPUT channels (mnf_conv.py:73), so with mean evaluated for z = 1 row r's mean is
// zs[r / rows_per_z, c] * mean.
struct PoolDivs {  // run-time divisors of the index decode, as multiply-shift pairs
    FastDiv pw2, ph, c;
};

template <bool IDX32>
__global__ void conv_noise_pool_kernel(const float *__restrict__ mean, const float *__restrict__ sd, int n_unique,
                                       NoiseSrc eps, float *__restrict__ out, long long n_rows, int C, int OH, int OW,
                                       const float *__restrict__ zs, long long rows_per_z, const PoolDivs dv) {
    // one thread = two horizontally adjacent pooled pixels = a 2 x 4 patch of the un-pooled map, so that each
    // Philox block (4 consecutive elements) is generated once and fully used.  Needs OW % 4 == 0 (host checks).
    // IDX32: fewer than 2^31 work items -- the decode runs on 32-bit multiply-shift divisions (the 64-bit
    // divide sequences were a third of the kernel's instructions).
    const int PH = OH >> 1, PW = OW >> 1, PW2 = PW >> 1;
    const long long total = n_rows * C * PH * PW2;
    const Philox rng(eps.seed);
    for (long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x; o < total;
         o += (long long)gridDim.x * blockDim.x) {
        int px2, py, c;
        long long r;
        if constexpr (IDX32) {
            uint32_t t, a, b, cc;
            dv.pw2.divmod((uint32_t)o, t, a);
            dv.ph.divmod(t, t, b);
            dv.c.divmod(t, t, cc);
            px2 = (int)a, py = (int)b, c = (int)cc, r = (long long)t;
        } else {
            px2 = (int)(o % PW2), py = (int)((o / PW2) % PH), c = (int)((o / ((long long)PW2 * PH)) % C);
            r = o / ((long long)PW2 * PH * C);
        }
        const size_t ub = (((size_t)(r % n_unique) * C + c) * OH + 2 * py) * OW + 4 * px2;
        const long long le = ((r * C + c) * OH + 2 * py) * OW + 4 * px2;  // index in the un-pooled [R, C, OH, OW]
        const long long ge = le + (long long)eps.row_offset * C * OH * OW;
        float best0 = 0.f, best1 = 0.f;  // ReLU floor
        const float zc = zs ? zs[(r / rows_per_z) * C + c] : 1.f;
#pragma unroll
        for (int dy = 0; dy < 2; ++dy) {
            float4 m4 = *reinterpret_cast<const float4 *>(mean + ub + dy * OW);
            m4.x *= zc, m4.y *= zc, m4.z *= zc, m4.w *= zc;
            const float4 s4 = *reinterpret_cast<const float4 *>(sd + ub + dy * OW);
            float4 n4;
            if (eps.ptr) {
                n4 = *reinterpret_cast<const float4 *>(eps.ptr + le + dy * OW);
            } else {
                const uint4 q = rng((uint64_t)(ge + (long long)dy * OW) >> 2, eps.stream);
                const float2 a = box_muller(q.x, q.y), b = box_muller(q.z, q.w);
                n4 = make_float4(a.x, a.y, b.x, b.y);
            }
            best0 = fmaxf(best0, fmaxf(fmaf(s4.x, n4.x, m4.x), fmaf(s4.y, n4.y, m4.y)));
            best1 = fmaxf(best1, fmaxf(fmaf(s4.z, n4.z, m4.z), fmaf(s4.w, n4.w, m4.w)));
        }
        *reinterpret_cast<float2 *>(out + ((r * C + c) * PH + py) * PW + 2 * px2) = make_float2(best0, best1);
    }
}

// im2col for the tensor-core conv: row m is pool-major (4 consecutive rows = one 2x2 window of one image),
// column k = (ci, ky, kx) padded with zeros to Kp; writes tf32(x) and tf32(x^2)
__global__ void __launch_bounds__(256)
conv_im2col_kernel(const float *__restrict__ x, float *__restrict__ a_mean, float *__restrict__ a_var,
                   long long n_imgs, int C, int H, int W, int ks, int OH, int OW, int Kp) {
    // one CTA per image: the image (C*H*W floats) and the tap-offset table live in shared memory, the CTA
    // then streams out its OH*OW rows of Kp columns as float4 (the kernel is write-bound: 2 * 4 * Kp bytes/row)
    extern __shared__ float sm[];
    float *xs = sm;
    int *koff = reinterpret_cast<int *>(sm + C * H * W);
    const int K = C * ks * ks, PW = OW >> 1, rows = OH * OW, k4n = Kp >> 2;
    auto rn = [](float f) {
        uint32_t b;
        asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(b) : "f"(f));
        return __uint_as_float(b);
    };
    for (int k = threadIdx.x; k < Kp; k += blockDim.x) {
        const int kx = k % ks, ky = (k / ks) % ks, ci = k / (ks * ks);
        koff[k] = k < K ? (ci * H + ky) * W + kx : -1;
    }
    for (long long img = blockIdx.x; img < n_imgs; img += gridDim.x) {
        __syncthreads();
        for (int i = threadIdx.x; i < C * H * W; i += blockDim.x) xs[i] = x[(size_t)img * C * H * W + i];
        __syncthreads();
        for (int t = threadIdx.x; t < rows * k4n; t += blockDim.x) {
            const int k4 = t % k4n, ml = t / k4n;  // ml: pool-major row inside the image
            const int q = ml & 3, w = ml >> 2;
            const int px = w % PW, py = w / PW;
            const int base = (2 * py + (q >> 1)) * W + 2 * px + (q & 1);
            float v[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int off = koff[4 * k4 + u];
                v[u] = off >= 0 ? xs[base + off] : 0.f;
            }
            const size_t o = ((size_t)img * rows + ml) * Kp + 4 * k4;
            *reinterpret_cast<float4 *>(a_mean + o) = make_float4(rn(v[0]), rn(v[1]), rn(v[2]), rn(v[3]));
            *reinterpret_cast<float4 *>(a_var + o) =
                make_float4(rn(v[0] * v[0]), rn(v[1] * v[1]), rn(v[2] * v[2]), rn(v[3] * v[3]));
        }
    }
}

// weights of the tensor-core conv: Bm[n][k] = tf32(W_mean[n][k] * z[n]), Bv[n][k] = tf32(exp(W_log_var[n][k])),
// rows padded to Np and columns to Kp with zeros; bvar_p[n] = b_log_var[n] (0 in the padding)
__global__ void conv_pack_weights_kernel(const float *__restrict__ Wm, const float *__restrict__ Wlv,
                                         const float *__restrict__ blv, const float *__restrict__ z, int N, int K,
                                         int Np, int Kp, float *__restrict__ Bm, float *__restrict__ Bv,
                                         float *__restrict__ bvar_p) {
    auto rn = [](float f) {
        uint32_t b;
        asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(b) : "f"(f));
        return __uint_as_float(b);
    };
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < Np * Kp; e += gridDim.x * blockDim.x) {
        const int n = e / Kp, k = e % Kp;
        const bool in = n < N && k < K;
        Bm[e] = in ? rn(Wm[(size_t)n * K + k] * (z ? z[n] : 1.f)) : 0.f;  // z == NULL: unit scale (per-sample z applied later)
        Bv[e] = in ? rn(expf(Wlv[(size_t)n * K + k])) : 0.f;
        if (k == 0) bvar_p[n] = n < N ? blv[n] : 0.f;
    }
}

// fp16 weights of the implicit-GEMM conv (tc_gemm.cu, conv_implicit_kernel): Bm = fp16(W_mean * z),
// Bv = fp16(exp(W_log_var) * 2^8) (scale undone by the kernel's epilogue: keeps variances down to 2.4e-7 in fp16's
// normal range), rows padded to Np and columns to Kp with zeros; bvar_p[n] = b_log_var[n]
__global__ void conv_pack_weights_f16_kernel(const float *__restrict__ Wm, const float *__restrict__ Wlv,
                                             const float *__restrict__ blv, const float *__restrict__ z, int N, int K,
                                             int Np, int Kp, __half *__restrict__ Bm, __half *__restrict__ Bv,
                                             float *__restrict__ bvar_p) {
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < Np * Kp; e += gridDim.x * blockDim.x) {
        const int n = e / Kp, k = e % Kp;
        const bool in = n < N && k < K;
        Bm[e] = __float2half_rn(in ? Wm[(size_t)n * K + k] * (z ? z[n] : 1.f) : 0.f);  // z == NULL: unit scale (per-sample z applied later)
        Bv[e] = __float2half_rn(in ? fminf(expf(Wlv[(size_t)n * K + k]) * 256.f, 65504.f) : 0.f);
        if (k == 0) bvar_p[n] = n < N ? blv[n] : 0.f;
    }
}

// ---------------------------------------------------------------------------------------
// One RNVP flow on ONE row (kl_div runs its q / r flows with a single z, mnf_linear.py:67, :83) in one launch:
// a thread-block cluster of 8 CTAs splits the conditioner's outputs (phase 1: y = W0 (mask*z) + b0, every CTA
// holds mask*z in shared memory), meets at a cluster barrier, then splits the dims (phase 2: shift / scale rows of
// t and s, gate, update, log-det partial).  The two-launch GEMV form took 23 + 13 us per flow at dim 4096.
// ---------------------------------------------------------------------------------------
constexpr int kRowCluster = 8;
__global__ void __cluster_dims__(kRowCluster, 1, 1) __launch_bounds__(256)
rnvp_row_kernel(const float *__restrict__ W0, const float *__restrict__ b0, int Hn, const float *__restrict__ Wt,
                const float *__restrict__ bt, const float *__restrict__ Ws, const float *__restrict__ bs, float *z,
                float *logdet, NoiseSrc mask, int dim, float *ybuf, float *inter) {
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    const int c = (int)cluster.block_rank(), tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    extern __shared__ float sm[];
    float *mz = sm, *ys = sm + dim, *red = ys + 64;
    for (int d = tid; d < dim; d += 256)
        mz[d] = noise_bernoulli(mask, d, (long long)mask.row_offset * dim + d) * z[d];
    __syncthreads();
    for (int j = c; j < Hn; j += kRowCluster) {  // phase 1: this CTA's conditioner outputs
        float acc = 0.f;
        for (int d = tid; d < dim; d += 256) acc = fmaf(W0[(size_t)j * dim + d], mz[d], acc);
        acc = warp_sum(acc);
        if (lane == 0) red[warp] = acc;
        __syncthreads();
        if (tid == 0) {
            float v = b0[j];
            for (int w = 0; w < 8; ++w) v += red[w];
            ybuf[j] = v;
        }
        __syncthreads();
    }
    __threadfence();
    cluster.sync();  // every y[j] is written, every CTA has finished reading z
    for (int j = tid; j < Hn; j += 256) ys[j] = __ldcg(ybuf + j);
    __syncthreads();
    const int per = (dim + kRowCluster - 1) / kRowCluster, d0 = c * per, d1 = min(dim, d0 + per);
    float ldsum = 0.f;
    for (int d = d0 + tid; d < d1; d += 256) {  // phase 2: this CTA's dims
        float shift = bt[d], scale = bs[d];
        const float *wt = Wt + (size_t)d * Hn, *ws = Ws + (size_t)d * Hn;
        for (int j = 0; j < Hn; ++j) {
            shift = fmaf(wt[j], ys[j], shift);
            scale = fmaf(ws[j], ys[j], scale);
        }
        const float mk = noise_bernoulli(mask, d, (long long)mask.row_offset * dim + d);
        const float gate = 1.f / (1.f + expf(-scale)), zz = z[d];
        const float zn = ((1.f - mk) * zz * gate + (1.f - gate) * shift) + mk * zz;  // rnvp.py:37
        z[d] = zn;
        if (inter) inter[d] = zn;
        ldsum += (1.f - mk) * logf(gate);  // rnvp.py:36
    }
    ldsum = warp_sum(ldsum);
    if (lane == 0) red[warp] = ldsum;
    __syncthreads();
    if (tid == 0) {
        float v = 0.f;
        for (int w = 0; w < 8; ++w) v += red[w];
        atomicAdd(logdet, v);
    }
}


// Direct form of the moments of a small MNFConv2d (few input taps, few output channels: MNF-LeNet's conv1 is
// 1 x 5 x 5 -> 20): as a GEMM it is M x 20 x 25, a shape the tiled SIMT GEMM runs at 1.4 TFLOP/s.  Here a CTA owns one
// image (staged in shared memory next to the folded weights [tap][channel]); a thread owns one output pixel and
// keeps the 2 x NP accumulators of all channels in registers: per tap one image load, NP / 2 broadcast LDS.128 and
// 2 NP FFMAs.
template <int NP>
__global__ void __launch_bounds__(256) conv_moments_direct_kernel(const float *__restrict__ x, const float *__restrict__ z,
                                                                  const float *__restrict__ Wm, const float *__restrict__ Wlv,
                                                                  const float *__restrict__ blv, float *__restrict__ mean_out,
                                                                  float *__restrict__ sd_out, long long n_imgs, int C, int H,
                                                                  int W, int ks, int N) {
    extern __shared__ __align__(16) float sm_direct[];
    const int K = C * ks * ks, OH = H - ks + 1, OW = W - ks + 1, img_floats = C * H * W;
    float *wm = sm_direct;                       // [K][NP]  W_mean * z
    float *wv = wm + K * NP;                     // [K][NP]  exp(W_log_var)
    float *bv = wv + K * NP;                     // [NP]     exp(b_log_var)
    int *koff = reinterpret_cast<int *>(bv + NP);  // [K]      offset of tap k inside an image
    float *xs = reinterpret_cast<float *>(koff + ((K + 3) & ~3));
    for (int i = threadIdx.x; i < K * NP; i += blockDim.x) {
        const int k = i / NP, n = i % NP;
        wm[i] = n < N ? Wm[(size_t)n * K + k] * (z ? z[n] : 1.f) : 0.f;  // z == NULL: unit scale (per-sample z applied later)
        wv[i] = n < N ? expf(Wlv[(size_t)n * K + k]) : 0.f;
    }
    for (int n = threadIdx.x; n < NP; n += blockDim.x) bv[n] = n < N ? expf(blv[n]) : 0.f;
    for (int k = threadIdx.x; k < K; k += blockDim.x) {
        const int kx = k % ks, ky = (k / ks) % ks, ci = k / (ks * ks);
        koff[k] = (ci * H + ky) * W + kx;
    }
    for (long long img = blockIdx.x; img < n_imgs; img += gridDim.x) {
        __syncthreads();
        for (int i = threadIdx.x; i < img_floats; i += blockDim.x) xs[i] = x[(size_t)img * img_floats + i];
        __syncthreads();
        for (int pix = threadIdx.x; pix < OH * OW; pix += blockDim.x) {
            const int oy = pix / OW, ox = pix % OW;
            const float *xp = xs + oy * W + ox;
            float am[NP], av[NP];
#pragma unroll
            for (int n = 0; n < NP; ++n) am[n] = 0.f, av[n] = 0.f;
#pragma unroll 5
            for (int k = 0; k < K; ++k) {
                const float xv = xp[koff[k]], x2 = xv * xv;
                const float4 *m4 = reinterpret_cast<const float4 *>(wm + k * NP), *v4 = reinterpret_cast<const float4 *>(wv + k * NP);
#pragma unroll
                for (int j = 0; j < NP / 4; ++j) {
                    const float4 a = m4[j], b = v4[j];
                    am[4 * j] = fmaf(xv, a.x, am[4 * j]), am[4 * j + 1] = fmaf(xv, a.y, am[4 * j + 1]);
                    am[4 * j + 2] = fmaf(xv, a.z, am[4 * j + 2]), am[4 * j + 3] = fmaf(xv, a.w, am[4 * j + 3]);
                    av[4 * j] = fmaf(x2, b.x, av[4 * j]), av[4 * j + 1] = fmaf(x2, b.y, av[4 * j + 1]);
                    av[4 * j + 2] = fmaf(x2, b.z, av[4 * j + 2]), av[4 * j + 3] = fmaf(x2, b.w, av[4 * j + 3]);
                }
            }
            const size_t o = (size_t)img * N * OH * OW + pix;
#pragma unroll
            for (int n = 0; n < NP; ++n) {
                if (n >= N) break;
                mean_out[o + (size_t)n * OH * OW] = am[n];
                sd_out[o + (size_t)n * OH * OW] = sqrtf(av[n] + bv[n]);
            }
        }
    }
}

template <int NP>
static int launch_conv_moments_direct(const float *x, const float *z, const float *Wm, const float *Wlv, const float *blv,
                                      float *mean_out, float *sd_out, long long n_imgs, int C, int H, int W, int ks, int N,
                                      cudaStream_t st) {
    const int K = C * ks * ks;
    const size_t smem = sizeof(float) * ((size_t)2 * K * NP + NP + ((K + 3) & ~3) + (size_t)C * H * W);
    if (smem > 48 * 1024)
        MNF_CUDA(cudaFuncSetAttribute(conv_moments_direct_kernel<NP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const DeviceProps *dp = device_props();
    MNF_REQUIRE(dp != nullptr, MNF_E_DEVICE, "no CUDA device");
    long long blocks = n_imgs < (long long)dp->sm_count * 8 ? n_imgs : (long long)dp->sm_count * 8;
    conv_moments_direct_kernel<NP><<<(unsigned)blocks, 256, smem, st>>>(x, z, Wm, Wlv, blv, mean_out, sd_out, n_imgs, C, H, W, ks, N);
    return launch_status("conv_moments_direct_kernel");
}

// Direct form of a grouped conv with few output channels per group (depthwise and its small channel multipliers):
// as a grouped GEMM a group is a tile of 64 columns with 1..8 useful ones.  A CTA owns one output channel c (grid
// dimension y) and a tile of output pixels (grid dimension x; with `pool`, of 2x2 windows) and walks the images
// r = blockIdx.z, blockIdx.z + gridDim.z, ...; it stages c's folded weights [cg * ks * ks] (W_mean * z, exp(W_log_var))
// in shared memory, and a thread walks the taps of its pixel over the cg input channels of c's group.  The sums run
// over the taps in the order of the implicit GEMM's K loop with the same operands, and the noise, moments and
// ReLU + pool epilogues are the GEMM's: the two kernels give the same bits for the same problem whenever the GEMM
// runs its tiled form (launch_simt_gemm's GEMV form for M <= 4, K >= 256 sums in another order).
struct ConvDirectArgs {
    const float *x;
    int x_imgs;  // image r reads x[r % x_imgs]
    int C, H, W, ks, OH, OW, pad, stride, dil, cg, ng, N;  // N = n_out, ng = n_out / groups, cg = c_in / groups
    const float *Wm, *Wlv, *blv, *z;  // z may be NULL (unit scale)
    float *out;
    float *sd_out;  // moments mode: out <- mean, sd_out <- sqrt(var), no noise
    NoiseSrc eps;   // indexed like the un-pooled output [R, N, OH, OW]
    int pool;
    long long R;
};

__global__ void __launch_bounds__(256) conv_grouped_direct_kernel(const ConvDirectArgs p) {
    extern __shared__ float sm_gd[];
    const int c = blockIdx.y, taps = p.cg * p.ks * p.ks;
    float *wm = sm_gd, *wv = sm_gd + taps;
    const float zc = p.z ? p.z[c] : 1.f;
    for (int t = threadIdx.x; t < taps; t += blockDim.x) {
        wm[t] = p.Wm[(size_t)c * taps + t] * zc;
        wv[t] = expf(p.Wlv[(size_t)c * taps + t]);
    }
    __syncthreads();
    const int H = p.H, W = p.W, ks = p.ks, dil = p.dil, OH = p.OH, OW = p.OW, N = p.N;
    const int PW = p.pool ? OW >> 1 : OW, PH = p.pool ? OH >> 1 : OH, sub = p.pool ? 4 : 1;
    const int pix = blockIdx.x * blockDim.x + threadIdx.x;
    if (pix >= PH * PW) return;
    const int px = pix % PW, py = pix / PW;
    const float bvar = expf(p.blv[c]);
    const size_t in_ch0 = (size_t)(c / p.ng) * p.cg;  // first input channel of c's group
    for (long long r = blockIdx.z; r < p.R; r += gridDim.z) {
        const float *xr = p.x + ((size_t)(r % p.x_imgs) * p.C + in_ch0) * H * W;
        float best = 0.f;  // ReLU floor
        for (int q = 0; q < sub; ++q) {
            const int oy = p.pool ? 2 * py + (q >> 1) : py, ox = p.pool ? 2 * px + (q & 1) : px;
            const int iy = oy * p.stride - p.pad, ix = ox * p.stride - p.pad;
            float am = 0.f, av = 0.f;
            const float *xc = xr;
            int t = 0;
            for (int ci = 0; ci < p.cg; ++ci, xc += (size_t)H * W) {
                for (int ky = 0; ky < ks; ++ky) {
                    const int y = iy + ky * dil;
                    const bool in_y = (unsigned)y < (unsigned)H;
                    for (int kx = 0; kx < ks; ++kx, ++t) {
                        const int xx = ix + kx * dil;
                        const float xv = in_y && (unsigned)xx < (unsigned)W ? xc[y * W + xx] : 0.f;
                        am = fmaf(xv, wm[t], am);
                        av = fmaf(xv * xv, wv[t], av);
                    }
                }
            }
            const long long e = ((r * N + c) * OH + oy) * OW + ox;
            if (p.sd_out) {
                p.out[e] = am;
                p.sd_out[e] = sqrtf(av + bvar);
                continue;
            }
            const long long ge = (((r + (long long)p.eps.row_offset) * N + c) * OH + oy) * OW + ox;
            const float v = am + sqrtf(av + bvar) * noise_normal(p.eps, e, ge);  // b_mean == 0
            if (p.pool)
                best = fmaxf(best, v);
            else
                p.out[e] = v;
        }
        if (p.pool) p.out[((r * N + c) * PH + py) * PW + px] = best;
    }
}

// the grouped direct kernel serves groups of at most this many output channels and this many taps (its weights stay
// in 32 KB of shared memory); wider groups run the grouped implicit GEMM.  On a B200, 64 -> 64 channels 3x3 on
// 256 x 32 x 32 images with 8 channels a group: 3.67 ms on the grouped GEMM, 1.43 ms on the direct kernel; with 16 a
// group the GEMM took 2.85 ms, about what the direct kernel's cost per channel predicts (profiles/r10_mnf_conv_groups.md).
constexpr int kDirectMaxNg = 8, kDirectMaxTaps = 4096;

// the conv of mnf_conv2d_forward_geom / mnf_conv2d_moments_geom: the implicit GEMM (tap offsets and, with GEOM, the
// dilated tap coordinates tabulated on the host), or for groups > 1 with few channels per group the direct kernel.
// sd_out != NULL: moments mode.
template <bool GEOM>
static int run_conv_gemm(const float *x, int x_imgs, const float *z, const float *Wm, const float *Wlv, const float *blv,
                         float *out, float *sd_out, NoiseSrc eps, int pool, long long M, int C, int H, int W, int ks,
                         int N, int OH, int OW, int pad, int stride, int dil, int groups, cudaStream_t st,
                         const char *what) {
    const int cg = C / groups, ng = N / groups, taps = cg * ks * ks;
    if (GEOM && groups > 1 && ng <= kDirectMaxNg && taps <= kDirectMaxTaps && N <= 65535) {
        const long long R = M / ((long long)OH * OW);
        if (R == 0) return 0;
        const int P = pool ? (OH / 2) * (OW / 2) : OH * OW;  // work items of one image and channel
        const int threads = P < 256 ? (P + 31) & ~31 : 256;
        const dim3 grid((unsigned)((P + threads - 1) / threads), (unsigned)N, (unsigned)(R < 65535 ? R : 65535));
        const ConvDirectArgs a{x, x_imgs, C, H, W, ks, OH, OW, pad, stride, dil, cg, ng, N, Wm, Wlv, blv, z, out, sd_out,
                               eps, pool, R};
        conv_grouped_direct_kernel<<<grid, threads, 2 * sizeof(float) * taps, st>>>(a);
        return launch_status("conv_grouped_direct_kernel");
    }
    MnfConvProb<GEOM> p{(int)M, ng, taps, x, x_imgs, C, H, W, ks, OH, OW, Wm, Wlv, blv, z, out, eps, pool, sd_out,
                        {}, pad, stride, {}, dil, cg};
    for (int k = 0; k < p.K && k < MnfConvProb<GEOM>::kMaxTaps; ++k) {
        const int kx = (k % ks) * dil, ky = ((k / ks) % ks) * dil, ci = k / (ks * ks);
        p.koff[k] = (ci * H + ky) * W + kx;
        if constexpr (GEOM) p.kyx[k] = (ky << 16) | kx;
    }
    return launch_simt_gemm<MnfConvProb<GEOM>, 2>(p, st, what, groups);
}

int conv_pack_weights_f16(const float *z, const float *W_mean, const float *W_log_var, const float *b_log_var, void *Bm,
                          void *Bv, float *bvar_p, int K, int c_out, int Np, int Kp, void *stream) {
    MNF_REQUIRE(W_mean && W_log_var && b_log_var && Bm && Bv && bvar_p, MNF_E_ARG, "NULL pointer");
    conv_pack_weights_f16_kernel<<<64, 256, 0, (cudaStream_t)stream>>>(W_mean, W_log_var, b_log_var, z, c_out, K, Np, Kp,
                                                                     (__half *)Bm, (__half *)Bv, bvar_p);
    return launch_status("conv_pack_weights_kernel");
}

}  // namespace mnf

using namespace mnf;

extern "C" {

// mean = conv2d(x, W_mean * z), sd = sqrt(conv2d(x^2, exp(W_log_var)) + exp(b_log_var)) without noise
// ([n_imgs, c_out, OH, OW] each): the sample-independent part of MNFConv2d.forward (mnf_conv.py:69-75).
int mnf_conv2d_moments(const float *x, const float *z, const float *W_mean, const float *W_log_var,
                       const float *b_log_var, float *mean_out, float *sd_out, int64_t n_imgs, int c_in, int height,
                       int width, int c_out, int ksize, void *stream) {
    return mnf_conv2d_moments_ps(x, z, W_mean, W_log_var, b_log_var, mean_out, sd_out, n_imgs, c_in, height, width, c_out,
                                 ksize, 0, 1, stream);
}

int mnf_conv2d_moments_ps(const float *x, const float *z, const float *W_mean, const float *W_log_var,
                          const float *b_log_var, float *mean_out, float *sd_out, int64_t n_imgs, int c_in, int height,
                          int width, int c_out, int ksize, int pad, int stride, void *stream) {
    return mnf_conv2d_moments_geom(x, z, W_mean, W_log_var, b_log_var, mean_out, sd_out, n_imgs, c_in, height, width,
                                   c_out, ksize, pad, stride, 1, 1, stream);
}

// checks shared by the _geom entry points: dilation, groups and the size of the tap table entries
#define MNF_CHECK_DIL_GROUPS(c_in, c_out, ksize, dilation, groups)                                                        \
    MNF_REQUIRE(dilation >= 1 && (long long)dilation * ((ksize) - 1) <= 0x7fff, MNF_E_ARG, "bad dilation %d", dilation); \
    MNF_REQUIRE(groups >= 1 && groups <= 65535 && (c_in) % groups == 0 && (c_out) % groups == 0, MNF_E_ARG,             \
                "groups %d must divide c_in %d and c_out %d", groups, c_in, c_out)

// the same with zero padding `pad`, stride `stride`, dilation and channel groups (OH = (H + 2 pad - dil (k-1) - 1) /
// stride + 1).  Only the default geometry takes the direct moments kernel; groups > 1 with few channels per group take
// the grouped direct kernel, every other geometry runs the implicit GEMM with bounds-tested tap loads.
int mnf_conv2d_moments_geom(const float *x, const float *z, const float *W_mean, const float *W_log_var,
                            const float *b_log_var, float *mean_out, float *sd_out, int64_t n_imgs, int c_in, int height,
                            int width, int c_out, int ksize, int pad, int stride, int dilation, int groups,
                            void *stream) {
    MNF_REQUIRE(x && W_mean && W_log_var && b_log_var && mean_out && sd_out, MNF_E_ARG, "NULL pointer");  // z may be NULL (= 1)
    MNF_REQUIRE(pad >= 0 && pad <= 0xffff && stride >= 1, MNF_E_ARG, "bad padding %d or stride %d", pad, stride);
    MNF_CHECK_DIL_GROUPS(c_in, c_out, ksize, dilation, groups);
    const int OH = conv_out_size(height, ksize, pad, stride, dilation), OW = conv_out_size(width, ksize, pad, stride, dilation);
    MNF_REQUIRE(n_imgs >= 0 && OH >= 1 && OW >= 1, MNF_E_SHAPE, "bad shape");
    const long long M = (long long)n_imgs * OH * OW;
    MNF_REQUIRE(M <= 0x7fffffff - 64, MNF_E_SHAPE, "too many output pixels for one call (%lld)", M);
    if (n_imgs == 0) return 0;
    const bool geom = pad != 0 || stride != 1 || dilation != 1 || groups != 1;
    if (!geom && c_in * ksize * ksize <= 64 && c_out <= 32 && c_in * height * width <= 4096) {  // few taps, few channels: direct form
        if (c_out <= 20)
            return launch_conv_moments_direct<20>(x, z, W_mean, W_log_var, b_log_var, mean_out, sd_out, n_imgs, c_in, height,
                                                  width, ksize, c_out, (cudaStream_t)stream);
        return launch_conv_moments_direct<32>(x, z, W_mean, W_log_var, b_log_var, mean_out, sd_out, n_imgs, c_in, height, width,
                                              ksize, c_out, (cudaStream_t)stream);
    }
    const NoiseSrc none{nullptr, 0, 0, 0};
    const int x_imgs = (int)(n_imgs > 0 ? n_imgs : 1);
    if (geom)
        return run_conv_gemm<true>(x, x_imgs, z, W_mean, W_log_var, b_log_var, mean_out, sd_out, none, 0, M, c_in, height,
                                   width, ksize, c_out, OH, OW, pad, stride, dilation, groups, (cudaStream_t)stream,
                                   "mnf_conv2d_moments");
    return run_conv_gemm<false>(x, x_imgs, z, W_mean, W_log_var, b_log_var, mean_out, sd_out, none, 0, M, c_in, height,
                                width, ksize, c_out, OH, OW, 0, 1, 1, 1, (cudaStream_t)stream, "mnf_conv2d_moments");
}

// out[r] = maxpool2(relu(mean[r % n_unique] + sd[r % n_unique] * eps[r])) -- the per-sample tail of an MNFConv2d
// under Monte-Carlo replication.  eps: [n_rows, c, OH, OW] or NULL (Philox, same element numbering).
int mnf_conv_noise_relu_pool(const float *mean, const float *sd, int64_t n_unique, const float *eps, uint64_t seed,
                             uint32_t noise_stream, uint64_t row_offset, float *out, int64_t n_rows, int channels,
                             int out_h, int out_w, void *stream) {
    return mnf_conv_noise_relu_pool_z(mean, sd, n_unique, eps, seed, noise_stream, row_offset, out, n_rows, channels, out_h,
                                      out_w, nullptr, 1, stream);
}

int mnf_conv_noise_relu_pool_z(const float *mean, const float *sd, int64_t n_unique, const float *eps, uint64_t seed,
                               uint32_t noise_stream, uint64_t row_offset, float *out, int64_t n_rows, int channels,
                               int out_h, int out_w, const float *z_rows, int64_t rows_per_z, void *stream) {
    MNF_REQUIRE(mean && sd && out, MNF_E_ARG, "NULL pointer");
    MNF_REQUIRE(rows_per_z >= 1, MNF_E_ARG, "rows_per_z must be positive");
    MNF_REQUIRE(n_rows >= 0 && n_unique >= 1 && out_h % 2 == 0 && out_w % 4 == 0, MNF_E_SHAPE,
                "conv output %dx%d: height must be even and width a multiple of 4", out_h, out_w);
    MNF_REQUIRE(((uintptr_t)mean % 16) == 0 && ((uintptr_t)sd % 16) == 0 && (!eps || ((uintptr_t)eps % 16) == 0) &&
                    ((uintptr_t)out % 8) == 0 && ((row_offset * channels * out_h * out_w) % 4) == 0,
                MNF_E_ALIGN, "pointers must be 16-byte aligned");
    if (n_rows == 0) return 0;
    const long long total = (long long)n_rows * channels * (out_h / 2) * (out_w / 4);
    long long blocks = (total + 255) / 256;
    if (blocks > 148 * 32) blocks = 148 * 32;
    PoolDivs dv;
    dv.pw2 = FastDiv((uint32_t)(out_w / 4)), dv.ph = FastDiv((uint32_t)(out_h / 2)), dv.c = FastDiv((uint32_t)channels);
    const NoiseSrc src{eps, seed, noise_stream, row_offset};
    if (total < 0x7fffffffLL)
        conv_noise_pool_kernel<true><<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
            mean, sd, (int)n_unique, src, out, n_rows, channels, out_h, out_w, z_rows, rows_per_z, dv);
    else
        conv_noise_pool_kernel<false><<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
            mean, sd, (int)n_unique, src, out, n_rows, channels, out_h, out_w, z_rows, rows_per_z, dv);
    return launch_status("conv_noise_pool_kernel");
}

// staging for mnf_conv2d_forward_tc (tc_gemm.cu): im2col of x and x^2 (pool-major rows) and packed weights
int mnf_conv_tc_stage(const float *x, const float *z, const float *W_mean, const float *W_log_var,
                      const float *b_log_var, float *a_mean, float *a_var, float *Bm, float *Bv, float *bvar_p,
                      int64_t n_imgs, int c_in, int height, int width, int c_out, int ksize, int Np, int Kp,
                      void *stream) {
    MNF_REQUIRE(x && W_mean && W_log_var && b_log_var && Bm && Bv && bvar_p, MNF_E_ARG, "NULL pointer");
    MNF_REQUIRE((a_mean == nullptr) == (a_var == nullptr), MNF_E_ARG, "a_mean and a_var must both be given or both be NULL");
    const int OH = height - ksize + 1, OW = width - ksize + 1, K = c_in * ksize * ksize;
    MNF_REQUIRE(OH >= 2 && OW >= 2 && OH % 2 == 0 && OW % 2 == 0 && Kp % 4 == 0 && Kp >= K && Np >= c_out, MNF_E_SHAPE,
                "bad shape");
    cudaStream_t st = (cudaStream_t)stream;
    conv_pack_weights_kernel<<<64, 256, 0, st>>>(W_mean, W_log_var, b_log_var, z, c_out, K, Np, Kp, Bm, Bv, bvar_p);
    if (a_mean == nullptr) return launch_status("conv_pack_weights_kernel");  // weights only (implicit-GEMM conv)
    const size_t smem = sizeof(float) * ((size_t)c_in * height * width + Kp);
    MNF_REQUIRE(smem <= 200 * 1024, MNF_E_SHAPE, "image of %d x %d x %d floats does not fit shared memory", c_in, height, width);
    if (smem > 48 * 1024)
        MNF_CUDA(cudaFuncSetAttribute(conv_im2col_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    long long blocks = n_imgs < 148 * 8 ? n_imgs : 148 * 8;
    if (blocks < 1) blocks = 1;
    conv_im2col_kernel<<<(unsigned)blocks, 256, smem, st>>>(x, a_mean, a_var, n_imgs, c_in, height, width, ksize, OH, OW, Kp);
    return launch_status("conv tc staging");
}

int mnf_sample_z0(const float *q0_mean, const float *q0_log_var, const float *eps, uint64_t seed,
                  uint32_t noise_stream, uint64_t row_offset, float *z, int64_t n_rows, int dim, void *stream) {
    MNF_REQUIRE(q0_mean && q0_log_var && z, MNF_E_ARG, "NULL pointer");
    MNF_REQUIRE(n_rows >= 0 && dim >= 1, MNF_E_ARG, "bad shape");
    if (n_rows == 0) return 0;
    const long long total = (long long)n_rows * dim;
    long long blocks = (total / 4 + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    if (blocks < 1) blocks = 1;
    sample_z0_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
        q0_mean, q0_log_var, NoiseSrc{eps, seed, noise_stream, row_offset}, z, n_rows, dim);
    return launch_status("sample_z0_kernel");
}

int mnf_rnvp_forward(const mnf_rnvp_flow *flows_host, int n_flows, float *z, float *log_det,
                     const float *const *masks_host, uint64_t seed, uint32_t first_noise_stream,
                     uint64_t row_offset, int64_t n_rows, int dim, float *workspace, float *intermediates,
                     void *stream) {
    MNF_REQUIRE(flows_host && z && log_det && workspace, MNF_E_ARG, "NULL pointer");
    MNF_REQUIRE(n_flows >= 0 && n_rows >= 0 && dim >= 1, MNF_E_ARG, "bad shape");
    MNF_REQUIRE(n_rows <= 0x7fffffff / 64, MNF_E_SHAPE, "too many rows for one call (%lld)", (long long)n_rows);
    cudaStream_t st = (cudaStream_t)stream;
    if (n_rows == 0) return 0;
    MNF_CUDA(cudaMemsetAsync(log_det, 0, sizeof(float) * n_rows, st));
    for (int f = 0; f < n_flows; ++f) {
        const mnf_rnvp_flow &fl = flows_host[f];
        MNF_REQUIRE(fl.n_net >= 1 && fl.n_net <= MNF_RNVP_MAX_NET, MNF_E_SHAPE, "flow %d: n_net=%d", f, fl.n_net);
        const NoiseSrc mask{masks_host ? masks_host[f] : nullptr, seed, first_noise_stream + (uint32_t)f, row_offset};
        // conditioner net (MLP(dim, *h_sizes), last activation dropped -- mlp.py:12)
        int maxh = 1;
        for (int g = 0; g < n_flows; ++g)
            for (int l = 0; l < flows_host[g].n_net && l < MNF_RNVP_MAX_NET; ++l)
                maxh = flows_host[g].net_sizes[l] > maxh ? flows_host[g].net_sizes[l] : maxh;
        float *ya = workspace, *yb = workspace + (size_t)n_rows * maxh;
        if (n_rows == 1 && fl.n_net == 1 && fl.net_sizes[0] <= 64 && dim <= 11000) {  // single-row cluster kernel
            float *inter_f = intermediates ? intermediates + (size_t)f * dim : nullptr;
            rnvp_row_kernel<<<kRowCluster, 256, sizeof(float) * (dim + 64 + 8), st>>>(
                fl.net_w[0], fl.net_b[0], fl.net_sizes[0], fl.t_w, fl.t_b, fl.s_w, fl.s_b, z, log_det, mask, dim, ya, inter_f);
            int rcr = launch_status("rnvp_row_kernel");
            if (rcr) return rcr;
            continue;
        }
        RnvpHiddenProb hp{(int)n_rows, fl.net_sizes[0], dim, z, fl.net_w[0], fl.net_b[0], ya, mask, fl.n_net > 1};
        int rc = launch_simt_gemm<RnvpHiddenProb, 1>(hp, st, "rnvp_hidden");
        if (rc) return rc;
        for (int l = 1; l < fl.n_net; ++l) {
            LinearProb lp{(int)n_rows, fl.net_sizes[l], fl.net_sizes[l - 1], ya, fl.net_w[l], fl.net_b[l], yb,
                          l + 1 < fl.n_net};
            rc = launch_simt_gemm<LinearProb, 1>(lp, st, "rnvp_net_layer");
            if (rc) return rc;
            float *t = ya;
            ya = yb;
            yb = t;
        }
        RnvpOutProb op{(int)n_rows, dim, fl.net_sizes[fl.n_net - 1], ya, fl.t_w, fl.t_b, fl.s_w, fl.s_b, z, log_det, mask};
        rc = launch_simt_gemm<RnvpOutProb, 2>(op, st, "rnvp_out");
        if (rc) return rc;
        if (intermediates)
            MNF_CUDA(cudaMemcpyAsync(intermediates + (size_t)f * n_rows * dim, z, sizeof(float) * n_rows * dim,
                                     cudaMemcpyDeviceToDevice, st));
    }
    return 0;
}

int mnf_linear_forward(const float *x, int64_t x_rows, const float *z, const float *W_mean, const float *W_log_var,
                       const float *b_mean, const float *b_log_var, const float *eps, uint64_t seed,
                       uint32_t noise_stream, uint64_t row_offset, float *out, int64_t n_rows, int n_in, int n_out,
                       int relu, void *stream) {
    return mnf_linear_forward_affine(x, x_rows, z, W_mean, W_log_var, b_mean, b_log_var, eps, seed, noise_stream,
                                     row_offset, out, n_rows, n_in, n_out, relu, nullptr, nullptr, stream);
}

int mnf_linear_forward_affine(const float *x, int64_t x_rows, const float *z, const float *W_mean,
                              const float *W_log_var, const float *b_mean, const float *b_log_var, const float *eps,
                              uint64_t seed, uint32_t noise_stream, uint64_t row_offset, float *out, int64_t n_rows,
                              int n_in, int n_out, int relu, const float *col_scale, const float *col_shift,
                              void *stream) {
    MNF_REQUIRE(x && z && W_mean && W_log_var && b_mean && b_log_var && out, MNF_E_ARG, "NULL pointer");
    MNF_REQUIRE((col_scale == nullptr) == (col_shift == nullptr), MNF_E_ARG,
                "col_scale and col_shift must both be given or both be NULL");
    MNF_REQUIRE(n_rows >= 0 && n_in >= 1 && n_out >= 1 && x_rows >= 1, MNF_E_ARG, "bad shape");
    MNF_REQUIRE(n_rows <= 0x7fffffff / 64, MNF_E_SHAPE, "too many rows for one call (%lld)", (long long)n_rows);
    MnfLinearProb p{(int)n_rows, n_out, n_in, x, (int)x_rows, z, W_mean, W_log_var, b_mean, b_log_var, out,
                    NoiseSrc{eps, seed, noise_stream, row_offset}, relu, col_scale, col_shift};
    return launch_simt_gemm<MnfLinearProb, 2>(p, (cudaStream_t)stream, "mnf_linear_forward");
}

int mnf_conv2d_forward(const float *x, int64_t x_imgs, const float *z, const float *W_mean, const float *W_log_var,
                       const float *b_log_var, const float *eps, uint64_t seed, uint32_t noise_stream,
                       uint64_t row_offset, float *out, int64_t n_imgs, int c_in, int height, int width, int c_out,
                       int ksize, int relu_pool, void *stream) {
    return mnf_conv2d_forward_ps(x, x_imgs, z, W_mean, W_log_var, b_log_var, eps, seed, noise_stream, row_offset, out,
                                 n_imgs, c_in, height, width, c_out, ksize, relu_pool, 0, 1, stream);
}

int mnf_conv2d_forward_ps(const float *x, int64_t x_imgs, const float *z, const float *W_mean, const float *W_log_var,
                          const float *b_log_var, const float *eps, uint64_t seed, uint32_t noise_stream,
                          uint64_t row_offset, float *out, int64_t n_imgs, int c_in, int height, int width, int c_out,
                          int ksize, int relu_pool, int pad, int stride, void *stream) {
    return mnf_conv2d_forward_geom(x, x_imgs, z, W_mean, W_log_var, b_log_var, eps, seed, noise_stream, row_offset, out,
                                   n_imgs, c_in, height, width, c_out, ksize, relu_pool, pad, stride, 1, 1, stream);
}

int mnf_conv2d_forward_geom(const float *x, int64_t x_imgs, const float *z, const float *W_mean,
                            const float *W_log_var, const float *b_log_var, const float *eps, uint64_t seed,
                            uint32_t noise_stream, uint64_t row_offset, float *out, int64_t n_imgs, int c_in, int height,
                            int width, int c_out, int ksize, int relu_pool, int pad, int stride, int dilation, int groups,
                            void *stream) {
    MNF_REQUIRE(x && z && W_mean && W_log_var && b_log_var && out, MNF_E_ARG, "NULL pointer");
    MNF_REQUIRE(n_imgs >= 0 && c_in >= 1 && c_out >= 1 && ksize >= 1 && x_imgs >= 1, MNF_E_ARG, "bad shape");
    MNF_REQUIRE(pad >= 0 && pad <= 0xffff && stride >= 1, MNF_E_ARG, "bad padding %d or stride %d", pad, stride);
    MNF_CHECK_DIL_GROUPS(c_in, c_out, ksize, dilation, groups);
    const int OH = conv_out_size(height, ksize, pad, stride, dilation), OW = conv_out_size(width, ksize, pad, stride, dilation);
    MNF_REQUIRE(OH >= 1 && OW >= 1, MNF_E_SHAPE, "kernel %d at dilation %d larger than input %dx%d padded by %d", ksize,
                dilation, height, width, pad);
    MNF_REQUIRE(!relu_pool || (OH % 2 == 0 && OW % 2 == 0), MNF_E_SHAPE,
                "fused 2x2 max-pool needs even output size, got %dx%d", OH, OW);
    const long long M = (long long)n_imgs * OH * OW;
    MNF_REQUIRE(M <= 0x7fffffff - 64, MNF_E_SHAPE, "too many output pixels for one call (%lld): chunk the batch", M);
    const NoiseSrc src{eps, seed, noise_stream, row_offset};
    if (pad != 0 || stride != 1 || dilation != 1 || groups != 1)
        return run_conv_gemm<true>(x, (int)x_imgs, z, W_mean, W_log_var, b_log_var, out, nullptr, src, relu_pool, M, c_in,
                                   height, width, ksize, c_out, OH, OW, pad, stride, dilation, groups, (cudaStream_t)stream,
                                   "mnf_conv2d_forward");
    return run_conv_gemm<false>(x, (int)x_imgs, z, W_mean, W_log_var, b_log_var, out, nullptr, src, relu_pool, M, c_in,
                                height, width, ksize, c_out, OH, OW, 0, 1, 1, 1, (cudaStream_t)stream,
                                "mnf_conv2d_forward");
}

}  // extern "C"
