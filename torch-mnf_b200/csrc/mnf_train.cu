// mnf_train.cu -- device primitives of the MNF layers' TRAINING path (SURVEY.md section 8f-1: the reference trains
// MNFLinear / kl_div through torch autograd, tests/test_mnf_mnist.py:28-43; these are the forward-with-saved-state and
// backward kernels the drop-in modules' autograd Functions call).  Exact fp32 throughout -- training batches are
// small (32 rows in the reference's test) and gradients should not carry TF32 rounding:
//   mnf_gemm_f32            C = op(A) op(B) + bias + beta C, any transposition / leading dimensions (dgrad, wgrad);
//                           mnf_gemm_f32_batched: a batch of such products at fixed strides in one launch
//   mnf_ew                  fused elementwise stages of the layer forward / backward
//   mnf_colsum              bias-style reductions over rows
//   mnf_rnvp_gate_*         the RNVP update z' = (1-m) z gate + (1-gate) shift + m z and its adjoint (rnvp.py:26-40)
//   mnf_kl_rows_*           the weight-sized part of MNFLinear.kl_div (mnf_linear.py:67-79) and its adjoint
#include "common.cuh"

namespace mnf {

// ---------------------------------------------------------------------------------------------------------------
// generic fp32 GEMM: 64 x 64 tile, 16-deep slices, 256 threads x (4 x 4) accumulators.  Grid dimension z walks a
// batch of products whose operands lie sA / sB / sC floats apart (the groups of a grouped convolution).
// ---------------------------------------------------------------------------------------------------------------
template <bool TA, bool TB>
__global__ void __launch_bounds__(256)
gemm_f32_kernel(long long M, int N, int K, const float *__restrict__ A, long long lda, const float *__restrict__ B,
                long long ldb, const float *__restrict__ bias, float beta, float *__restrict__ C, long long ldc,
                long long sA, long long sB, long long sC) {
    __shared__ float As[16][64 + 4], Bs[16][64 + 4];
    A += blockIdx.z * sA, B += blockIdx.z * sB, C += blockIdx.z * sC;
    const int tid = threadIdx.x, tx = tid % 16, ty = tid / 16;
    const long long m0 = (long long)blockIdx.y * 64;
    const int n0 = blockIdx.x * 64;
    float acc[4][4] = {};
    for (int k0 = 0; k0 < K; k0 += 16) {
#pragma unroll
        for (int e = tid; e < 1024; e += 256) {
            int m, k;
            if (TA) k = e / 64, m = e % 64;  // stored [K, M]: consecutive threads walk m
            else m = e / 16, k = e % 16;     // stored [M, K]: consecutive threads walk k
            const bool ok = m0 + m < M && k0 + k < K;
            As[k][m] = ok ? (TA ? A[(long long)(k0 + k) * lda + m0 + m] : A[(m0 + m) * lda + k0 + k]) : 0.f;
            int n, kb;
            if (TB) n = e / 16, kb = e % 16;  // stored [N, K]
            else kb = e / 64, n = e % 64;     // stored [K, N]
            const bool okb = n0 + n < N && k0 + kb < K;
            Bs[kb][n] = okb ? (TB ? B[(long long)(n0 + n) * ldb + k0 + kb] : B[(long long)(k0 + kb) * ldb + n0 + n]) : 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < 16; ++k) {
            float a[4], b[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) a[i] = As[k][ty * 4 + i], b[i] = Bs[k][tx * 4 + i];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const long long m = m0 + ty * 4 + i;
        if (m >= M) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int n = n0 + tx * 4 + j;
            if (n >= N) continue;
            float v = acc[i][j] + (bias ? bias[n] : 0.f);
            if (beta != 0.f) v = fmaf(beta, C[m * ldc + n], v);
            C[m * ldc + n] = v;
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------
// elementwise stages.  "v" operands are [ncols] vectors broadcast over rows (index i % ncols).
// ---------------------------------------------------------------------------------------------------------------
__global__ void ew_kernel(int op, const float *__restrict__ a, const float *__restrict__ b, const float *__restrict__ c,
                          const float *__restrict__ d, float *__restrict__ out, float *__restrict__ out2, long long n,
                          int ncols) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const int col = (int)(i % ncols);
        switch (op) {
            case MNF_EW_MUL: out[i] = a[i] * b[i]; break;
            case MNF_EW_MUL_ROWVEC: out[i] = a[i] * b[col]; break;
            case MNF_EW_FMA: out[i] = fmaf(b[i], c[i], a[i]); break;
            case MNF_EW_SQUARE: out[i] = a[i] * a[i]; break;
            case MNF_EW_EXP: out[i] = expf(a[i]); break;
            case MNF_EW_LEAKY: out[i] = fmaxf(a[i], 0.2f * a[i]); break;
            case MNF_EW_LEAKY_BWD: out[i] = a[i] * (b[i] > 0.f ? 1.f : 0.2f); break;  // a = grad, b = pre-activation
            case MNF_EW_NOISE_OUT: out[i] = fmaf(sqrtf(b[i]), c[i], a[i]); break;     // mean + sqrt(var) eps
            case MNF_EW_GVAR: out[i] = a[i] * c[i] * 0.5f / sqrtf(b[i]); break;        // g eps / (2 sqrt(var))
            case MNF_EW_LIN_IN_BWD:  // a = d/d(xz), b = d/d(x^2), c = z, d = x
                out[i] = fmaf(a[i], c[i], 2.f * d[i] * b[i]);
                out2[i] = a[i] * d[i];
                break;
            case MNF_EW_Z0: out[i] = fmaf(expf(0.5f * b[col]), c[i], a[col]); break;  // q0_mean + std eps
            case MNF_EW_MUL_COLVEC: out[i] = a[i] * b[i / ncols]; break;              // per-row scale (W_mean * z[c_out])
            case MNF_EW_ADD_2MUL: out[i] = fmaf(2.f * b[i], c[i], a[i]); break;       // a + 2 b c
            case MNF_EW_ADD_COLVEC: out[i] = a[i] + b[i / ncols]; break;              // per-row bias
            case MNF_EW_RELU: out[i] = fmaxf(a[i], 0.f); break;                       // nn.ReLU between MaskedLinears
            case MNF_EW_RELU_BWD: out[i] = b[i] > 0.f ? a[i] : 0.f; break;            // a = grad, b = pre-activation
            default: break;
        }
    }
}

// out[n] = sum_r a[r, n] * (b ? b[r, n] : 1); out must be zeroed (atomics across row chunks)
__global__ void colsum_kernel(const float *__restrict__ a, const float *__restrict__ b, long long R, int N,
                              float *__restrict__ out) {
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    const long long chunk = (R + gridDim.y - 1) / gridDim.y, r0 = blockIdx.y * chunk;
    const long long r1 = r0 + chunk < R ? r0 + chunk : R;
    float s = 0.f;
    for (long long r = r0; r < r1; ++r) s += b ? a[r * N + n] * b[r * N + n] : a[r * N + n];
    if (r1 > r0) atomicAdd(&out[n], s);
}

// ---------------------------------------------------------------------------------------------------------------
// RNVP update (rnvp.py:26-40): gate = sigmoid(scale); z' = (1-m) z gate + (1-gate) shift + m z;
// log_det = sum_cols (1-m) log(gate).  One warp per row.
// ---------------------------------------------------------------------------------------------------------------
__global__ void rnvp_gate_fwd_kernel(const float *__restrict__ z, const float *__restrict__ m,
                                     const float *__restrict__ shift, const float *__restrict__ scale,
                                     float *__restrict__ z_out, float *__restrict__ ld, long long R, int n) {
    const long long row = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (row >= R) return;
    float acc = 0.f;
    for (int c = lane; c < n; c += 32) {
        const long long i = row * n + c;
        const float gate = 1.f / (1.f + expf(-scale[i])), mk = m[i];
        z_out[i] = (1.f - mk) * z[i] * gate + (1.f - gate) * shift[i] + mk * z[i];
        acc += (1.f - mk) * logf(gate);
    }
    acc = warp_sum(acc);
    if (lane == 0) ld[row] = acc;
}

__global__ void rnvp_gate_bwd_kernel(const float *__restrict__ z, const float *__restrict__ m,
                                     const float *__restrict__ shift, const float *__restrict__ scale,
                                     const float *__restrict__ g_out, const float *__restrict__ g_ld,
                                     float *__restrict__ g_shift, float *__restrict__ g_scale, float *__restrict__ g_z,
                                     long long total, int n) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
         i += (long long)gridDim.x * blockDim.x) {
        const float gate = 1.f / (1.f + expf(-scale[i])), mk = m[i], go = g_out ? g_out[i] : 0.f;
        const float gl = g_ld ? g_ld[i / n] : 0.f;
        const float g_gate = go * ((1.f - mk) * z[i] - shift[i]) + gl * (1.f - mk) / gate;
        g_shift[i] = go * (1.f - gate);
        g_scale[i] = g_gate * gate * (1.f - gate);
        g_z[i] = go * ((1.f - mk) * gate + mk);
    }
}

// ---------------------------------------------------------------------------------------------------------------
// weight-sized part of MNFLinear.kl_div (mnf_linear.py:67-79), one warp per output row j:
//   pre[j]   = sum_i (W_mean[j,i] z_i + exp(W_log_var[j,i] / 2) eps[j,i]) c_i          (argument of the tanh)
//   klrow[j] = 0.5 sum_i (-W_log_var + exp(W_log_var) + (W_mean z)^2 - 1)
// ---------------------------------------------------------------------------------------------------------------
__global__ void kl_rows_fwd_kernel(const float *__restrict__ z, const float *__restrict__ Wm,
                                   const float *__restrict__ Wlv, const float *__restrict__ c,
                                   const float *__restrict__ eps, float *__restrict__ pre, float *__restrict__ klrow,
                                   int n_out, int n_in) {
    const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (row >= n_out) return;
    float p = 0.f, k = 0.f;
    for (int i = lane; i < n_in; i += 32) {
        const long long e = (long long)row * n_in + i;
        const float wm = Wm[e] * z[i], lv = Wlv[e];
        p = fmaf(wm + expf(0.5f * lv) * eps[e], c[i], p);
        k += -lv + expf(lv) + wm * wm - 1.f;
    }
    p = warp_sum(p), k = warp_sum(k);
    if (lane == 0) pre[row] = p, klrow[row] = 0.5f * k;
}

// adjoint: thread per column i, blocks over row chunks; gz / gc reduced with atomics (zeroed by the caller)
__global__ void kl_rows_bwd_kernel(const float *__restrict__ z, const float *__restrict__ Wm,
                                   const float *__restrict__ Wlv, const float *__restrict__ c,
                                   const float *__restrict__ eps, const float *__restrict__ g_pre,
                                   const float *__restrict__ g_kl, float *__restrict__ gWm, float *__restrict__ gWlv,
                                   float *__restrict__ gz, float *__restrict__ gc, int n_out, int n_in) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_in) return;
    const int chunk = (n_out + gridDim.y - 1) / gridDim.y, j0 = blockIdx.y * chunk;
    const int j1 = j0 + chunk < n_out ? j0 + chunk : n_out;
    const float zi = z[i], ci = c[i];
    float az = 0.f, ac = 0.f;
    for (int j = j0; j < j1; ++j) {
        const long long e = (long long)j * n_in + i;
        const float w = Wm[e], lv = Wlv[e], sd = expf(0.5f * lv), ep = eps[e];
        const float gp = g_pre[j], gk = g_kl[j];
        const float g_wm = gk * w * zi + gp * ci;  // d / d(W_mean z)
        gWm[e] = g_wm * zi;
        gWlv[e] = gk * 0.5f * (expf(lv) - 1.f) + gp * ci * 0.5f * sd * ep;
        az = fmaf(g_wm, w, az);
        ac = fmaf(gp, fmaf(w, zi, sd * ep), ac);
    }
    if (j1 > j0) atomicAdd(&gz[i], az), atomicAdd(&gc[i], ac);
}

// ---------------------------------------------------------------------------------------------------------------
// convolution as GEMM with zero padding `pad`, stride `st` and dilation `dl`: transposed im2col
// colsT[(ci,kh,kw)][(r,oh,ow)] = x[r, ci, oh*st - pad + kh*dl, ow*st - pad + kw*dl] (0 in the padding), its adjoint
// (gather form, no atomics), and the [A,B,inner] -> [B,A,inner] layout swap between the GEMM's [c_out, R*OH*OW] and
// the module's [R, c_out, OH, OW].  With pad 0, stride 1 and dilation 1 every bounds test passes and the adjoint sums
// the same terms in the same order as the unpadded form.  Channel groups need nothing here: group g's rows of colsT
// are the contiguous block of its input channels.
// ---------------------------------------------------------------------------------------------------------------
__global__ void im2col_t_kernel(const float *__restrict__ x, float *__restrict__ colsT, long long R, int c_in, int H,
                                int W, int ks, int pad, int st, int dl) {
    const int OH = conv_out_size(H, ks, pad, st, dl), OW = conv_out_size(W, ks, pad, st, dl);
    const long long P = R * OH * OW, total = (long long)c_in * ks * ks * P;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long p = i % P;
        const int f = (int)(i / P), kw = f % ks, kh = (f / ks) % ks, ci = f / (ks * ks);
        const int ow = (int)(p % OW), oh = (int)((p / OW) % OH);
        const long long r = p / ((long long)OW * OH);
        const int ih = oh * st - pad + kh * dl, iw = ow * st - pad + kw * dl;
        colsT[i] = ((unsigned)ih < (unsigned)H && (unsigned)iw < (unsigned)W) ? x[((r * c_in + ci) * H + ih) * W + iw] : 0.f;
    }
}

__global__ void col2im_t_kernel(const float *__restrict__ g_colsT, float *__restrict__ gx, long long R, int c_in, int H,
                                int W, int ks, int pad, int st, int dl) {
    const int OH = conv_out_size(H, ks, pad, st, dl), OW = conv_out_size(W, ks, pad, st, dl);
    const long long P = R * OH * OW, total = R * c_in * H * W;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int w = (int)(i % W), h = (int)((i / W) % H), ci = (int)((i / ((long long)W * H)) % c_in);
        const long long r = i / ((long long)W * H * c_in);
        float acc = 0.f;
        for (int kh = 0; kh < ks; ++kh) {
            const int th = h + pad - kh * dl;  // oh * st when input row h is tap row kh of output row oh
            if (th < 0 || th % st != 0 || th / st >= OH) continue;
            const int oh = th / st;
            for (int kw = 0; kw < ks; ++kw) {
                const int tw = w + pad - kw * dl;
                if (tw < 0 || tw % st != 0 || tw / st >= OW) continue;
                const int ow = tw / st;
                acc += g_colsT[(long long)((ci * ks + kh) * ks + kw) * P + (r * OH + oh) * OW + ow];
            }
        }
        gx[i] = acc;
    }
}

__global__ void swap01_kernel(const float *__restrict__ in, float *__restrict__ out, long long A, long long B,
                              long long inner) {
    const long long total = A * B * inner;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long t = i % inner, b = (i / inner) % B, a = i / (inner * B);  // i walks the input [A, B, inner]
        out[(b * A + a) * inner + t] = in[i];
    }
}

// out[r] = sum_c a[r, c]; one warp per row
__global__ void rowsum_kernel(const float *__restrict__ a, long long rows, long long cols, float *__restrict__ out) {
    const long long row = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (row >= rows) return;
    float s = 0.f;
    for (long long c = lane; c < cols; c += 32) s += a[row * cols + c];
    s = warp_sum(s);
    if (lane == 0) out[row] = s;
}

static unsigned ew_blocks(long long n) {
    long long b = (n + 255) / 256;
    return (unsigned)(b < 1 ? 1 : (b > 148 * 16 ? 148 * 16 : b));
}

}  // namespace mnf

using namespace mnf;

extern "C" {

int mnf_gemm_f32(int trans_a, int trans_b, int64_t M, int N, int K, const float *A, int64_t lda, const float *B,
                 int64_t ldb, const float *bias, float beta, float *C, int64_t ldc, void *stream) {
    return mnf_gemm_f32_batched(trans_a, trans_b, 1, M, N, K, A, lda, 0, B, ldb, 0, bias, beta, C, ldc, 0, stream);
}

int mnf_gemm_f32_batched(int trans_a, int trans_b, int batch, int64_t M, int N, int K, const float *A, int64_t lda,
                         int64_t stride_a, const float *B, int64_t ldb, int64_t stride_b, const float *bias, float beta,
                         float *C, int64_t ldc, int64_t stride_c, void *stream) {
    MNF_REQUIRE(A && B && C, MNF_E_ARG, "NULL pointer");
    MNF_REQUIRE(M >= 0 && N >= 0 && K >= 0, MNF_E_ARG, "negative size");
    MNF_REQUIRE(batch >= 0 && batch <= 65535, MNF_E_ARG, "bad batch count %d", batch);
    if (M == 0 || N == 0 || batch == 0) return 0;
    const long long gy = (M + 63) / 64;
    MNF_REQUIRE(gy <= 65535, MNF_E_SHAPE, "M=%lld too large for one launch", (long long)M);
    dim3 grid((N + 63) / 64, (unsigned)gy, (unsigned)batch);
    cudaStream_t st = (cudaStream_t)stream;
    const long long sa = stride_a, sb = stride_b, sc = stride_c;
    if (trans_a && trans_b)
        gemm_f32_kernel<true, true><<<grid, 256, 0, st>>>(M, N, K, A, lda, B, ldb, bias, beta, C, ldc, sa, sb, sc);
    else if (trans_a)
        gemm_f32_kernel<true, false><<<grid, 256, 0, st>>>(M, N, K, A, lda, B, ldb, bias, beta, C, ldc, sa, sb, sc);
    else if (trans_b)
        gemm_f32_kernel<false, true><<<grid, 256, 0, st>>>(M, N, K, A, lda, B, ldb, bias, beta, C, ldc, sa, sb, sc);
    else
        gemm_f32_kernel<false, false><<<grid, 256, 0, st>>>(M, N, K, A, lda, B, ldb, bias, beta, C, ldc, sa, sb, sc);
    return launch_status("gemm_f32_kernel");
}

int mnf_ew(int op, const float *a, const float *b, const float *c, const float *d, float *out, float *out2, int64_t n,
           int ncols, void *stream) {
    MNF_REQUIRE(op >= MNF_EW_MUL && op <= MNF_EW_RELU_BWD, MNF_E_ARG, "unknown elementwise op %d", op);
    MNF_REQUIRE(a && out && n >= 0 && ncols >= 1, MNF_E_ARG, "bad argument");
    if (n == 0) return 0;
    ew_kernel<<<ew_blocks(n), 256, 0, (cudaStream_t)stream>>>(op, a, b, c, d, out, out2, n, ncols);
    return launch_status("ew_kernel");
}

int mnf_colsum(const float *a, const float *b, int64_t R, int N, float *out, void *stream) {
    MNF_REQUIRE(a && out && R >= 0 && N >= 1, MNF_E_ARG, "bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    MNF_CUDA(cudaMemsetAsync(out, 0, sizeof(float) * N, st));
    if (R == 0) return 0;
    long long gy = (R + 63) / 64;
    if (gy > 128) gy = 128;
    colsum_kernel<<<dim3((N + 127) / 128, (unsigned)gy), 128, 0, st>>>(a, b, R, N, out);
    return launch_status("colsum_kernel");
}

int mnf_im2col_t(const float *x, float *cols_t, int64_t n_imgs, int c_in, int height, int width, int ksize, void *stream) {
    return mnf_im2col_t_ps(x, cols_t, n_imgs, c_in, height, width, ksize, 0, 1, stream);
}

int mnf_im2col_t_ps(const float *x, float *cols_t, int64_t n_imgs, int c_in, int height, int width, int ksize, int pad,
                    int stride, void *stream) {
    return mnf_im2col_t_geom(x, cols_t, n_imgs, c_in, height, width, ksize, pad, stride, 1, stream);
}

// argument checks shared by the _geom im2col / col2im
static int check_unfold_geom(int height, int width, int ksize, int pad, int stride, int dilation) {
    MNF_REQUIRE(pad >= 0 && stride >= 1, MNF_E_ARG, "bad padding %d or stride %d", pad, stride);
    MNF_REQUIRE(dilation >= 1 && (ksize < 1 || (long long)dilation * (ksize - 1) <= 0x7fff), MNF_E_ARG,
                "bad dilation %d", dilation);
    MNF_REQUIRE(ksize >= 1 && conv_out_size(height, ksize, pad, stride, dilation) >= 1 &&
                    conv_out_size(width, ksize, pad, stride, dilation) >= 1,
                MNF_E_SHAPE, "kernel larger than the padded image");
    return 0;
}

int mnf_im2col_t_geom(const float *x, float *cols_t, int64_t n_imgs, int c_in, int height, int width, int ksize,
                      int pad, int stride, int dilation, void *stream) {
    MNF_REQUIRE(x && cols_t, MNF_E_ARG, "NULL pointer");
    if (const int rc = check_unfold_geom(height, width, ksize, pad, stride, dilation)) return rc;
    const long long total = (long long)c_in * ksize * ksize * n_imgs * conv_out_size(height, ksize, pad, stride, dilation) *
                            conv_out_size(width, ksize, pad, stride, dilation);
    if (total == 0) return 0;
    im2col_t_kernel<<<ew_blocks(total), 256, 0, (cudaStream_t)stream>>>(x, cols_t, n_imgs, c_in, height, width, ksize, pad,
                                                                        stride, dilation);
    return launch_status("im2col_t_kernel");
}

int mnf_col2im_t(const float *grad_cols_t, float *grad_x, int64_t n_imgs, int c_in, int height, int width, int ksize,
                 void *stream) {
    return mnf_col2im_t_ps(grad_cols_t, grad_x, n_imgs, c_in, height, width, ksize, 0, 1, stream);
}

int mnf_col2im_t_ps(const float *grad_cols_t, float *grad_x, int64_t n_imgs, int c_in, int height, int width, int ksize,
                    int pad, int stride, void *stream) {
    return mnf_col2im_t_geom(grad_cols_t, grad_x, n_imgs, c_in, height, width, ksize, pad, stride, 1, stream);
}

int mnf_col2im_t_geom(const float *grad_cols_t, float *grad_x, int64_t n_imgs, int c_in, int height, int width,
                      int ksize, int pad, int stride, int dilation, void *stream) {
    MNF_REQUIRE(grad_cols_t && grad_x, MNF_E_ARG, "NULL pointer");
    if (const int rc = check_unfold_geom(height, width, ksize, pad, stride, dilation)) return rc;
    const long long total = n_imgs * c_in * height * width;
    if (total == 0) return 0;
    col2im_t_kernel<<<ew_blocks(total), 256, 0, (cudaStream_t)stream>>>(grad_cols_t, grad_x, n_imgs, c_in, height, width,
                                                                        ksize, pad, stride, dilation);
    return launch_status("col2im_t_kernel");
}

int mnf_swap01(const float *in, float *out, int64_t dim0, int64_t dim1, int64_t inner, void *stream) {
    MNF_REQUIRE(in && out && in != out, MNF_E_ARG, "NULL or aliased pointer");
    const long long total = dim0 * dim1 * inner;
    if (total == 0) return 0;
    swap01_kernel<<<ew_blocks(total), 256, 0, (cudaStream_t)stream>>>(in, out, dim0, dim1, inner);
    return launch_status("swap01_kernel");
}

int mnf_rowsum(const float *a, int64_t n_rows, int64_t n_cols, float *out, void *stream) {
    MNF_REQUIRE(a && out, MNF_E_ARG, "NULL pointer");
    if (n_rows == 0) return 0;
    const long long threads = n_rows * 32;
    rowsum_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, (cudaStream_t)stream>>>(a, n_rows, n_cols, out);
    return launch_status("rowsum_kernel");
}

int mnf_rnvp_gate_forward(const float *z, const float *mask, const float *shift, const float *scale, float *z_out,
                          float *log_det, int64_t n_rows, int dim, void *stream) {
    MNF_REQUIRE(z && mask && shift && scale && z_out && log_det, MNF_E_ARG, "NULL pointer");
    if (n_rows == 0) return 0;
    const long long threads = n_rows * 32;
    rnvp_gate_fwd_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, (cudaStream_t)stream>>>(z, mask, shift, scale, z_out,
                                                                                            log_det, n_rows, dim);
    return launch_status("rnvp_gate_fwd_kernel");
}

int mnf_rnvp_gate_backward(const float *z, const float *mask, const float *shift, const float *scale,
                           const float *grad_out, const float *grad_log_det, float *grad_shift, float *grad_scale,
                           float *grad_z, int64_t n_rows, int dim, void *stream) {
    MNF_REQUIRE(z && mask && shift && scale && grad_shift && grad_scale && grad_z, MNF_E_ARG, "NULL pointer");
    const long long total = n_rows * dim;
    if (total == 0) return 0;
    rnvp_gate_bwd_kernel<<<ew_blocks(total), 256, 0, (cudaStream_t)stream>>>(z, mask, shift, scale, grad_out, grad_log_det,
                                                                           grad_shift, grad_scale, grad_z, total, dim);
    return launch_status("rnvp_gate_bwd_kernel");
}

int mnf_kl_rows_forward(const float *z, const float *W_mean, const float *W_log_var, const float *r0_c, const float *eps_w,
                        float *pre, float *kl_rows, int n_out, int n_in, void *stream) {
    MNF_REQUIRE(z && W_mean && W_log_var && r0_c && eps_w && pre && kl_rows, MNF_E_ARG, "NULL pointer");
    MNF_REQUIRE(n_out >= 0 && n_in >= 0, MNF_E_ARG, "negative size n_out=%d n_in=%d", n_out, n_in);
    if (n_out == 0) return 0;  // n_in == 0 still writes the empty sums: pre = kl_rows = 0
    const long long threads = (long long)n_out * 32;
    kl_rows_fwd_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, (cudaStream_t)stream>>>(z, W_mean, W_log_var, r0_c, eps_w,
                                                                                          pre, kl_rows, n_out, n_in);
    return launch_status("kl_rows_fwd_kernel");
}

int mnf_kl_rows_backward(const float *z, const float *W_mean, const float *W_log_var, const float *r0_c,
                         const float *eps_w, const float *grad_pre, const float *grad_kl_rows, float *grad_W_mean,
                         float *grad_W_log_var, float *grad_z, float *grad_r0_c, int n_out, int n_in, void *stream) {
    MNF_REQUIRE(z && W_mean && W_log_var && r0_c && eps_w && grad_pre && grad_kl_rows && grad_W_mean && grad_W_log_var &&
                    grad_z && grad_r0_c,
                MNF_E_ARG, "NULL pointer");
    MNF_REQUIRE(n_out >= 0 && n_in >= 0, MNF_E_ARG, "negative size n_out=%d n_in=%d", n_out, n_in);
    if (n_in == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    MNF_CUDA(cudaMemsetAsync(grad_z, 0, sizeof(float) * n_in, st));
    MNF_CUDA(cudaMemsetAsync(grad_r0_c, 0, sizeof(float) * n_in, st));
    if (n_out == 0) return 0;  // grad_z = grad_r0_c = 0, no weights
    int gy = (n_out + 31) / 32;
    if (gy > 64) gy = 64;
    kl_rows_bwd_kernel<<<dim3((n_in + 127) / 128, gy), 128, 0, st>>>(z, W_mean, W_log_var, r0_c, eps_w, grad_pre,
                                                                    grad_kl_rows, grad_W_mean, grad_W_log_var, grad_z,
                                                                    grad_r0_c, n_out, n_in);
    return launch_status("kl_rows_bwd_kernel");
}

}  // extern "C"
