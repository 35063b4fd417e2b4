// flow_generic.cu -- generic flow-stack interpreter: one thread per point, any dim <= 64,
// any conditioner widths <= 128, any spline bin count <= 32, every flow type of the
// reference (flows/core.py:17-35 and the modules it iterates over).  This is the
// correctness-complete path; the BASELINE shapes (dim 2) take the table kernel in
// flow_pl.cu instead.  Parameters are staged in shared memory when the blob
// fits, otherwise read through L1.
#include "flow_math.cuh"

namespace mnf {

struct Net {
    const float *w;  // start of the packed net
    int n_lin;
    const int *sizes;  // n_lin + 1 entries
};

__device__ __forceinline__ int net_floats(const int *sizes, int n_lin) {
    int n = 0;
    for (int l = 0; l < n_lin; ++l) n += sizes[l + 1] * sizes[l] + sizes[l + 1];
    return n;
}

// Runs all layers except the last; leaves the last hidden activation in `a` (returns its width)
// and the pointer to the last layer's weights in *last_w.  relu: ReLU (MADE) else LeakyReLU(0.2).
__device__ int mlp_hidden(const Net &net, const float *in, int n_in, float *a, float *b, bool relu,
                          const float **last_w) {
    const float *w = net.w;
    int width = n_in;
    const float *cur = in;
    float *dst = a;
    for (int l = 0; l + 1 < net.n_lin; ++l) {
        const int n_out = net.sizes[l + 1];
        const float *bias = w + n_out * width;
        for (int j = 0; j < n_out; ++j) {
            float acc = bias[j];
            const float *row = w + j * width;
            for (int i = 0; i < width; ++i) acc = fmaf(row[i], cur[i], acc);
            dst[j] = relu ? fmaxf(acc, 0.f) : leaky02(acc);
        }
        w = bias + n_out;
        width = n_out;
        cur = dst;
        dst = (dst == a) ? b : a;
    }
    if (cur != a) {
        for (int i = 0; i < width; ++i) a[i] = cur[i];
    }
    *last_w = w;
    return width;
}

// One output of the last Linear layer.
__device__ __forceinline__ float mlp_out(const float *last_w, int width, int n_out, const float *h, int j) {
    float acc = last_w[n_out * width + j];
    const float *row = last_w + j * width;
    for (int i = 0; i < width; ++i) acc = fmaf(row[i], h[i], acc);
    return acc;
}

__device__ void op_affine_const(const mnf_flow_op &op, const float *P, float *v, int D, bool inverse, float &ld) {
    const float *s = P + op.aux_off, *t = s + D;
    float sum = 0.f;
    for (int d = 0; d < D; ++d) {
        if (inverse)
            v[d] = (v[d] - t[d]) * expf(-s[d]);  // affine_constant_flow.py:24
        else
            v[d] = v[d] * expf(s[d]) + t[d];  // affine_constant_flow.py:19
        sum += s[d];
    }
    ld += inverse ? -sum : sum;
}

__device__ void op_glow(const mnf_flow_op &op, const float *P, float *v, float *tmp, int D, bool inverse,
                        float &ld) {
    const float *W = P + op.aux_off + (inverse ? D * D : 0);  // glow.py:28 / :35-36 (right multiply)
    for (int j = 0; j < D; ++j) {
        float acc = 0.f;
        for (int i = 0; i < D; ++i) acc = fmaf(v[i], W[i * D + j], acc);
        tmp[j] = acc;
    }
    for (int j = 0; j < D; ++j) v[j] = tmp[j];
    const float logdet = P[op.aux_off + 2 * D * D];
    ld += inverse ? -logdet : logdet;
}

__device__ void op_affine_half(const mnf_flow_op &op, const float *P, float *v, float *a, float *b, float *a2,
                               int D, bool inverse, float &ld) {
    const int h = D / 2;
    const bool parity = op.flags & MNF_FLAG_PARITY;
    float *cond = v + (parity ? h : 0);   // untouched half (affine_half_flow.py:46-50)
    float *trans = v + (parity ? 0 : h);  // transformed half
    const float *ws = nullptr, *wt = nullptr;
    int width_s = 0, width_t = 0;
    Net net{nullptr, op.n_lin, op.sizes};
    if (op.flags & MNF_FLAG_SCALE) {
        net.w = P + op.net_off[0];
        width_s = mlp_hidden(net, cond, h, a, b, false, &ws);
    }
    if (op.flags & MNF_FLAG_SHIFT) {
        net.w = P + op.net_off[1];
        width_t = mlp_hidden(net, cond, h, a2, b, false, &wt);
    }
    float sum = 0.f;
    for (int j = 0; j < h; ++j) {
        const float s = ws ? mlp_out(ws, width_s, h, a, j) : 0.f;
        const float t = wt ? mlp_out(wt, width_t, h, a2, j) : 0.f;
        if (inverse)
            b[j] = (trans[j] - t) / expf(s);  // affine_half_flow.py:54
        else
            b[j] = expf(s) * trans[j] + t;  // affine_half_flow.py:58
        sum += s;
    }
    for (int j = 0; j < h; ++j) trans[j] = b[j];
    ld += inverse ? -sum : sum;
}

// conditioner -> spline over `n_t` transformed dims; raw params of dim j are outputs
// [j*(3K-1), (j+1)*(3K-1)) of the net (spline_flow.py:252-253 reshape).
__device__ void spline_block(const mnf_flow_op &op, const float *net_w, const float *cond, int n_cond,
                             float *trans, int n_t, float *a, float *b, float *raw, bool rqs_inverse,
                             float &ld) {
    const int nb = 3 * op.K - 1;
    Net net{net_w, op.n_lin, op.sizes};
    const float *lw;
    const int width = mlp_hidden(net, cond, n_cond, a, b, false, &lw);
    const int n_out = op.sizes[op.n_lin];
    for (int j = 0; j < n_t; ++j) {
        for (int o = 0; o < nb; ++o) raw[o] = mlp_out(lw, width, n_out, a, j * nb + o);
        rq_spline<0, false>(raw, op.K, op.bound, op.edge_deriv, rqs_inverse, trans[j], ld);
    }
}

__device__ void op_nsf_cl(const mnf_flow_op &op, const float *P, float *v, float *a, float *b, float *raw, int D,
                          bool inverse, float &ld) {
    const int h = D / 2;
    float *lower = v, *upper = v + h;
    const float *f1 = P + op.net_off[0], *f2 = P + op.net_off[1];
    if (!inverse) {  // spline_flow.py:249-266
        spline_block(op, f1, lower, h, upper, h, a, b, raw, false, ld);
        spline_block(op, f2, upper, h, lower, h, a, b, raw, false, ld);
    } else {  // spline_flow.py:268-285
        spline_block(op, f2, upper, h, lower, h, a, b, raw, true, ld);
        spline_block(op, f1, lower, h, upper, h, a, b, raw, true, ld);
    }
}

__device__ void op_nsf_ar(const mnf_flow_op &op, const float *P, float *v, float *out, float *a, float *b,
                          float *raw, int D, bool inverse, float &ld) {
    // spline_flow.py:199-235.  forward conditions on its own outputs and runs the spline
    // inverse; inverse conditions on its inputs and runs the spline forward.
    const int nb = 3 * op.K - 1;
    int sizes[MNF_MAX_LIN + 1];
    for (int l = 0; l <= op.n_lin; ++l) sizes[l] = op.sizes[l];
    const float *w = P + op.net_off[0];
    for (int i = 0; i < D; ++i) {
        float x = v[i];
        if (i == 0) {
            for (int o = 0; o < nb; ++o) raw[o] = P[op.aux_off + o];
        } else {
            sizes[0] = i;
            Net net{w, op.n_lin, sizes};
            const float *lw;
            const int width = mlp_hidden(net, inverse ? v : out, i, a, b, false, &lw);
            for (int o = 0; o < nb; ++o) raw[o] = mlp_out(lw, width, nb, a, o);
            w += net_floats(sizes, op.n_lin);
        }
        rq_spline<0, false>(raw, op.K, op.bound, op.edge_deriv, !inverse, x, ld);
        out[i] = x;
    }
    for (int i = 0; i < D; ++i) v[i] = out[i];
}

__device__ void op_made(const mnf_flow_op &op, const float *P, float *v, float *out, float *a, float *b, int D,
                        bool inverse, float &ld) {
    const bool parity = op.flags & MNF_FLAG_PARITY;
    const bool seq_on_forward = op.flags & MNF_FLAG_MADE_SEQ;
    const bool sequential = seq_on_forward ? !inverse : inverse;
    Net net{P + op.net_off[0], op.n_lin, op.sizes};
    const float *lw;
    if (!sequential) {
        // maf.py:53-62: one pass, z = x*exp(s)+t, flip afterwards, ld = sum s
        const int width = mlp_hidden(net, v, D, a, b, true, &lw);
        float sum = 0.f;
        for (int i = 0; i < D; ++i) {
            const float s = mlp_out(lw, width, 2 * D, a, i);
            const float t = mlp_out(lw, width, 2 * D, a, D + i);
            out[parity ? D - 1 - i : i] = v[i] * expf(s) + t;
            sum += s;
        }
        for (int i = 0; i < D; ++i) v[i] = out[i];
        ld += sum;
    } else {
        // maf.py:39-51: flip first, then D sequential passes over the partially built x
        for (int i = 0; i < D; ++i) out[i] = 0.f;
        for (int i = 0; i < D; ++i) {
            const int width = mlp_hidden(net, out, D, a, b, true, &lw);
            const float s = mlp_out(lw, width, 2 * D, a, i);
            const float t = mlp_out(lw, width, 2 * D, a, D + i);
            const float z = v[parity ? D - 1 - i : i];
            out[i] = (z - t) * expf(-s);
            ld -= s;
        }
        for (int i = 0; i < D; ++i) v[i] = out[i];
    }
}

__global__ void __launch_bounds__(128)
flow_generic_kernel(const __grid_constant__ FlowProgram prog, const float *__restrict__ params, int n_params,
                    int params_in_smem, const float *__restrict__ x, float *__restrict__ y,
                    float *__restrict__ log_det, float *__restrict__ base_lp, float *__restrict__ inter,
                    long long n_rows, int D, int dir_flags) {
    extern __shared__ float smem[];
    const int inverse = dir_flags & 1;
    const bool sum_lp = dir_flags & 2;
    const float *P = params;
    if (params_in_smem) {
        for (int i = threadIdx.x; i < n_params; i += blockDim.x) smem[i] = params[i];
        __syncthreads();
        P = smem;
    }
    float v[MNF_MAX_DIM], tmp[MNF_MAX_DIM];
    float a[MNF_MAX_HIDDEN], b[MNF_MAX_HIDDEN], a2[MNF_MAX_HIDDEN];
    float raw[3 * MNF_MAX_BINS];

    for (long long row = (long long)blockIdx.x * blockDim.x + threadIdx.x; row < n_rows;
         row += (long long)gridDim.x * blockDim.x) {
        for (int d = 0; d < D; ++d) v[d] = x[row * D + d];
        float ld = 0.f;
        for (int k = 0; k < prog.n_ops; ++k) {
            const mnf_flow_op &op = prog.ops[inverse ? prog.n_ops - 1 - k : k];
            switch (op.type) {
                case MNF_OP_AFFINE_CONST: op_affine_const(op, P, v, D, inverse, ld); break;
                case MNF_OP_GLOW: op_glow(op, P, v, tmp, D, inverse, ld); break;
                case MNF_OP_AFFINE_HALF: op_affine_half(op, P, v, a, b, a2, D, inverse, ld); break;
                case MNF_OP_NSF_CL: op_nsf_cl(op, P, v, a, b, raw, D, inverse, ld); break;
                case MNF_OP_NSF_AR: op_nsf_ar(op, P, v, tmp, a, b, raw, D, inverse, ld); break;
                case MNF_OP_MADE: op_made(op, P, v, tmp, a, b, D, inverse, ld); break;
                default: break;
            }
            if (inter) {
                float *dst = inter + ((size_t)k * n_rows + row) * D;
                for (int d = 0; d < D; ++d) dst[d] = v[d];
            }
        }
        if (y)
            for (int d = 0; d < D; ++d) y[row * D + d] = v[d];
        if (log_det) log_det[row] = ld;
        if (base_lp) {
            float ss = 0.f;
            for (int d = 0; d < D; ++d) ss = fmaf(v[d], v[d], ss);
            const float lp = -0.5f * ss - 0.5f * (float)D * 1.8378770664093453f;  // log(2 pi)
            base_lp[row] = sum_lp ? lp + ld : lp;
        }
    }
}

int validate_program(const mnf_flow_op *ops, int n_ops, int dim, int64_t n_params) {
    MNF_REQUIRE(ops != nullptr, MNF_E_ARG, "ops_host is NULL");
    MNF_REQUIRE(n_ops >= 0 && n_ops <= MNF_MAX_OPS, MNF_E_SHAPE, "n_ops=%d outside [0,%d]", n_ops, MNF_MAX_OPS);
    MNF_REQUIRE(dim >= 1 && dim <= MNF_MAX_DIM, MNF_E_SHAPE, "dim=%d outside [1,%d]", dim, MNF_MAX_DIM);
    for (int k = 0; k < n_ops; ++k) {
        const mnf_flow_op &op = ops[k];
        MNF_REQUIRE(op.type >= MNF_OP_AFFINE_CONST && op.type <= MNF_OP_MADE, MNF_E_ARG, "op %d: bad type %d", k,
                    op.type);
        const bool has_net = op.type >= MNF_OP_AFFINE_HALF;
        if (has_net) {
            MNF_REQUIRE(op.n_lin >= 1 && op.n_lin <= MNF_MAX_LIN, MNF_E_SHAPE, "op %d: n_lin=%d outside [1,%d]", k,
                        op.n_lin, MNF_MAX_LIN);
            for (int l = 1; l < op.n_lin; ++l)
                MNF_REQUIRE(op.sizes[l] >= 1 && op.sizes[l] <= MNF_MAX_HIDDEN, MNF_E_SHAPE,
                            "op %d: hidden width %d outside [1,%d]", k, op.sizes[l], MNF_MAX_HIDDEN);
            MNF_REQUIRE(op.net_off[0] >= 0 && op.net_off[0] < n_params, MNF_E_ARG, "op %d: net offset out of range",
                        k);
        }
        if (op.type == MNF_OP_AFFINE_HALF || op.type == MNF_OP_NSF_CL)
            MNF_REQUIRE(dim % 2 == 0, MNF_E_SHAPE, "op %d: coupling flows need an even dim, got %d", k, dim);
        if (op.type == MNF_OP_NSF_CL || op.type == MNF_OP_NSF_AR) {
            MNF_REQUIRE(op.K >= 2 && op.K <= MNF_MAX_BINS, MNF_E_SHAPE, "op %d: K=%d outside [2,%d]", k, op.K,
                        MNF_MAX_BINS);
            MNF_REQUIRE(kMinBin * op.K <= 1.0f, MNF_E_SHAPE, "op %d: minimal bin width too large for K=%d", k,
                        op.K);  // spline_flow.py:90-93
            MNF_REQUIRE(op.bound > 0.f, MNF_E_ARG, "op %d: tail bound must be positive", k);
        }
        if (op.type <= MNF_OP_GLOW || op.type == MNF_OP_NSF_AR)
            MNF_REQUIRE(op.aux_off >= 0 && op.aux_off < n_params, MNF_E_ARG, "op %d: aux offset out of range", k);
    }
    return 0;
}

int launch_flow_generic(const mnf_flow_op *ops, int n_ops, const float *params, int64_t n_params, const float *x,
                        float *y, float *log_det, float *base_lp, float *inter, int64_t n_rows, int dim,
                        int inverse, cudaStream_t stream) {
    const DeviceProps *dp = device_props();
    MNF_REQUIRE(dp != nullptr, MNF_E_DEVICE, "no CUDA device");
    FlowProgram prog;
    prog.n_ops = n_ops;
    for (int k = 0; k < n_ops; ++k) prog.ops[k] = ops[k];
    const size_t smem_bytes = (size_t)n_params * sizeof(float);
    const int in_smem = smem_bytes <= (size_t)dp->smem_optin - 1024;
    const size_t dyn = in_smem ? smem_bytes : 0;
    if (dyn > 48 * 1024)
        MNF_CUDA(cudaFuncSetAttribute(flow_generic_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));
    const int threads = 128;
    long long blocks = (n_rows + threads - 1) / threads;
    const long long cap = (long long)dp->sm_count * 8;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    flow_generic_kernel<<<(unsigned)blocks, threads, dyn, stream>>>(prog, params, (int)n_params, in_smem, x, y,
                                                                     log_det, base_lp, inter, n_rows, dim, inverse);
    return launch_status("flow_generic_kernel");
}

}  // namespace mnf
