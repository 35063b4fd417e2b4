// flow_stack.cu -- C-ABI entry points for flow stacks (dispatch: MADE kernels, the dim-2 table kernel or affine
// stream when the program qualifies, generic interpreter otherwise) and the two small parameter-side kernels (Glow
// assembly, ActNorm data-dependent init).
#include <cstdint>
#include <new>

#include "common.cuh"
#include "flow_math.cuh"
#include "mnf_common.cuh"

namespace mnf {
int validate_program(const mnf_flow_op *ops, int n_ops, int dim, int64_t n_params);
int launch_flow_generic(const mnf_flow_op *ops, int n_ops, const float *params, int64_t n_params, const float *x,
                        float *y, float *log_det, float *base_lp, float *inter, int64_t n_rows, int dim,
                        int inverse, cudaStream_t stream);
bool flow_pl_accepts(const mnf_flow_op *ops, int n_ops, int dim);
int launch_flow_pl(const mnf_flow_op *ops, int n_ops, const float *params, const float *x, float *y, float *log_det,
                   float *base_lp, float *inter, int64_t n_rows, int dim, int dir_flags, float *workspace,
                   const mnf_gather_out *gather, cudaStream_t stream);
int64_t flow_pl_workspace_floats(int n_ops);
int64_t flow_pl_image_floats(const mnf_flow_op *ops, int n_ops, int dim);
int flow_pl_build(const mnf_flow_op *ops, int n_ops, const float *params, int dim, float *image, cudaStream_t stream);
int launch_made_fast(const mnf_flow_op *ops, int n_ops, const float *params, const float *x, float *y, float *log_det,
                     float *base_lp, float *inter, int64_t n_rows, int dim, int dir_flags, float *scratch,
                     cudaStream_t stream, bool plan_only);
int launch_flow_pl_sample(const mnf_flow_op *ops, int n_ops, const float *params, uint64_t seed, uint32_t noise_stream,
                          uint64_t row_offset, float *x, float *log_prob, float *z, int64_t n_rows, int dim, bool staged,
                          float *workspace, cudaStream_t stream);

// ---------------------------------------------------------------------------------------------------
// Conditioner-free stacks (AffineConstantFlow / ActNormFlow / Glow only, dim 2): the whole stack is ONE
// affine map v -> v A + b with a constant log-det.  A one-thread kernel composes it (fp64) from the packed
// parameters, then a streaming kernel applies it: 8 points per thread in flight, 128-bit accesses, nothing
// but HBM traffic (8 B in, 8 B out, 4 B log-det per point) -- the one flow kernel that is truly HBM-bound.
// ---------------------------------------------------------------------------------------------------
__global__ void affine_compose_kernel(const __grid_constant__ FlowProgram prog, const float *__restrict__ params,
                                      int inverse, float *__restrict__ comp) {
    double A[4] = {1, 0, 0, 1}, b[2] = {0, 0}, ld = 0;
    for (int kk = 0; kk < prog.n_ops; ++kk) {
        const mnf_flow_op &op = prog.ops[inverse ? prog.n_ops - 1 - kk : kk];
        double W[4], t[2] = {0, 0};
        if (op.type == MNF_OP_AFFINE_CONST) {
            const double s0 = params[op.aux_off], s1 = params[op.aux_off + 1];
            const double t0 = params[op.aux_off + 2], t1 = params[op.aux_off + 3];
            if (inverse) {  // (v - t) * exp(-s), affine_constant_flow.py:24
                W[0] = exp(-s0), W[3] = exp(-s1), W[1] = W[2] = 0;
                t[0] = -t0 * W[0], t[1] = -t1 * W[3];
                ld -= s0 + s1;
            } else {  // v * exp(s) + t, affine_constant_flow.py:19
                W[0] = exp(s0), W[3] = exp(s1), W[1] = W[2] = 0;
                t[0] = t0, t[1] = t1;
                ld += s0 + s1;
            }
        } else {  // Glow: v @ W (glow.py:28) or v @ W^-1 (glow.py:36)
            const float *Wp = params + op.aux_off + (inverse ? 4 : 0);
            for (int i = 0; i < 4; ++i) W[i] = Wp[i];
            ld += inverse ? -(double)params[op.aux_off + 8] : (double)params[op.aux_off + 8];
        }
        const double n00 = A[0] * W[0] + A[1] * W[2], n01 = A[0] * W[1] + A[1] * W[3];
        const double n10 = A[2] * W[0] + A[3] * W[2], n11 = A[2] * W[1] + A[3] * W[3];
        const double nb0 = b[0] * W[0] + b[1] * W[2] + t[0], nb1 = b[0] * W[1] + b[1] * W[3] + t[1];
        A[0] = n00, A[1] = n01, A[2] = n10, A[3] = n11, b[0] = nb0, b[1] = nb1;
    }
    for (int i = 0; i < 4; ++i) comp[i] = (float)A[i];
    comp[4] = (float)b[0], comp[5] = (float)b[1], comp[6] = (float)ld;
}

__global__ void __launch_bounds__(256)
affine_stream_kernel(const float *__restrict__ comp, const float4 *__restrict__ x, float4 *__restrict__ y,
                     float2 *__restrict__ log_det, float2 *__restrict__ base_lp, long long n_pairs, int sum_lp) {
    const float a00 = comp[0], a01 = comp[1], a10 = comp[2], a11 = comp[3], b0 = comp[4], b1 = comp[5], ld = comp[6];
    const float c = -1.8378770664093453f;
    constexpr int U = 4;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long p0 = (long long)blockIdx.x * blockDim.x + threadIdx.x; p0 < n_pairs; p0 += U * stride) {
        float4 v[U];
#pragma unroll
        for (int u = 0; u < U; ++u)
            if (p0 + u * stride < n_pairs) v[u] = ld_stream4(x + p0 + u * stride);
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const long long p = p0 + u * stride;
            if (p >= n_pairs) break;
            const float4 q = v[u];
            const float4 o = make_float4(fmaf(q.y, a10, fmaf(q.x, a00, b0)), fmaf(q.y, a11, fmaf(q.x, a01, b1)),
                                         fmaf(q.w, a10, fmaf(q.z, a00, b0)), fmaf(q.w, a11, fmaf(q.z, a01, b1)));
            if (y) st_stream4(y + p, o);
            if (log_det) st_stream2(log_det + p, make_float2(ld, ld));
            if (base_lp) {
                float2 lp = make_float2(fmaf(-0.5f, fmaf(o.x, o.x, o.y * o.y), c), fmaf(-0.5f, fmaf(o.z, o.z, o.w * o.w), c));
                if (sum_lp) lp = make_float2(lp.x + ld, lp.y + ld);
                st_stream2(base_lp + p, lp);
            }
        }
    }
}

static int launch_affine_stream(const FlowProgram &prog, const float *params, const float *x, float *y, float *log_det,
                                float *base_lp, int64_t n_rows, int dir_flags, float *workspace, const DeviceProps *dp,
                                cudaStream_t stream) {
    affine_compose_kernel<<<1, 1, 0, stream>>>(prog, params, dir_flags & 1, workspace);
    int rc = launch_status("affine_compose_kernel");
    if (rc) return rc;
    const long long n_pairs = n_rows / 2;
    long long blocks = (n_pairs + 256 * 4 - 1) / (256 * 4);
    const long long cap = (long long)dp->sm_count * 8;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    affine_stream_kernel<<<(unsigned)blocks, 256, 0, stream>>>(workspace, (const float4 *)x, (float4 *)y, (float2 *)log_det,
                                                             (float2 *)base_lp, n_pairs, (dir_flags & 2) != 0);
    return launch_status("affine_stream_kernel");
}

// Dim-2 dispatch.  Returns 1 if no dim-2 kernel takes the program (the caller runs the interpreter).  dir_flags: bit0
// inverse, bit1 log-det summed into base_lp, bit2 `workspace` holds the staged tables.
//   * conditioner-free stacks (AffineConstantFlow / ActNormFlow / Glow only): affine_stream_kernel when the call suits its
//     128-bit point pairs (even row count, no intermediates, 16-byte aligned points, a workspace for the composed map, not
//     staged), else the table kernel, which then has no tables to build;
//   * every other program flow_pl.cu accepts: the table kernel, with the staged tables or tables built into the workspace
//     (MNF_E_ARG without a workspace).
// The fused peer-memory gather stores log-probabilities: outside MNF_RUN_LOGPROB mode the caller reports it.
static int launch_flow_dim2(const mnf_flow_op *ops, int n_ops, const float *params, const float *x, float *y, float *log_det,
                            float *base_lp, float *inter, int64_t n_rows, int dim, int dir_flags, float *workspace,
                            const mnf_gather_out *gather, cudaStream_t stream) {
    if (dim != 2 || n_ops < 1) return 1;
    const bool want_gather = gather && (gather->n_peers > 0 || gather->multicast_ptr);
    if (want_gather && !(dir_flags & 2)) return 1;
    bool affine_only = true;
    for (int k = 0; k < n_ops; ++k) affine_only &= ops[k].type == MNF_OP_AFFINE_CONST || ops[k].type == MNF_OP_GLOW;
    const bool pairs_aligned = (uintptr_t)x % 16 == 0 && (uintptr_t)y % 16 == 0 && (uintptr_t)log_det % 8 == 0 &&
                               (uintptr_t)base_lp % 8 == 0;
    if (affine_only && !want_gather && !inter && workspace && !(dir_flags & 4) && n_rows % 2 == 0 && n_rows >= 2 &&
        pairs_aligned) {
        FlowProgram prog;
        prog.n_ops = n_ops;
        for (int k = 0; k < n_ops; ++k) prog.ops[k] = ops[k];
        const DeviceProps *dp = device_props();
        MNF_REQUIRE(dp != nullptr, MNF_E_DEVICE, "no CUDA device");
        return launch_affine_stream(prog, params, x, y, log_det, base_lp, n_rows, dir_flags, workspace, dp, stream);
    }
    return launch_flow_pl(ops, n_ops, params, x, y, log_det, base_lp, inter, n_rows, dim, dir_flags, workspace, gather, stream);
}

// ---- base draws of mnf_flow_stack_sample for the programs the table kernel does not run ----
// One thread per row: z[r, c] = philox_normal(element (row_offset + r) dim + c).  finish = 0 stores z; finish = 1 draws the
// same numbers again and turns the log-det the forward pass left in log_prob into log N(z) - log_det (re-drawing costs
// a few hundred instructions per row and needs no [n_rows] buffer between the launches, while the forward pass may have
// overwritten z with x in place).
__global__ void flow_base_draw_kernel(uint64_t seed, uint32_t noise_stream, uint64_t row_offset, float *__restrict__ z,
                                      float *__restrict__ log_prob, long long n_rows, int dim, int finish) {
    const Philox g(seed);
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < n_rows; r += stride) {
        const uint64_t e0 = (row_offset + (uint64_t)r) * (uint64_t)dim;
        float sq = 0.f;
        for (int c = 0; c < dim; ++c) {
            const float v = philox_normal(g, e0 + c, noise_stream);
            if (finish) sq = fmaf(v, v, sq);
            else z[r * dim + c] = v;
        }
        if (finish) log_prob[r] = fmaf(-0.5f, sq, -0.9189385332046727f * (float)dim) - log_prob[r];  // log N(z) - log_det
    }
}

static int launch_base_draw(uint64_t seed, uint32_t noise_stream, uint64_t row_offset, float *z, float *log_prob,
                            int64_t n_rows, int dim, int finish, cudaStream_t stream) {
    const DeviceProps *dp = device_props();
    MNF_REQUIRE(dp != nullptr, MNF_E_DEVICE, "no CUDA device");
    const int threads = 256;
    long long blocks = (n_rows + threads - 1) / threads;
    const long long cap = (long long)dp->sm_count * 8;
    if (blocks > cap) blocks = cap;
    flow_base_draw_kernel<<<(unsigned)blocks, threads, 0, stream>>>(seed, noise_stream, row_offset, z, log_prob, n_rows, dim,
                                                                    finish);
    return launch_status("flow_base_draw_kernel");
}

// ---- Glow: W = P (tril(L,-1)+I) (triu(U,1)+diag S), W^-1 = Um^-1 Lm^-1 P^T (glow.py:20-24,35) ----
// one thread per column; fp64 internally, rounded once to fp32.
__global__ void glow_assemble_kernel(const float *__restrict__ P, const float *__restrict__ L,
                                     const float *__restrict__ U, const float *__restrict__ S,
                                     float *__restrict__ out, int D) {
    const int j = threadIdx.x;
    if (j < D) {
        double c[MNF_MAX_DIM], t[MNF_MAX_DIM];
        // column j of W
        for (int i = 0; i < D; ++i) c[i] = i < j ? (double)U[i * D + j] : (i == j ? (double)S[j] : 0.0);
        for (int i = 0; i < D; ++i) {  // t = Lm c
            double acc = c[i];
            for (int k = 0; k < i; ++k) acc += (double)L[i * D + k] * c[k];
            t[i] = acc;
        }
        for (int i = 0; i < D; ++i) {  // W[:, j] = P t
            double acc = 0.0;
            for (int k = 0; k < D; ++k) acc += (double)P[i * D + k] * t[k];
            out[i * D + j] = (float)acc;
        }
        // column j of W^-1: solve Lm y = P^T e_j, then Um w = y
        for (int i = 0; i < D; ++i) {
            double acc = (double)P[j * D + i];  // (P^T)[i][j]
            for (int k = 0; k < i; ++k) acc -= (double)L[i * D + k] * t[k];
            t[i] = acc;  // reuse t as y (entries < i already final)
        }
        for (int i = D - 1; i >= 0; --i) {
            double acc = t[i];
            for (int k = i + 1; k < D; ++k) acc -= (double)U[i * D + k] * c[k];
            c[i] = acc / (double)S[i];
        }
        for (int i = 0; i < D; ++i) out[D * D + i * D + j] = (float)c[i];
    }
    if (j == 0) {
        float acc = 0.f;
        for (int i = 0; i < D; ++i) acc += logf(fabsf(S[i]));  // glow.py:29
        out[2 * D * D] = acc;
    }
}

// ---- ActNorm init: per-dim sum and sum of squares in fp64, then s, t ----
__global__ void actnorm_stats_kernel(const float *__restrict__ x, long long n_elems, int D,
                                     double *__restrict__ ws) {
    // total thread count is a multiple of D, so a thread always meets the same column
    const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    double s = 0.0, ss = 0.0;
    for (long long e = tid; e < n_elems; e += stride) {
        const double v = (double)x[e];
        s += v;
        ss += v * v;
    }
    const int d = (int)(tid % D);
    atomicAdd(&ws[d], s);
    atomicAdd(&ws[D + d], ss);
}

__global__ void actnorm_finish_kernel(const double *__restrict__ ws, long long n_rows, int D, float *s, float *t,
                                      int do_s, int do_t) {
    const int d = blockIdx.x * blockDim.x + threadIdx.x;
    if (d >= D) return;
    const double n = (double)n_rows;
    const double mean = ws[d] / n;
    if (do_s) {
        const double var = (ws[D + d] - n * mean * mean) / (n - 1.0);  // unbiased, torch.std default
        s[d] = (float)(0.5 * log(var));                                // affine_constant_flow.py:46
    }
    if (do_t) t[d] = (float)(mean * exp((double)s[d]));  // mean(x * exp(s)), affine_constant_flow.py:48
}

}  // namespace mnf

using namespace mnf;

extern "C" {

int mnf_flow_stack_plan(const mnf_flow_op *ops_host, int n_ops, int dim, int64_t n_params) {
    int rc = validate_program(ops_host, n_ops, dim, n_params);
    if (rc) return rc;
    float dummy = 0.f;  // a non-NULL output so that the plan does not depend on a scratch buffer
    for (int inverse = 0; inverse < 2; ++inverse)
        if (launch_made_fast(ops_host, n_ops, nullptr, nullptr, &dummy, nullptr, nullptr, nullptr, 0, dim, inverse,
                             nullptr, nullptr, true) == 0)
            return 2;
    return flow_pl_accepts(ops_host, n_ops, dim) ? 1 : 0;
}

int mnf_flow_stack_run(const mnf_flow_op *ops_host, int n_ops, const float *params, int64_t n_params,
                       const float *x, float *y, float *log_det, float *base_log_prob, float *intermediates,
                       int64_t n_rows, int dim, int flags, float *workspace, const mnf_gather_out *gather,
                       void *stream) {
    int rc = validate_program(ops_host, n_ops, dim, n_params);
    if (rc) return rc;
    MNF_REQUIRE(n_rows >= 0, MNF_E_ARG, "n_rows=%lld is negative", (long long)n_rows);
    MNF_REQUIRE((flags & ~(MNF_RUN_INVERSE | MNF_RUN_GENERIC | MNF_RUN_LOGPROB | MNF_RUN_STAGED | MNF_RUN_VARIANT_MASK)) == 0, MNF_E_ARG,
                "unknown bits in flags=0x%x", flags);
    // bit1: sum into base_lp; bit2: workspace holds the staged tables of the dim-2 table kernel
    const int inverse = (flags & MNF_RUN_INVERSE) | ((flags & MNF_RUN_LOGPROB) ? 2 : 0) |
                        ((flags & MNF_RUN_STAGED) && workspace && dim == 2 ? 4 : 0);
    if (n_rows == 0) return 0;
    MNF_REQUIRE(x != nullptr, MNF_E_ARG, "x is NULL");
    MNF_REQUIRE(y || log_det || base_log_prob, MNF_E_ARG, "no output requested");
    MNF_REQUIRE(params || n_params == 0, MNF_E_ARG, "params is NULL");
    cudaStream_t st = (cudaStream_t)stream;
    if (!(flags & MNF_RUN_GENERIC) && !gather) {
        rc = launch_made_fast(ops_host, n_ops, params, x, y, log_det, base_log_prob, intermediates, n_rows, dim,
                              inverse, workspace, st, false);
        if (rc != 1) return rc;
    }
    if (!(flags & MNF_RUN_GENERIC)) {
        rc = launch_flow_dim2(ops_host, n_ops, params, x, y, log_det, base_log_prob, intermediates, n_rows, dim, inverse,
                              workspace, gather, st);
        if (rc != 1) return rc;
    }
    MNF_REQUIRE(!gather || (gather->n_peers == 0 && !gather->multicast_ptr), MNF_E_SHAPE,
                "peer-memory gather output needs the dim-2 table kernel (a program it runs, in log-prob mode)");
    return launch_flow_generic(ops_host, n_ops, params, n_params, x, y, log_det, base_log_prob, intermediates,
                               n_rows, dim, inverse & 3, st);
}

int mnf_flow_stack_sample(const mnf_flow_op *ops_host, int n_ops, const float *params, int64_t n_params, uint64_t seed,
                          uint32_t noise_stream, uint64_t row_offset, float *x, float *log_prob, float *z, int64_t n_rows,
                          int dim, int flags, float *workspace, void *stream) {
    int rc = validate_program(ops_host, n_ops, dim, n_params);
    if (rc) return rc;
    MNF_REQUIRE(n_rows >= 0, MNF_E_ARG, "n_rows=%lld is negative", (long long)n_rows);
    MNF_REQUIRE((flags & ~(MNF_RUN_GENERIC | MNF_RUN_STAGED | MNF_RUN_VARIANT_MASK)) == 0, MNF_E_ARG,
                "flags=0x%x: sampling takes MNF_RUN_GENERIC, MNF_RUN_STAGED and MNF_RUN_VARIANT(v) only", flags);
    if (n_rows == 0) return 0;
    MNF_REQUIRE(x || log_prob || z, MNF_E_ARG, "no output requested");
    MNF_REQUIRE(params || n_params == 0, MNF_E_ARG, "params is NULL");
    cudaStream_t st = (cudaStream_t)stream;
    const bool staged = (flags & MNF_RUN_STAGED) && workspace && dim == 2;
    // whole call in the table kernel: the draw, the stack and log N(z) - log_det in one pass
    if (!(flags & MNF_RUN_GENERIC) && n_ops > 0 && (x || log_prob)) {
        rc = launch_flow_pl_sample(ops_host, n_ops, params, seed, noise_stream, row_offset, x, log_prob, z, n_rows, dim, staged,
                                   workspace, st);
        if (rc != 1) return rc;
    }
    // otherwise: draw z (into x when the caller does not want z, the forward pass then runs in place), run the forward
    // dispatch of mnf_flow_stack_run with its log-det in log_prob, and finish log_prob with the re-drawn log N(z)
    float *zb = z ? z : x;
    MNF_REQUIRE(zb != nullptr, MNF_E_ARG,
                "this program is not run by the table kernel (or no workspace was given): pass x or z to hold the drawn points");
    rc = launch_base_draw(seed, noise_stream, row_offset, zb, nullptr, n_rows, dim, 0, st);
    if (rc || !(x || log_prob)) return rc;
    if (n_ops == 0) {
        if (x && x != zb) MNF_CUDA(cudaMemcpyAsync(x, zb, sizeof(float) * n_rows * dim, cudaMemcpyDeviceToDevice, st));
        if (log_prob) MNF_CUDA(cudaMemsetAsync(log_prob, 0, sizeof(float) * n_rows, st));
    } else {
        const int dir = staged ? 4 : 0;  // forward; a staged image is passed on as such
        rc = 1;
        if (!(flags & MNF_RUN_GENERIC))
            rc = launch_made_fast(ops_host, n_ops, params, zb, x, log_prob, nullptr, nullptr, n_rows, dim, dir, workspace, st, false);
        if (rc == 1 && !(flags & MNF_RUN_GENERIC))
            rc = launch_flow_dim2(ops_host, n_ops, params, zb, x, log_prob, nullptr, nullptr, n_rows, dim, dir, workspace, nullptr, st);
        if (rc == 1)
            rc = launch_flow_generic(ops_host, n_ops, params, n_params, zb, x, log_prob, nullptr, nullptr, n_rows, dim, 0, st);
        if (rc) return rc;
    }
    return log_prob ? launch_base_draw(seed, noise_stream, row_offset, nullptr, log_prob, n_rows, dim, 1, st) : 0;
}

struct mnf_flow_handle {
    int n_ops, dim;
    int64_t n_params, workspace_rows;
    const float *params, *staged;
    float *workspace;
    mnf_flow_op ops[MNF_MAX_OPS];
};

int mnf_flow_handle_create(const mnf_flow_op *ops_host, int n_ops, const float *params, int64_t n_params, int dim,
                           const float *staged, float *workspace, int64_t workspace_rows, mnf_flow_handle **out) {
    MNF_REQUIRE(out != nullptr, MNF_E_ARG, "out is NULL");
    *out = nullptr;
    int rc = validate_program(ops_host, n_ops, dim, n_params);
    if (rc) return rc;
    MNF_REQUIRE(n_ops >= 1 && n_ops <= MNF_MAX_OPS, MNF_E_SHAPE, "n_ops=%d outside [1,%d]", n_ops, MNF_MAX_OPS);
    MNF_REQUIRE(params || n_params == 0, MNF_E_ARG, "params is NULL");
    MNF_REQUIRE(!staged || dim == 2, MNF_E_ARG, "a staged image exists for dim-2 programs only");
    mnf_flow_handle *h = new (std::nothrow) mnf_flow_handle();
    MNF_REQUIRE(h != nullptr, MNF_E_ARG, "out of host memory");
    h->n_ops = n_ops, h->dim = dim, h->n_params = n_params, h->workspace_rows = workspace_rows;
    h->params = params, h->staged = staged, h->workspace = workspace;
    for (int k = 0; k < n_ops; ++k) h->ops[k] = ops_host[k];
    *out = h;
    return 0;
}

void mnf_flow_handle_destroy(mnf_flow_handle *handle) { delete handle; }

int mnf_flow_handle_log_prob(const mnf_flow_handle *h, const float *x, float *log_prob, int64_t n_rows, void *stream) {
    MNF_REQUIRE(h && x && log_prob, MNF_E_ARG, "NULL pointer");
    MNF_REQUIRE(n_rows >= 0, MNF_E_ARG, "n_rows=%lld is negative", (long long)n_rows);
    if (n_rows == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    const int base = 1 | 2;  // inverse direction, log_det summed into the base log-density
    int rc;
    if (h->dim != 2) {
        rc = launch_made_fast(h->ops, h->n_ops, h->params, x, nullptr, nullptr, log_prob, nullptr, n_rows, h->dim, base,
                              n_rows <= h->workspace_rows ? h->workspace : nullptr, st, false);
        if (rc != 1) return rc;
    } else if (h->staged) {  // the staged conditioner tables: the table kernel, any batch
        rc = launch_flow_dim2(h->ops, h->n_ops, h->params, x, nullptr, nullptr, log_prob, nullptr, n_rows, 2, base | 4,
                              const_cast<float *>(h->staged), nullptr, st);
        if (rc != 1) return rc;
    } else {
        MNF_REQUIRE(n_rows <= h->workspace_rows && h->workspace, MNF_E_ARG,
                    "handle was created with a workspace for %lld rows, call has %lld", (long long)h->workspace_rows,
                    (long long)n_rows);
        rc = launch_flow_dim2(h->ops, h->n_ops, h->params, x, nullptr, nullptr, log_prob, nullptr, n_rows, 2, base, h->workspace,
                              nullptr, st);
        if (rc != 1) return rc;
    }
    return launch_flow_generic(h->ops, h->n_ops, h->params, h->n_params, x, nullptr, nullptr, log_prob, nullptr, n_rows,
                               h->dim, base, st);
}

int64_t mnf_flow_stack_stage_size(const mnf_flow_op *ops_host, int n_ops, int dim, int64_t n_params) {
    if (validate_program(ops_host, n_ops, dim, n_params)) return 0;
    return flow_pl_image_floats(ops_host, n_ops, dim);
}

int64_t mnf_flow_stack_stage_max_rows(const mnf_flow_op *ops_host, int n_ops, int dim, int64_t n_params) {
    if (validate_program(ops_host, n_ops, dim, n_params)) return 0;
    return flow_pl_image_floats(ops_host, n_ops, dim) > 0 ? INT64_MAX : 0;
}

int mnf_flow_stack_stage(const mnf_flow_op *ops_host, int n_ops, const float *params, int64_t n_params, int dim,
                         float *staged, void *stream) {
    int rc = validate_program(ops_host, n_ops, dim, n_params);
    if (rc) return rc;
    return flow_pl_build(ops_host, n_ops, params, dim, staged, (cudaStream_t)stream);
}

int64_t mnf_flow_stack_workspace(int n_ops, int64_t n_rows, int dim) {
    if (dim == 64) return n_rows * 64;  // MADE density stack in log-prob mode parks z here between flows
    // dim 2: the conditioner tables of the table kernel (the constants of affine_stream_kernel fit in less)
    (void)n_rows;
    return dim == 2 ? flow_pl_workspace_floats(n_ops) : 0;
}

int mnf_glow_assemble(const float *P, const float *L, const float *U, const float *S, float *out, int dim,
                      void *stream) {
    MNF_REQUIRE(P && L && U && S && out, MNF_E_ARG, "NULL pointer");
    MNF_REQUIRE(dim >= 1 && dim <= MNF_MAX_DIM, MNF_E_SHAPE, "dim=%d outside [1,%d]", dim, MNF_MAX_DIM);
    glow_assemble_kernel<<<1, 64, 0, (cudaStream_t)stream>>>(P, L, U, S, out, dim);
    return launch_status("glow_assemble_kernel");
}

int mnf_actnorm_init(const float *x, int64_t n_rows, int dim, float *s, float *t, int do_s, int do_t,
                     double *workspace, void *stream) {
    MNF_REQUIRE(x && s && t && workspace, MNF_E_ARG, "NULL pointer");
    MNF_REQUIRE(dim >= 1 && dim <= MNF_MAX_DIM, MNF_E_SHAPE, "dim=%d outside [1,%d]", dim, MNF_MAX_DIM);
    MNF_REQUIRE(n_rows >= 2, MNF_E_SHAPE, "ActNorm init needs at least 2 rows, got %lld", (long long)n_rows);
    cudaStream_t st = (cudaStream_t)stream;
    MNF_CUDA(cudaMemsetAsync(workspace, 0, sizeof(double) * 2 * dim, st));
    const int threads = 4 * dim * (256 / (4 * dim) > 0 ? 256 / (4 * dim) : 1);  // multiple of dim, <= 256
    const long long n_elems = (long long)n_rows * dim;
    long long blocks = (n_elems + threads - 1) / threads;
    if (blocks > 592) blocks = 592;
    actnorm_stats_kernel<<<(unsigned)blocks, threads, 0, st>>>(x, n_elems, dim, workspace);
    int rc = launch_status("actnorm_stats_kernel");
    if (rc) return rc;
    actnorm_finish_kernel<<<1, 64, 0, st>>>(workspace, n_rows, dim, s, t, do_s, do_t);
    return launch_status("actnorm_finish_kernel");
}

}  // extern "C"
