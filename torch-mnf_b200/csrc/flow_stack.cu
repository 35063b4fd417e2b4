// flow_stack.cu -- C-ABI entry points for flow stacks (dispatch: dim-2 register-resident
// kernel when the program qualifies, generic interpreter otherwise) and the two small
// parameter-side kernels (Glow assembly, ActNorm data-dependent init).
#include <cstdint>
#include <new>

#include "common.cuh"
#include "mnf_common.cuh"

namespace mnf {
int validate_program(const mnf_flow_op *ops, int n_ops, int dim, int64_t n_params);
int launch_flow_generic(const mnf_flow_op *ops, int n_ops, const float *params, int64_t n_params, const float *x,
                        float *y, float *log_det, float *base_lp, float *inter, int64_t n_rows, int dim,
                        int inverse, cudaStream_t stream);
int launch_flow_fast(const mnf_flow_op *ops, int n_ops, const float *params, int64_t n_params, const float *x,
                     float *y, float *log_det, float *base_lp, float *inter, int64_t n_rows, int dim, int inverse,
                     int mode, float *workspace, const mnf_gather_out *gather, cudaStream_t stream, bool plan_only);
int64_t flow_pl_workspace_floats(int n_ops);
int64_t flow_pl_image_floats(const mnf_flow_op *ops, int n_ops, int dim);
int flow_pl_build(const mnf_flow_op *ops, int n_ops, const float *params, int dim, float *image, cudaStream_t stream);
int launch_made_fast(const mnf_flow_op *ops, int n_ops, const float *params, const float *x, float *y, float *log_det,
                     float *base_lp, float *inter, int64_t n_rows, int dim, int dir_flags, float *scratch,
                     cudaStream_t stream, bool plan_only);
int launch_flow_pl_sample(const mnf_flow_op *ops, int n_ops, const float *params, uint64_t seed, uint32_t noise_stream,
                          uint64_t row_offset, float *x, float *log_prob, float *z, int64_t n_rows, int dim, bool staged,
                          float *workspace, cudaStream_t stream);

// MNF_RUN_VARIANT(v) of a call, -1 = library default.  Variant 4 named a kernel the table kernel replaced: its requests run
// the library default.
static int requested_variant(int flags) {
    const int v = ((flags & MNF_RUN_VARIANT_MASK) >> 4) - 1;
    return v == 4 ? -1 : v;
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
    return launch_flow_fast(ops_host, n_ops, nullptr, n_params, nullptr, nullptr, nullptr, nullptr, nullptr, 0,
                            dim, 0, -1, nullptr, nullptr, nullptr, true) == 0
               ? 1
               : 0;
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
    const int variant = requested_variant(flags);
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
        rc = launch_flow_fast(ops_host, n_ops, params, n_params, x, y, log_det, base_log_prob, intermediates,
                              n_rows, dim, inverse, variant, workspace, gather, st, false);
        if (rc != 1) return rc;
    }
    MNF_REQUIRE(!gather || (gather->n_peers == 0 && !gather->multicast_ptr), MNF_E_SHAPE,
                "peer-memory gather output needs the piecewise-linear dim-2 kernel (AffineHalfFlow / NSF_CL stack in log-prob mode, with a workspace)");
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
    const int variant = requested_variant(flags);
    // whole call in the table kernel: the draw, the stack and log N(z) - log_det in one pass
    if (!(flags & MNF_RUN_GENERIC) && (variant < 0 || variant == 6 || staged) && n_ops > 0 && (x || log_prob)) {
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
            rc = launch_flow_fast(ops_host, n_ops, params, n_params, zb, x, log_prob, nullptr, nullptr, n_rows, dim, dir, variant,
                                  workspace, nullptr, st, false);
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
        rc = launch_flow_fast(h->ops, h->n_ops, h->params, h->n_params, x, nullptr, nullptr, log_prob, nullptr, n_rows, 2,
                              base | 4, -1, const_cast<float *>(h->staged), nullptr, st, false);
        if (rc != 1) return rc;
    } else {
        MNF_REQUIRE(n_rows <= h->workspace_rows && h->workspace, MNF_E_ARG,
                    "handle was created with a workspace for %lld rows, call has %lld", (long long)h->workspace_rows,
                    (long long)n_rows);
        rc = launch_flow_fast(h->ops, h->n_ops, h->params, h->n_params, x, nullptr, nullptr, log_prob, nullptr, n_rows, 2,
                              base, -1, h->workspace, nullptr, st, false);
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
    // dim 2: the conditioner tables of the piecewise-linear kernel (the constants of affine_stream_kernel fit in less;
    // every other dim-2 kernel needs none)
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
