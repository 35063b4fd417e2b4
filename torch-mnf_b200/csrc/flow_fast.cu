// flow_fast.cu -- host-side planning and dispatch for the dim-2 register-resident flow kernel
// (templates in flow_fast.cuh; one translation unit per (H, K) instantiation so they build
// in parallel).
#include "flow_fast.cuh"

namespace mnf {

// (hidden width, spline bins) instantiations, one translation unit each (flow_fast_h*k*.cu): the BASELINE shapes
// (16, 8), (24, 8) and the reference's defaults (8, 5), plus neighbours so that common variations stay off the interpreter
#define MNF_FLOW_FAST_SHAPES(X) X(16, 8) X(24, 8) X(8, 5) X(8, 8) X(16, 5) X(32, 8)
#define MNF_DECLARE_SHAPE(HH, KK) int launch_fast_##HH##_##KK(MNF_FLOW_FAST_ARGS);
MNF_FLOW_FAST_SHAPES(MNF_DECLARE_SHAPE)
#undef MNF_DECLARE_SHAPE

int launch_flow_pl(const mnf_flow_op *ops, int n_ops, const float *params, const float *x, float *y, float *log_det,
                   float *base_lp, float *inter, int64_t n_rows, int dim, int dir_flags, float *workspace,
                   const mnf_gather_out *gather, cudaStream_t stream, bool plan_only);

int launch_flow_lanes(const mnf_flow_op *ops, int n_ops, const float *params, const float *x, float *y, float *log_det,
                      float *base_lp, float *inter, int64_t n_rows, int dim, int dir_flags, cudaStream_t stream, bool plan_only,
                      bool forced);

// ---- host side: plan + launch ---------------------------------------------------------

struct FastPlan {
    int H = 0, K = 0;
    bool ok = false;
    FastLayout lay;
};

static FastPlan plan_fast(const mnf_flow_op *ops, int n_ops, int dim) {
    FastPlan p;
    if (dim != 2 || n_ops < 1) return p;
    int H = 0, K = 0, slots = 0;
    bool has_spline_op = false;
    for (int k = 0; k < n_ops; ++k) {
        const mnf_flow_op &op = ops[k];
        has_spline_op |= op.type == MNF_OP_NSF_CL;
        p.lay.net_slot[k][0] = p.lay.net_slot[k][1] = 0;
        if (op.type == MNF_OP_AFFINE_CONST || op.type == MNF_OP_GLOW) continue;
        if (op.type != MNF_OP_AFFINE_HALF && op.type != MNF_OP_NSF_CL) return p;
        if (op.n_lin != 4 || op.sizes[0] != 1) return p;
        const int h = op.sizes[1];
        if (op.sizes[2] != h || op.sizes[3] != h) return p;
        if (H && h != H) return p;
        H = h;
        int n_out = 1;
        if (op.type == MNF_OP_NSF_CL) {
            if (K && op.K != K) return p;
            K = op.K;
            n_out = 3 * K - 1;
        }
        if (op.sizes[4] != n_out) return p;
        const int per_net = fast_net_slots(h, n_out);
        for (int which = 0; which < 2; ++which) {
            p.lay.net_slot[k][which] = slots;
            slots += per_net;
        }
    }
    if (H == 0) H = 8, K = 5;  // conditioner-free stack (ActNorm / Glow only): pure streaming, any instantiation does
    if (K == 0) K = 8;
    bool have = false;
#define MNF_HAVE_SHAPE(HH, KK) have |= (H == HH && K == KK);
    MNF_FLOW_FAST_SHAPES(MNF_HAVE_SHAPE)
#undef MNF_HAVE_SHAPE
    if (!have && !has_spline_op) {  // AffineHalfFlow-only stacks do not care about K: any instantiation of their width does
#define MNF_HAVE_WIDTH(HH, KK) if (!have && H == HH) have = true, K = KK;
        MNF_FLOW_FAST_SHAPES(MNF_HAVE_WIDTH)
#undef MNF_HAVE_WIDTH
    }
    if (!have) return p;
    p.H = H;
    p.K = K;
    p.lay.total_slots = slots;
    p.ok = true;
    return p;
}

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

// returns 1 if the program is not eligible (caller falls back to the generic kernel)
int launch_flow_fast(const mnf_flow_op *ops, int n_ops, const float *params, int64_t n_params, const float *x,
                     float *y, float *log_det, float *base_lp, float *inter, int64_t n_rows, int dim, int inverse,
                     int variant, float *workspace, const mnf_gather_out *gather, cudaStream_t stream,
                     bool plan_only) {
    bool has_net = false;
    for (int k = 0; k < n_ops; ++k) has_net |= ops[k].type == MNF_OP_NSF_CL || ops[k].type == MNF_OP_AFFINE_HALF;
    const bool want_gather = gather && (gather->n_peers > 0 || gather->multicast_ptr);
    // variant 6 (default wherever it applies): every conditioner as a piecewise-linear table of its scalar input
    // (flow_pl.cu), one launch for the whole stack after the table builder; any hidden widths up to 64, K in {4, 5, 6, 8, 10, 12, 16}.
    // A staged image (bit 2) holds such tables (mnf_flow_stack_stage stages nothing else), so a staged call always lands here.
    if ((variant == 6 || variant < 0 || (inverse & 4)) && (!want_gather || (inverse & 2)) && (workspace || plan_only)) {
        const int rc = launch_flow_pl(ops, n_ops, params, x, y, log_det, base_lp, inter, n_rows, dim, inverse & 7, workspace, gather,
                                      stream, plan_only);
        if (rc != 1) return rc;
    }
    if (variant == 6) variant = -1;
    // variant 5: eight lanes per point (flow_lanes.cu) -- small batches of AffineHalfFlow stacks, where a call is bound by
    // the latency of one point's chain.  Default for its class up to 2048 rows (a staged image, bit 2, is simply not needed by it).
    if (!want_gather && (variant == 5 || (variant < 0 && !plan_only))) {
        const int rc = launch_flow_lanes(ops, n_ops, params, x, y, log_det, base_lp, inter, n_rows, dim, inverse & 3, stream, plan_only,
                                         variant == 5);
        if (rc != 1) return rc;
    }
    if (variant == 5) variant = -1;
    // variant 2, also run for requests of 0, 1 and 3 (variants removed earlier): the shared-memory FFMA2 kernel, which
    // needs no workspace
    if (want_gather) return 1;  // the fused peer-memory gather lives in the table kernel only: caller reports the restriction
    FastPlan p = plan_fast(ops, n_ops, dim);
    if (!p.ok) return 1;
    const DeviceProps *dp = plan_only ? nullptr : device_props();
    const size_t smem_bytes = (size_t)p.lay.total_slots * sizeof(float);
    if (plan_only) return smem_bytes <= 227 * 1024 ? 0 : 1;
    MNF_REQUIRE(dp != nullptr, MNF_E_DEVICE, "no CUDA device");
    if (smem_bytes > (size_t)dp->smem_optin) return 1;
    MNF_REQUIRE(((uintptr_t)x % 16) == 0 && (!y || ((uintptr_t)y % 16) == 0), MNF_E_ALIGN,
                "x and y must be 16-byte aligned for the dim-2 kernel");
    MNF_REQUIRE(!log_det || ((uintptr_t)log_det % 8) == 0, MNF_E_ALIGN, "log_det must be 8-byte aligned");
    MNF_REQUIRE(!base_lp || ((uintptr_t)base_lp % 8) == 0, MNF_E_ALIGN, "base_log_prob must be 8-byte aligned");
    if (inter && (n_rows % 2)) return 1;  // per-flow outputs of an odd batch are not 16 B aligned: generic path
    MNF_REQUIRE(!inter || ((uintptr_t)inter % 16) == 0, MNF_E_ALIGN, "intermediates must be 16-byte aligned");
    FlowProgram prog;
    prog.n_ops = n_ops;
    for (int k = 0; k < n_ops; ++k) prog.ops[k] = ops[k];
    (void)n_params;
    if (!has_net && variant < 0 && !inter && workspace && !(inverse & 4) && n_rows % 2 == 0 && n_rows >= 2)
        return launch_affine_stream(prog, params, x, y, log_det, base_lp, n_rows, inverse, workspace, dp, stream);
#define MNF_LAUNCH_SHAPE(HH, KK)                                                                                           \
    if (p.H == HH && p.K == KK)                                                                                            \
        return launch_fast_##HH##_##KK(prog, p.lay, smem_bytes, params, x, y, log_det, base_lp, inter, n_rows, inverse, dp, \
                                       stream);
    MNF_FLOW_FAST_SHAPES(MNF_LAUNCH_SHAPE)
#undef MNF_LAUNCH_SHAPE
    return 1;
}

}  // namespace mnf
