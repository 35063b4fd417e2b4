/*
 * mnf_b200.h -- C ABI of libmnf_b200.so: the sm_100a (B200) implementation of the
 * torch-mnf hot path (flow forward/inverse + log-det, MNF layer forward, kl_div).
 *
 * The reference (janosh/torch-mnf) is pure Python on ATen and has no FFI layer; the
 * boundary a maintainer binds is therefore the set of module methods listed beside
 * each entry point (file:line relative to the reference checkout).  The ctypes stub
 * that binds these symbols is shown in INTEGRATION.md and lives in
 * torch-mnf_b200/torch_mnf/_lib.py.
 *
 * Conventions (all entry points):
 *   - plain C: pointers, sizes, POD structs.  No torch / C++ types cross the boundary.
 *   - every data pointer is a DEVICE pointer to contiguous fp32 unless its name ends
 *     in `_host`.  The caller owns all memory (inputs, outputs, packed parameters,
 *     workspaces); the library allocates nothing persistent and frees nothing.
 *   - work is enqueued on `stream` (a cudaStream_t passed as void*); no hidden
 *     synchronisation, no default-stream use.
 *   - return value: 0 = OK, negative = argument/shape error (MNF_E_*), positive =
 *     cudaError_t.  mnf_last_error() returns a thread-local message.  Nothing throws
 *     or exits across the boundary.
 */
#ifndef MNF_B200_H
#define MNF_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MNF_ABI_VERSION 1

#define MNF_E_ARG (-1)     /* null pointer / bad enum / negative size        */
#define MNF_E_SHAPE (-2)   /* shape outside what the kernels support          */
#define MNF_E_ALIGN (-3)   /* pointer not aligned as documented               */
#define MNF_E_DEVICE (-4)  /* no sm_100 device / wrong architecture           */

int mnf_abi_version(void);
const char *mnf_last_error(void);
/* Kernels launched by this library in this process so far (diagnostics; bench.py's gpu_launches). */
uint64_t mnf_launch_count(void);
/* Per-launch-site tally since the last reset, written as "site=count;site=count;..." (sites are the kernel names the
 * library launches); returns the length needed.  Diagnostics only: bench.py uses it to NAME the kernels of a timed region
 * from what actually ran instead of from a literal. */
int64_t mnf_launch_stats(char *buf, int64_t size);
void mnf_launch_stats_reset(void);
/* Fills SM count, max opt-in shared memory per block, compute capability major/minor of
 * the current device.  Any pointer may be NULL. */
int mnf_device_info(int *sm_count, int *smem_optin, int *cc_major, int *cc_minor);

/* ------------------------------------------------------------------------------------
 * Flow stacks: NormalizingFlow.forward / .inverse (flows/core.py:17-35) over
 * AffineConstantFlow/ActNormFlow (affine_constant_flow.py:18-26), AffineHalfFlow
 * (affine_half_flow.py:44-66), Glow (glow.py:26-37), MAF/IAF (maf.py:39-62),
 * NSF_CL / NSF_AR (spline_flow.py:199-285).  One launch runs the whole stack: each
 * point stays in registers across all flows and its log-det is accumulated on chip.
 * ---------------------------------------------------------------------------------- */
enum mnf_flow_type {
    MNF_OP_AFFINE_CONST = 1, /* aux: s[D], t[D]                                         */
    MNF_OP_GLOW = 2,         /* aux: W[D*D], Winv[D*D], logdet[1] (mnf_glow_assemble)    */
    MNF_OP_AFFINE_HALF = 3,  /* net[0] = s_net, net[1] = t_net (MLP, LeakyReLU 0.2)      */
    MNF_OP_NSF_CL = 4,       /* net[0] = f1, net[1] = f2                                 */
    MNF_OP_NSF_AR = 5,       /* aux: init_param[3K-1]; net[0] = layers.0, rest follow    */
    MNF_OP_MADE = 6,         /* net[0] = MADE with masks folded in (ReLU); see flags     */
};

#define MNF_FLAG_PARITY 1u    /* AffineHalfFlow / MAF parity                              */
#define MNF_FLAG_SCALE 2u     /* AffineHalfFlow has s_net                                 */
#define MNF_FLAG_SHIFT 4u     /* AffineHalfFlow has t_net                                 */
#define MNF_FLAG_MADE_SEQ 8u  /* MADE op runs the D-pass sequential direction when the    */
                              /* stack runs forward (MAF) -- if clear, when it runs inverse (IAF) */

#define MNF_MAX_OPS 32
#define MNF_MAX_LIN 6
#define MNF_MAX_DIM 64
#define MNF_MAX_HIDDEN 128
#define MNF_MAX_BINS 32

/* One flow of the stack.  Offsets are in floats into the packed parameter blob.  A net is
 * stored as, per Linear layer l: weight[sizes[l+1]][sizes[l]] (torch's [out][in] order)
 * followed by bias[sizes[l+1]]. */
typedef struct mnf_flow_op {
    int32_t type;                   /* enum mnf_flow_type                               */
    uint32_t flags;                 /* MNF_FLAG_*                                       */
    int32_t K;                      /* spline bins (NSF_*)                              */
    float bound;                    /* spline tail bound B (NSF_*)                      */
    int32_t n_lin;                  /* Linear layers per conditioner net                */
    int32_t sizes[MNF_MAX_LIN + 1]; /* layer widths, sizes[0] = net input width         */
    int32_t net_off[2];             /* offsets of the conditioner nets                  */
    int32_t aux_off;                /* offset of the op's auxiliary parameters          */
    float edge_deriv;               /* NSF: min_deriv + softplus(log(exp(1-min_deriv)-1)) */
} mnf_flow_op;

/* Runs `n_ops` flows over `n_rows` points of dimension `dim`.
 *   ops_host     : host array of descriptors, in module order (flows[0] first).
 *   params       : device fp32 blob the offsets refer to, `n_params` floats.
 *   x            : input  [n_rows, dim];   y: output [n_rows, dim] (may alias x; NULL = do not
 *                  store the transformed points, e.g. when only log-probabilities are wanted).
 *   log_det      : output [n_rows] -- sum of the flows' log|det J| (core.py:19,23).
 *   base_log_prob: optional output [n_rows]: standard-normal log-density of y
 *                  (NormalizingFlowModel.base_log_prob, core.py:46-49, for a N(0,I) base).
 *   intermediates: optional output [n_ops, n_rows, dim]: the output of every flow in
 *                  execution order (core.py:20-25 returns them as a list).
 *   workspace    : mnf_flow_stack_workspace() floats of scratch (caller-owned), or NULL if that is 0.
 *   flags        : MNF_RUN_INVERSE = inverse direction (flows[n-1] first), else forward;
 *                  MNF_RUN_GENERIC forces the generic interpreter; MNF_RUN_VARIANT(v) picks a
 *                  code variant of the dim-2 kernel (tests / tuning; 0 = library default);
 *                  MNF_RUN_LOGPROB makes base_log_prob receive log_det + base log-density, i.e.
 *                  log p(x) of tests/test_flows.py:22-24 in one pass.
 * Replaces NormalizingFlow.forward/inverse (flows/core.py:17-35). */
/* Optional fused result gather over NVLink / NVSwitch peer memory: besides base_log_prob the kernel stores every
 * log-probability straight into the gather buffers of the other ranks (peer-mapped device pointers, e.g. from
 * torch.distributed._symmetric_memory) at element row_offset + i -- or, when multicast_ptr is set, with ONE
 * multimem.st per element that the switch replicates to every rank.  The data transfer overlaps the kernel's
 * arithmetic; the only collective left after the launch is a barrier.  Supported by the piecewise-linear and the
 * tensor-core dim-2 kernels in MNF_RUN_LOGPROB mode. */
#define MNF_MAX_PEERS 8
typedef struct mnf_gather_out {
    int32_t n_peers;                 /* entries of peer_ptrs in use (0 with multicast)       */
    int32_t reserved;
    int64_t row_offset;              /* first element of this rank's slice in every gather buffer */
    float *peer_ptrs[MNF_MAX_PEERS]; /* base of the [world * n_rows] buffer on each OTHER rank */
    float *multicast_ptr;            /* NVLS multicast address of the same buffer, or NULL    */
} mnf_gather_out;

int mnf_flow_stack_run(const mnf_flow_op *ops_host, int n_ops, const float *params,
                       int64_t n_params, const float *x, float *y, float *log_det,
                       float *base_log_prob, float *intermediates, int64_t n_rows, int dim,
                       int flags, float *workspace, const mnf_gather_out *gather /* may be NULL */,
                       void *stream);

/* A flow program bound once, for call sites that evaluate the same model over and over (BASELINE config 1: 4096
 * points per call, where a call is latency-bound): the handle keeps a host copy of the descriptors and the device
 * pointers of the packed parameters and of the pre-staged net image, so that a log-probability call is five arguments
 * and no validation.  The caller owns every device buffer and must keep them alive and UNCHANGED while the handle is in
 * use (re-create it after a parameter update); the handle itself is a small host allocation freed by
 * mnf_flow_handle_destroy.  staged: mnf_flow_stack_stage output for these parameters or NULL; workspace:
 * mnf_flow_stack_workspace(n_ops, max_rows, dim) floats or NULL if that is 0 (with `staged`, programs of the
 * piecewise-linear kernel need none at any batch size, others none below 65536 rows).
 *   mnf_flow_handle_log_prob: log_prob[r] = log|det J|(x_r) + standard-normal log-density of the result, i.e.
 *   NormalizingFlowModel.log_prob (flows/core.py:46-49 over :27-35) for an N(0, I) base, one fused pass. */
typedef struct mnf_flow_handle mnf_flow_handle;
int mnf_flow_handle_create(const mnf_flow_op *ops_host, int n_ops, const float *params, int64_t n_params, int dim,
                           const float *staged, float *workspace, int64_t workspace_rows, mnf_flow_handle **out);
void mnf_flow_handle_destroy(mnf_flow_handle *handle);
int mnf_flow_handle_log_prob(const mnf_flow_handle *handle, const float *x, float *log_prob, int64_t n_rows,
                             void *stream);

/* Reverse-mode pass of mnf_flow_stack_run (the reference trains through torch autograd:
 * tests/test_flows.py:14-31 calls loss.backward() on -(log_det + base_log_prob)).
 *   x              [n_rows, dim]         the input the forward run saw
 *   intermediates  [n_ops, n_rows, dim]  what the forward run stored (output of every flow, execution order)
 *   grad_intermediates  same shape or NULL: d loss / d (each flow's output), the last slice being the stack's result
 *   grad_y         [n_rows, dim] or NULL: extra d loss / d result (added to the last slice above)
 *   grad_log_det   [n_rows] or NULL
 *   grad_x         [n_rows, dim] or NULL (out): d loss / d x
 *   grad_params    [n_params] (in/out): parameter gradients are ADDED at the offsets the parameters have in
 *                  `params` (zero it first); for a Glow op it receives d/dW, d/dW^-1 and d/dlogdet of the assembled
 *                  block and the host chains them to L, S, U.
 * flags: MNF_RUN_INVERSE or 0 -- the direction of the forward run.  Every flow type in both directions.
 * Exact-fp32 arithmetic, one thread per point. */
int mnf_flow_stack_backward(const mnf_flow_op *ops_host, int n_ops, const float *params, int64_t n_params,
                            float *grad_params, const float *x, const float *intermediates,
                            const float *grad_y, const float *grad_log_det, const float *grad_intermediates,
                            float *grad_x, int64_t n_rows, int dim, int flags, void *stream);

/* Floats of scratch `workspace` must provide for a run of this shape (0 = none needed; NULL is then
 * accepted).  dim 2: room for the conditioner tables of the piecewise-linear kernel (built per call when no staged image
 * is passed) or the weight image of the tensor-core kernel, whichever is larger (the library keeps no device state of
 * its own: per-call staging lives here; without a workspace a dim-2 run takes the shared-memory kernels, which need
 * none); dim 64: a log-prob-only MADE run parks the points between flows. */
int64_t mnf_flow_stack_workspace(int n_ops, int64_t n_rows, int dim);

#define MNF_RUN_INVERSE 1
#define MNF_RUN_GENERIC 2
#define MNF_RUN_LOGPROB 4
#define MNF_RUN_STAGED 8  /* `workspace` holds the image written by mnf_flow_stack_stage for these params (below) */
#define MNF_RUN_VARIANT_MASK 0x70
#define MNF_RUN_VARIANT(v) ((((v) + 1) << 4) & MNF_RUN_VARIANT_MASK)
/* v: 6 = every conditioner as a piecewise-linear table of its scalar input (csrc/flow_pl.cu) -- the library default for
 *        dim-2 stacks of AffineConstantFlow / ActNormFlow / Glow / AffineHalfFlow / NSF_CL(K in {4, 5, 6, 8, 10, 12, 16}) whose conditioners
 *        have 1..5 hidden layers of width <= 64, any batch size;
 *    0, 1, 2 = shared-memory weight variants of the register-resident dim-2 kernel (2 = default of the remaining shapes of
 *        its (hidden, bins) grid, and of calls without a workspace);
 *    4 = conditioner MLPs on the tensor cores (NSF_CL(K=8, n_h=16) stacks);
 *    5 = eight lanes per point (AffineHalfFlow stacks up to 32768 rows); 3 (round 1's constant-bank variant, removed) runs 2.
 *    A variant the program is not eligible for falls back to the library default. */

/* Draws n_rows points of the flow model (standard-normal base, flows in module order) together with their log-density:
 *   z[r]        = N(0, I) draw of global row row_offset + r (Noise convention of the MNF layers below: Philox4x32-10
 *                 keyed by `seed`, stream `noise_stream`, GLOBAL element index (row_offset + r) * dim + c as counter, the
 *                 same numbers as every other Philox draw of the library -- shards of one draw, each with its
 *                 row_offset, reproduce the single call bit for bit);
 *   x[r]        = forward pass of z[r] (NormalizingFlowModel.sample, flows/core.py:51-55);
 *   log_prob[r] = log N(z[r]) - log|det J|(z[r]) = log q(x[r]), the density of the drawn point, without the inverse pass.
 * x, log_prob and z are each optional (NULL), at least one must be given.  flags: MNF_RUN_STAGED, MNF_RUN_GENERIC and
 * MNF_RUN_VARIANT(v) as for mnf_flow_stack_run (forward direction only: MNF_RUN_INVERSE and MNF_RUN_LOGPROB are
 * MNF_E_ARG).  Programs of the piecewise-linear kernel with a workspace or staged image take ONE launch (after the table
 * builder when not staged); every other program draws z, runs the forward dispatch of mnf_flow_stack_run and finishes
 * log_prob: at most three launches, and x or z must be given to hold the draw.  Box-Muller draws u1 >= 2^-23, so every
 * pair lies within radius 5.65 (a pair of true normals exceeds it with probability 2^-23). */
int mnf_flow_stack_sample(const mnf_flow_op *ops_host, int n_ops, const float *params, int64_t n_params,
                          uint64_t seed, uint32_t noise_stream, uint64_t row_offset,
                          float *x, float *log_prob, float *z, int64_t n_rows, int dim,
                          int flags, float *workspace, void *stream);

/* Per-parameter-version preparation of a dim-2 stack, done ONCE instead of in every call (call it again whenever a
 * parameter changes): mnf_flow_stack_stage writes into a caller-owned, 16-byte aligned buffer of
 * mnf_flow_stack_stage_size() floats (0 = the program has no such form)
 *   - the conditioner TABLES of the piecewise-linear kernel (sorted breakpoints and per-piece slopes / values of every
 *     conditioner, found in fp64) for the programs that kernel runs -- any batch size; a run with MNF_RUN_STAGED and that
 *     buffer as `workspace` is then ONE launch, always of that kernel (a variant request is ignored);
 *   - otherwise the shared-memory layout of the nets for the register-resident kernel (variant 2), for runs of fewer
 *     than 65 536 rows: the kernel then starts with a plain vector copy. */
int64_t mnf_flow_stack_stage_size(const mnf_flow_op *ops_host, int n_ops, int dim, int64_t n_params);
/* Largest batch a MNF_RUN_STAGED run of this program accepts: INT64_MAX when the staged image holds the conditioner
 * tables (any batch), 65535 when it is the shared-memory layout of the register-resident kernel, 0 without a staged form. */
int64_t mnf_flow_stack_stage_max_rows(const mnf_flow_op *ops_host, int n_ops, int dim, int64_t n_params);
int mnf_flow_stack_stage(const mnf_flow_op *ops_host, int n_ops, const float *params, int64_t n_params, int dim,
                         float *staged, void *stream);

/* Which kernel mnf_flow_stack_run would pick: 0 = generic interpreter, 1 = specialised
 * D=2 kernels (tensor cores / register-resident / lane-split by shape and batch), 2 = the exact-fp32 MADE kernels
 * (all-MAF/IAF stacks of an instantiated (dim, hidden) shape with three hidden layers).  Host-only, no launch. */
int mnf_flow_stack_plan(const mnf_flow_op *ops_host, int n_ops, int dim, int64_t n_params);

/* Glow._assemble_W + torch.inverse (glow.py:20-24, 34-35):  W = P (tril(L,-1)+I)(triu(U,1)+diag S),
 * W^-1 by triangular solves, logdet = sum log|S|.  out = [W (D*D) | Winv (D*D) | logdet (1)].
 * All pointers device; D <= MNF_MAX_DIM. */
int mnf_glow_assemble(const float *P, const float *L, const float *U, const float *S, float *out,
                      int dim, void *stream);

/* ActNormFlow data-dependent init (affine_constant_flow.py:44-49):
 * s = log(std(x, dim 0, unbiased)), t = mean(x * exp(s), dim 0).  `do_s` / `do_t` select which
 * are (re)computed (the reference skips an all-zero parameter).  workspace: 4*dim doubles,
 * zero-initialised by the call. */
int mnf_actnorm_init(const float *x, int64_t n_rows, int dim, float *s, float *t, int do_s,
                     int do_t, double *workspace, void *stream);

/* ------------------------------------------------------------------------------------
 * MNF layers.  Noise convention: every noise tensor pointer may be NULL, in which case the
 * kernel draws from Philox4x32-10 keyed by `seed`, with `noise_stream` distinguishing the
 * draws of one call and the GLOBAL element index (row_offset + local row) as counter, so a
 * batch sharded over GPUs sees the same numbers as a single-device call.  Injected tensors
 * follow the reference's draw order (SURVEY.md section 8c) for parity tests.
 * ---------------------------------------------------------------------------------- */

/* z0 = q0_mean + sqrt(exp(q0_log_var)) * eps, eps ~ N(0,1) [n_rows, dim]
 * (MNFLinear.sample_z mnf_linear.py:58-62; MNFConv2d.sample_z mnf_conv.py:80-84 with n_rows = 1). */
int mnf_sample_z0(const float *q0_mean, const float *q0_log_var, const float *eps, uint64_t seed,
                  uint32_t noise_stream, uint64_t row_offset, float *z, int64_t n_rows, int dim,
                  void *stream);

#define MNF_RNVP_MAX_NET 4
/* One RNVP flow (flows/rnvp.py:19-23): net = MLP(dim, *h_sizes) (Linear/LeakyReLU(0.2), last
 * activation dropped), t, s = Linear(h_sizes[-1], dim).  Device pointers, torch [out][in] layout. */
typedef struct mnf_rnvp_flow {
    int32_t n_net;                       /* Linear layers in `net` (= len(h_sizes))          */
    int32_t net_sizes[MNF_RNVP_MAX_NET]; /* their output widths                               */
    const float *net_w[MNF_RNVP_MAX_NET];
    const float *net_b[MNF_RNVP_MAX_NET];
    const float *t_w, *t_b, *s_w, *s_b;
} mnf_rnvp_flow;

/* NormalizingFlow([RNVP...]).forward (core.py:17-25 over rnvp.py:25-39), in place on z [n_rows, dim]:
 *   mask ~ Bernoulli(.5); y = net(mask*z); g = sigmoid(s(y)); z <- (1-mask) z g + (1-g) t(y) + mask z;
 *   log_det[r] = sum over flows and dims of (1-mask) log g   (written, not accumulated).
 * masks_host: host array of n_flows device pointers [n_rows, dim] of 0/1 floats, or NULL (Philox,
 * flow f uses noise stream first_noise_stream + f).  workspace: 2 * n_rows * max(net_sizes) floats.
 * intermediates: optional [n_flows, n_rows, dim]. */
int mnf_rnvp_forward(const mnf_rnvp_flow *flows_host, int n_flows, float *z, float *log_det,
                     const float *const *masks_host, uint64_t seed, uint32_t first_noise_stream,
                     uint64_t row_offset, int64_t n_rows, int dim, float *workspace,
                     float *intermediates, void *stream);

/* MNFLinear.forward after sample_z (mnf_linear.py:46-56):
 *   out = (x*z) W_mean^T + b_mean + sqrt(x^2 exp(W_log_var)^T + exp(b_log_var)) * eps
 * x: [x_rows, n_in]; output row r reads x[r % x_rows], i.e. x.repeat(n_rows / x_rows, 1) without
 * materialising it (Monte-Carlo replication, mnf_mnist.ipynb:316-318).  z: [n_rows, n_in],
 * eps: [n_rows, n_out] or NULL, out: [n_rows, n_out]; relu = 1 applies the nn.ReLU that follows
 * the layer in MNFLeNet / MNFFeedForward in the epilogue. */
int mnf_linear_forward(const float *x, int64_t x_rows, const float *z, const float *W_mean,
                       const float *W_log_var, const float *b_mean, const float *b_log_var,
                       const float *eps, uint64_t seed, uint32_t noise_stream, uint64_t row_offset,
                       float *out, int64_t n_rows, int n_in, int n_out, int relu, void *stream);

/* Tensor-core (tcgen05, TF32 inputs, fp32 accumulation in TMEM, TMA-fed) variant of mnf_linear_forward
 * for n_in % 4 == 0 and 16-byte aligned operands; results agree with the fp32 path to the 2e-3 relative
 * tolerance BASELINE.json states for tensor-core GEMM outputs.  workspace: mnf_linear_tc_workspace()
 * floats.  The variance GEMM runs once per DISTINCT input row (x_rows), not per Monte-Carlo sample. */
int64_t mnf_linear_tc_workspace(int64_t x_rows, int64_t n_rows, int n_in, int n_out);
int mnf_linear_forward_tc(const float *x, int64_t x_rows, const float *z, const float *W_mean,
                          const float *W_log_var, const float *b_mean, const float *b_log_var,
                          const float *eps, uint64_t seed, uint32_t noise_stream, uint64_t row_offset,
                          float *out, int64_t n_rows, int n_in, int n_out, int relu, float *workspace,
                          void *stream);
/* mnf_rnvp_forward on the tensor cores (single-Linear conditioners of width <= 64, dim % 16 == 0).
 * Optionally leaves xz_out = tf32(x[m % x_rows] * z_final), the A operand of mnf_linear_forward_tc's mean
 * GEMM (pass z = NULL there and put xz_out at the start of its workspace).  workspace:
 * mnf_rnvp_tc_workspace() floats. */
int64_t mnf_rnvp_tc_workspace(int n_flows, int64_t n_rows, int dim);
int mnf_rnvp_forward_tc(const mnf_rnvp_flow *flows_host, int n_flows, float *z, float *log_det,
                        const float *const *masks_host, uint64_t seed, uint32_t first_noise_stream,
                        uint64_t row_offset, int64_t n_rows, int dim, const float *x, int64_t x_rows,
                        float *xz_out, float *workspace,
                        /* optional: draw z0 = q0_mean + sqrt(exp(q0_log_var)) * eps_z here (z is then output only) */
                        const float *q0_mean, const float *q0_log_var, const float *eps_z, uint32_t eps_stream,
                        /* 1: the caller consumes only xz_out; z is scratch and its final value may be left unwritten */
                        int z_is_scratch, void *stream);

/* out = A W^T (+ bias) (+ ReLU) on the tensor cores: A [M,K], W [N,K] (torch Linear layout). */
int mnf_tc_linear(const float *A, const float *W, const float *bias, float *out, int64_t M, int N, int K,
                  int relu, int round_out, void *stream);

/* MAF.inverse -- the density direction -- for a stack of MAF flows (flows/maf.py:53-62 over
 * layers/made.py:22-23) as a chain of TF32 tensor-core GEMMs; the last GEMM of every flow applies
 * z = x*exp(s) + t, the parity flip and the log-det row sum in its epilogue.  Weights are packed by the
 * host once per parameter version: mask folded in (W * mask^T), rounded to TF32, output layer rows
 * interleaved (s_0, t_0, s_1, t_1, ...).  Tolerance class: tensor-core GEMM (2e-3). */
#define MNF_MADE_MAX_HIDDEN 4
typedef struct mnf_made_layer {
    int32_t n_hidden;                    /* hidden MaskedLinear layers                       */
    int32_t hidden[MNF_MADE_MAX_HIDDEN]; /* their widths (multiples of 4)                    */
    int32_t parity;                      /* flip dims after the transform (maf.py:60)        */
    const float *w[MNF_MADE_MAX_HIDDEN]; /* [hidden[l], in_l] masked, TF32-rounded           */
    const float *b[MNF_MADE_MAX_HIDDEN]; /* [hidden[l]]                                      */
    const float *w_out;                  /* [2*dim, hidden[last]] interleaved s/t rows       */
    const float *b_out;                  /* [2*dim] interleaved                              */
} mnf_made_layer;
int64_t mnf_made_workspace(int64_t n_rows, int dim, int max_hidden);
int mnf_made_density_tc(const mnf_made_layer *layers_host, int n_flows, const float *x, float *z,
                        float *log_det, float *intermediates /* optional [n_flows, n_rows, dim] */,
                        int64_t n_rows, int dim, float *workspace, void *stream);
/* The same direction for a whole stack of dim-64 MAF flows as ONE persistent tcgen05 kernel (csrc/made_fused.cu): a
 * 128-row tile arrives by TMA, every thread of an epilogue group keeps (half of) one row's exact fp32 coordinates in
 * registers across ALL flows, the hidden activations travel TMEM -> registers -> shared memory (the next MMA's operand)
 * and never reach HBM; traffic is the algorithmic 516 B/row.  Hidden widths <= 31 (column 31 of every padded hidden layer
 * is a constant one that carries the next layer's bias), 1..4 hidden layers, <= 16 flows per call.  MMA operands are
 * fp16 (kind::f16, fp32 accumulation): the 11-bit significand of TF32 at half the shared-memory traffic, which is what
 * bounds the kernel; operands saturate at +-65504, the running point stays exact fp32.
 *   weight_images: per flow, mnf_made_fused_image_bytes(n_hidden) bytes of fp16: W1 [32, 64] | hidden [32, 32] x
 *     (n_hidden-1) | W_out [128, 32] (rows interleaved s_0, t_0, s_1, ...; the s rows and their biases pre-multiplied
 *     by log2(e)), every matrix stored as rows of 128 bytes (K padded to 64 with zeros) in the K-major, 128-byte-swizzled
 *     shared-memory image the UMMA descriptor reads: element (n, k) at fp16 offset (n/8)*512 + (n%8)*64 + (((k/8) ^
 *     (n%8))*8) + k%8, so that one bulk copy per flow stages it.  The parity flips of maf.py:60 are folded in by the
 *     packer: a flow that runs on a reversed row has its input columns and output pairs permuted; final_reversed says
 *     whether the last flow leaves the row reversed (the final store undoes it).
 *   b1: [n_flows, 32] first-layer biases (exact fp32, added in the epilogue).
 *   z / log_det / log_prob: any may be NULL; log_prob = log_det + standard-normal log-density of z.
 *   variant: 0 = default, or 10 * (tiles in flight per CTA) + (threads per row): 21, 31, 41, 32 (tuning / tests).
 * Tolerance class: tensor-core GEMM (2e-3). */
int64_t mnf_made_fused_image_bytes(int n_hidden);
int mnf_made_density_fused(const void *weight_images, const float *b1, int n_flows, int n_hidden, int final_reversed,
                           const float *x, float *z, float *log_det, float *log_prob, int64_t n_rows, int dim,
                           int variant, void *stream);
/* 1 if (A, W, M, N, K) can take the tensor-core path (alignment / shape), else 0.  Host-only. */
int mnf_tc_eligible(const float *A, const float *W, int64_t M, int N, int K);

/* MNFConv2d.forward after sample_z (mnf_conv.py:67-78), stride 1, no padding, NCHW:
 *   out = conv2d(x, W_mean * z[:,None,None,None]) + sqrt(conv2d(x^2, exp(W_log_var)) + exp(b_log_var)) * eps
 * x: [x_imgs, c_in, H, W], image r reads x[r % x_imgs]; z: [c_out] (one draw shared by the batch);
 * eps: [n_imgs, c_out, OH, OW] or NULL.  relu_pool = 1 fuses the nn.ReLU + nn.MaxPool2d(2) that
 * follow each MNFConv2d in MNFLeNet (mnf_lenet.py:16-21): out is then [n_imgs, c_out, OH/2, OW/2]. */
int mnf_conv2d_forward(const float *x, int64_t x_imgs, const float *z, const float *W_mean,
                       const float *W_log_var, const float *b_log_var, const float *eps, uint64_t seed,
                       uint32_t noise_stream, uint64_t row_offset, float *out, int64_t n_imgs, int c_in,
                       int height, int width, int c_out, int ksize, int relu_pool, void *stream);

/* Pieces of the MNF-LeNet Monte-Carlo pipeline (models/mnf_lenet.py:13-26 driven as in mnf_mnist.ipynb:316-318).
 * mnf_conv2d_moments: the sample-independent mean and standard deviation of an MNFConv2d (z is shared by the
 *   call, mnf_conv.py:72), [n_imgs, c_out, OH, OW] each.
 * mnf_conv_noise_relu_pool: out[r] = maxpool2(relu(mean[r % n_unique] + sd[r % n_unique] * eps[r])).
 * mnf_conv2d_forward_tc: MNFConv2d.forward + ReLU + MaxPool2d(2) on the TF32 tensor cores (workspace:
 *   mnf_conv_tc_workspace() floats; tolerance class 2e-3).  When 128 is a multiple of OH*OW, c_out <= 64 and OW % 4 == 0
 *   (MNF-LeNet's second conv) it is an implicit GEMM: x is read once, the x and x^2 operand tiles are generated in
 *   shared memory and both moments come out of one kernel; otherwise im2col + two GEMMs.
 * mnf_conv_tc_stage: packed TF32 weights (and, unless a_mean = a_var = NULL, the materialised im2col operands). */
int mnf_conv2d_moments(const float *x, const float *z, const float *W_mean, const float *W_log_var,
                       const float *b_log_var, float *mean_out, float *sd_out, int64_t n_imgs, int c_in,
                       int height, int width, int c_out, int ksize, void *stream);
int mnf_conv_noise_relu_pool(const float *mean, const float *sd, int64_t n_unique, const float *eps,
                             uint64_t seed, uint32_t noise_stream, uint64_t row_offset, float *out,
                             int64_t n_rows, int channels, int out_h, int out_w, void *stream);
/* Per-sample conv-z variants (the MC predict option of SURVEY 8f-4: every Monte-Carlo sample draws its own z, as
 * S separate reference calls would, mnf_conv.py:80-88).  z scales OUTPUT channels (mnf_conv.py:73), so the moments
 * are evaluated once with unit z and row r's mean is scaled by z_rows[r / rows_per_z, c] in the noise / pool pass.
 * mnf_conv2d_forward_tc_z takes exactly one of z ([c_out], folded into the packed weights) and z_rows. */
int mnf_conv_noise_relu_pool_z(const float *mean, const float *sd, int64_t n_unique, const float *eps,
                               uint64_t seed, uint32_t noise_stream, uint64_t row_offset, float *out,
                               int64_t n_rows, int channels, int out_h, int out_w, const float *z_rows,
                               int64_t rows_per_z, void *stream);
int mnf_conv2d_forward_tc_z(const float *x, const float *z, const float *z_rows, int64_t rows_per_z,
                            const float *W_mean, const float *W_log_var, const float *b_log_var, const float *eps,
                            uint64_t seed, uint32_t noise_stream, uint64_t row_offset, float *out, int64_t n_imgs,
                            int c_in, int height, int width, int c_out, int ksize, float *workspace, void *stream);
int64_t mnf_conv_tc_workspace(int64_t n_imgs, int c_in, int height, int width, int c_out, int ksize);
int mnf_conv2d_forward_tc(const float *x, const float *z, const float *W_mean, const float *W_log_var,
                          const float *b_log_var, const float *eps, uint64_t seed, uint32_t noise_stream,
                          uint64_t row_offset, float *out, int64_t n_imgs, int c_in, int height, int width,
                          int c_out, int ksize, float *workspace, void *stream);
int mnf_conv_tc_stage(const float *x, const float *z, const float *W_mean, const float *W_log_var,
                      const float *b_log_var, float *a_mean, float *a_var, float *Bm, float *Bv, float *bvar_p,
                      int64_t n_imgs, int c_in, int height, int width, int c_out, int ksize, int Np, int Kp,
                      void *stream);

/* Weight-space part of MNFLinear.kl_div (mnf_linear.py:66-90, conv = 0) and MNFConv2d.kl_div
 * (mnf_conv.py:90-133, conv = 1).  z / ld_q come from sample_z (flow_q), zT / ld_r from
 * flow_r.forward(z); both are produced by mnf_rnvp_forward with one row.  out[0] is the KL
 * estimate; out[1..4] = kl_W, kl_b, log_q, log_r.  workspace: 2 * max(n_out, n_in*k*k) floats. */
typedef struct mnf_kl_args {
    int32_t conv, n_out, n_in, ksize; /* linear: ksize = 1                                     */
    const float *W_mean, *W_log_var;  /* [n_out, n_in, k, k]                                   */
    const float *b_mean;              /* linear only (conv: the reference's b_mean is zero)    */
    const float *b_log_var;           /* [n_out]                                               */
    const float *q0_log_var, *r0_c, *r0_b1, *r0_b2; /* [n_in] linear / [n_out] conv            */
    const float *z, *zT;              /* [n_in] linear / [n_out] conv                          */
    const float *ld_q, *ld_r;         /* device scalars                                        */
    const float *eps_w;               /* linear: [n_out, n_in]; conv: [n_in*k*k]; NULL = Philox */
    const float *eps_b;               /* conv: scalar; NULL = Philox                           */
    uint64_t seed;
    uint32_t noise_stream;
    float *workspace;
    float *out;                       /* [5]                                                   */
} mnf_kl_args;
int mnf_kl_div(const mnf_kl_args *args_host, void *stream);

/* The whole kl_div() of a layer (mnf_linear.py:66-90 / mnf_conv.py:90-133) in THREE launches: one thread-block cluster
 * draws z0 = q0_mean + sqrt(exp(q0_log_var)) eps_z and runs flow_q (-> z, ld_q) and flow_r (-> zT, ld_r) on that single
 * row, then the weight pass and the final reduction of mnf_kl_div.  Needs single-Linear RNVP conditioners of width <= 64
 * and at most MNF_KL_MAX_FLOWS flows per stack (otherwise: mnf_sample_z0 + mnf_rnvp_forward + mnf_kl_div).
 *   kl        as for mnf_kl_div, except that kl.z, kl.zT ([n_in] linear / [n_out] conv) and kl.ld_q, kl.ld_r ([1]) are
 *             OUTPUT buffers of this call; kl.workspace: 2 * max(n_out, n_in*k*k) + 64 floats.
 *   eps_z     injected z0 noise or NULL (Philox stream z_stream); masks[f]: injected Bernoulli mask of flow f or NULL
 *             (Philox stream mask_streams[f]); flows / masks / mask_streams hold flow_q's flows first, then flow_r's. */
#define MNF_KL_MAX_FLOWS 4
typedef struct mnf_kl_fused_args {
    mnf_kl_args kl;
    const float *q0_mean;
    const float *eps_z;
    uint32_t z_stream;
    int32_t n_flows_q, n_flows_r, reserved;
    mnf_rnvp_flow flows[2 * MNF_KL_MAX_FLOWS];
    const float *masks[2 * MNF_KL_MAX_FLOWS];
    uint32_t mask_streams[2 * MNF_KL_MAX_FLOWS];
} mnf_kl_fused_args;
int mnf_kl_div_fused(const mnf_kl_fused_args *args_host, void *stream);
/* The same for n_layers layers at once (MNFLeNet.kl_div sums four, mnf_lenet.py:28-32): still three launches -- the
 * layers are independent and each one's flow kernel is latency-bound on 8 SMs, so they run side by side.  layers[l] as
 * for mnf_kl_div_fused (host array of host pointers); every layer writes its own kl.out[5]. */
int mnf_kl_div_fused_multi(const mnf_kl_fused_args *const *layers_host, int n_layers, void *stream);

/* ------------------------------------------------------------------------------------
 * Training path of the MNF layers (SURVEY.md 8f-1).  The reference differentiates MNFLinear.forward /
 * kl_div with torch autograd (tests/test_mnf_mnist.py:28-43: loss = nll + 1e-3 kl_div, loss.backward());
 * the drop-in modules' autograd Functions (torch_mnf/layers/_train.py) are built from these exact-fp32
 * primitives.  Row-major everywhere; every pointer is a device pointer.
 * ---------------------------------------------------------------------------------- */
/* C[M,N] = op(A)[M,K] op(B)[K,N] + bias[N] (optional) + beta C.  trans_a: A is stored [K,M] with leading
 * dimension lda, else [M,K]; trans_b: B is stored [N,K] (torch's Linear.weight), else [K,N]. */
int mnf_gemm_f32(int trans_a, int trans_b, int64_t M, int N, int K, const float *A, int64_t lda, const float *B,
                 int64_t ldb, const float *bias, float beta, float *C, int64_t ldc, void *stream);

enum mnf_ew_op {
    MNF_EW_MUL = 1,        /* out = a b                                                                    */
    MNF_EW_MUL_ROWVEC = 2, /* out = a b[col]                       (W_mean * z, mnf_linear.py:69)           */
    MNF_EW_FMA = 3,        /* out = a + b c                                                                */
    MNF_EW_SQUARE = 4,     /* out = a^2                            (x**2, mnf_linear.py:54)                 */
    MNF_EW_EXP = 5,        /* out = exp(a)                         (W_log_var.exp(), :51)                   */
    MNF_EW_LEAKY = 6,      /* out = LeakyReLU_0.2(a)               (models/mlp.py:9)                        */
    MNF_EW_LEAKY_BWD = 7,  /* out = a (b > 0 ? 1 : 0.2)            a = gradient, b = pre-activation         */
    MNF_EW_NOISE_OUT = 8,  /* out = a + sqrt(b) c                  (mean + var.sqrt() * eps, :57)           */
    MNF_EW_GVAR = 9,       /* out = a c / (2 sqrt(b))              d loss / d var from d loss / d out       */
    MNF_EW_LIN_IN_BWD = 10,/* out = a c + 2 d b, out2 = a d        a = d/d(xz), b = d/d(x^2), c = z, d = x  */
    MNF_EW_Z0 = 11,        /* out = a[col] + exp(b[col] / 2) c     (q0_mean + q0_std * eps, :62-64)         */
    MNF_EW_MUL_COLVEC = 12,/* out = a b[row]                       (W_mean * z.view(-1,1,1,1), mnf_conv.py:73) */
    MNF_EW_ADD_2MUL = 13,  /* out = a + 2 b c                      d/dx of the x^2 branch added to the x branch */
    MNF_EW_ADD_COLVEC = 14,/* out = a + b[row]                     (conv bias in the [c_out, pixels] GEMM layout) */
    MNF_EW_RELU = 15,      /* out = max(a, 0)                      (nn.ReLU between MaskedLinears, made.py:43)      */
    MNF_EW_RELU_BWD = 16,  /* out = b > 0 ? a : 0                  a = gradient, b = pre-activation                 */
};
/* n elements; operands not used by `op` may be NULL; [col] operands are vectors of ncols entries. */
int mnf_ew(int op, const float *a, const float *b, const float *c, const float *d, float *out, float *out2, int64_t n,
           int ncols, void *stream);
/* out[n] = sum_r a[r,n] * (b ? b[r,n] : 1) */
int mnf_colsum(const float *a, const float *b, int64_t n_rows, int n_cols, float *out, void *stream);

/* MNFConv2d as GEMM (mnf_conv.py:68-79; stride 1, no padding).  cols_t[(ci,kh,kw)][(r,oh,ow)] = x[r,ci,oh+kh,ow+kw], so
 * conv(x, W)[c_out, (r,oh,ow)] = W[c_out, fan] cols_t; mnf_col2im_t is the adjoint (d loss / d x from d loss / d cols_t);
 * mnf_swap01 turns [dim0, dim1, inner] into [dim1, dim0, inner] (GEMM layout <-> NCHW); mnf_rowsum: out[r] = sum_c a[r,c]. */
int mnf_im2col_t(const float *x, float *cols_t, int64_t n_imgs, int c_in, int height, int width, int ksize, void *stream);
int mnf_col2im_t(const float *grad_cols_t, float *grad_x, int64_t n_imgs, int c_in, int height, int width, int ksize,
                 void *stream);
int mnf_swap01(const float *in, float *out, int64_t dim0, int64_t dim1, int64_t inner, void *stream);
int mnf_rowsum(const float *a, int64_t n_rows, int64_t n_cols, float *out, void *stream);

/* RNVP.forward after the conditioner (rnvp.py:33-40): gate = sigmoid(scale), z_out = (1-mask) z gate +
 * (1-gate) shift + mask z, log_det[row] = sum (1-mask) log(gate); and its adjoint (grad_z holds only the direct
 * path, the caller adds mask * d loss / d(mask z) coming back through the conditioner). */
int mnf_rnvp_gate_forward(const float *z, const float *mask, const float *shift, const float *scale, float *z_out,
                          float *log_det, int64_t n_rows, int dim, void *stream);
int mnf_rnvp_gate_backward(const float *z, const float *mask, const float *shift, const float *scale,
                           const float *grad_out, const float *grad_log_det, float *grad_shift, float *grad_scale,
                           float *grad_z, int64_t n_rows, int dim, void *stream);

/* Weight-sized part of MNFLinear.kl_div (mnf_linear.py:67-79) with injected eps_w [n_out, n_in]:
 *   pre[j] = sum_i (W_mean[j,i] z_i + exp(W_log_var[j,i]/2) eps_w[j,i]) r0_c[i]   (the tanh argument, :77)
 *   kl_rows[j] = 0.5 sum_i (-W_log_var + exp(W_log_var) + (W_mean z)^2 - 1)       (kl_div_W = sum_j, :72)
 * and the adjoint (grad_W_* overwritten, grad_z / grad_r0_c overwritten). */
int mnf_kl_rows_forward(const float *z, const float *W_mean, const float *W_log_var, const float *r0_c, const float *eps_w,
                        float *pre, float *kl_rows, int n_out, int n_in, void *stream);
int mnf_kl_rows_backward(const float *z, const float *W_mean, const float *W_log_var, const float *r0_c,
                         const float *eps_w, const float *grad_pre, const float *grad_kl_rows, float *grad_W_mean,
                         float *grad_W_log_var, float *grad_z, float *grad_r0_c, int n_out, int n_in, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* MNF_B200_H */
