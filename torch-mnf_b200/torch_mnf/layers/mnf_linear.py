"""Multiplicative-normalizing-flow linear layer (reference: layers/mnf_linear.py:7-90;
Louizos & Welling 2017, https://arxiv.org/abs/1703.01961)."""

import torch
from torch import nn

from .. import _lib, flows
from .._program import state_without_caches
from . import _mnf_ops as ops
from . import _train


class MNFLinear(nn.Module):
    """Bayesian affine layer.  ``forward(x)``: z ~ q0 pushed through the RNVP flow_q (one z per
    row), then the local-reparameterisation pair mean = (x*z) W_mean^T + b_mean,
    var = x^2 exp(W_log_var)^T + exp(b_log_var), out = mean + sqrt(var) * eps -- one fused CUDA
    GEMM kernel sharing the x tile.  ``kl_div()``: single-sample KL estimate with the auxiliary
    flow_r.  Parameter names / shapes / initialisation follow the reference.

    Additive options: ``noise=`` (a tape with ``normal(shape)`` / ``bernoulli(shape)``, consumed
    in the reference's draw order) for parity runs; ``forward_mc(x, n_samples)`` evaluates
    ``forward(x.repeat(n_samples, 1))`` without materialising the repeat."""

    #: "auto" (TF32 tensor cores for large aligned shapes, exact fp32 otherwise), "fp32" or "tf32"
    precision = "auto"

    __getstate__ = state_without_caches  # copy.deepcopy / pickle drop cached device scratch

    def __init__(self, n_in, n_out, n_flows_q=2, n_flows_r=2, h_sizes=(50,)):
        super().__init__()
        self.n_in, self.n_out = n_in, n_out
        self.W_mean = nn.Parameter(0.1 * torch.randn([n_out, n_in]))
        self.W_log_var = nn.Parameter(-9 + 0.1 * torch.randn([n_out, n_in]))
        self.b_mean = nn.Parameter(torch.zeros(n_out))
        self.b_log_var = nn.Parameter(-9 + 0.1 * torch.randn(n_out))
        self.q0_mean = nn.Parameter(0.1 * torch.randn(n_in))
        self.q0_log_var = nn.Parameter(-9 + 0.1 * torch.randn(n_in))
        self.r0_c = nn.Parameter(0.1 * torch.randn(n_in))
        self.r0_b1 = nn.Parameter(0.1 * torch.randn(n_in))
        self.r0_b2 = nn.Parameter(0.1 * torch.randn(n_in))
        self.flow_q = flows.NormalizingFlow([flows.RNVP(n_in, h_sizes=h_sizes) for _ in range(n_flows_q)])
        self.flow_r = flows.NormalizingFlow([flows.RNVP(n_in, h_sizes=h_sizes) for _ in range(n_flows_r)])

    def _noise(self, noise, device, row_offset=0):
        return noise if isinstance(noise, ops.Noise) else ops.Noise(noise, device, row_offset)

    def sample_z(self, batch_size=1, noise=None, row_offset=0):
        """z_T = flow_q(q0_mean + sqrt(exp(q0_log_var)) * eps) -> (z [B, n_in], log_det_q)."""
        dev = self.W_mean.device
        if dev.type != "cuda":
            raise RuntimeError("torch_mnf (B200) runs only on CUDA parameters (no CPU fallback)")
        if _train.needs_grad(self):  # differentiable, like the reference's (mnf_linear.py:58-64 under autograd)
            z, ld = _train.sample_z(self, batch_size, _train._tape(noise, dev), self.n_in)
            return z, ld.squeeze()
        noise = self._noise(noise, dev, row_offset)
        z = ops.sample_z0(self.q0_mean, self.q0_log_var, batch_size, noise)
        ld, _ = ops.rnvp_stack_inplace(list(self.flow_q.flows), z, noise)
        return z, ld.squeeze()

    def _forward_rows(self, x, n_rows, noise, relu, precision=None, affine=None):
        """forward over n_rows output rows, row r reading x[r % len(x)].  affine: optional (col_scale, col_shift)
        [n_out] applied after the ReLU in the kernel epilogue (a folded eval-mode BatchNorm1d)."""
        precision = precision or self.precision
        flows_q = list(self.flow_q.flows)
        if ops.use_tensor_cores(self, n_rows, precision) and ops.rnvp_tc_ok(flows_q, self.n_in):
            # all-tensor-core pipeline: the last RNVP epilogue leaves tf32(x*z) where the mean GEMM expects it
            ws = torch.empty(_lib.lib().mnf_linear_tc_workspace(x.size(0), n_rows, self.n_in, self.n_out),
                             device=x.device, dtype=torch.float32)
            ok4 = self.n_in % 4 == 0 and (noise.row_offset * self.n_in) % 16 == 0
            if ok4:  # z0 drawn inside the RNVP call (one pass less over z)
                ops.rnvp_stack_tc(flows_q, None, noise, x=x, x_rows=x.size(0), xz_out=ws,
                                  q0=(self.q0_mean, self.q0_log_var), n_rows=n_rows, z_is_scratch=True)
            else:
                z = ops.sample_z0(self.q0_mean, self.q0_log_var, n_rows, noise)
                ops.rnvp_stack_tc(flows_q, z, noise, x=x, x_rows=x.size(0), xz_out=ws, z_is_scratch=True)
            return ops.linear_forward(self, x, None, noise, x_rows=x.size(0), relu=relu, staged_ws=ws, n_rows=n_rows,
                                      affine=affine)
        z, _ = self.sample_z(n_rows, noise)
        return ops.linear_forward(self, x, z, noise, x_rows=x.size(0), relu=relu, precision=precision, affine=affine)

    def forward(self, x, noise=None, row_offset=0, relu=False, precision=None):
        if _train.needs_grad(self, x):  # training: differentiable exact-fp32 path (layers/_train.py)
            return _train.linear_forward(self, x, noise, relu)
        x = _lib.require_cuda_f32(x, "input")
        return self._forward_rows(x, x.size(0), self._noise(noise, x.device, row_offset), relu, precision)

    def forward_mc(self, x, n_samples, noise=None, row_offset=0, relu=False):
        """== forward(x.repeat(n_samples, 1)): row r uses x[r % len(x)], own z and eps per row."""
        x = _lib.require_cuda_f32(x, "input")
        return self._forward_rows(x, x.size(0) * n_samples, self._noise(noise, x.device, row_offset), relu)

    def _function_noise(self, noise, seed, device):
        """Noise of a function-sample call: ``noise`` (a tape or an ops.Noise) as given, else Philox keyed by ``seed``
        (drawn from torch's generator when None; a device tape under CUDA-graph capture, as ops.Noise does)."""
        return noise if isinstance(noise, ops.Noise) else ops.Noise(noise, device, seed=seed)

    @torch.no_grad()
    def sample_weights(self, n_samples, seed=None, sample_offset=0, noise=None):
        """``n_samples`` draws of the layer's weights from the posterior: (W [S, n_out, n_in], b [S, n_out]) with
        W_s = W_mean * z_s[None, :] + exp(0.5 W_log_var) * E_s and b_s = b_mean + exp(0.5 b_log_var) * e_s, z_s row s
        of sample_z(S).  Draws, in order: normal[S, n_in] and one Bernoulli[S, n_in] per q-flow (sample_z with
        row_offset = sample_offset), normal[S, n_out, n_in] (E), normal[S, n_out] (e).  Philox elements are keyed by
        ``(seed, sample_offset + s)``, so a sample does not depend on how the samples are split between calls."""
        ops.check_function_args(n_samples, sample_offset)
        dev = self.W_mean.device
        if dev.type != "cuda":
            raise RuntimeError("torch_mnf (B200) runs only on CUDA parameters (no CPU fallback)")
        noise = self._function_noise(noise, seed, dev)
        z = ops.linear_function_z(self, int(n_samples), noise, int(sample_offset))
        return ops.linear_sample_weights(self, z, noise, int(sample_offset))

    @torch.no_grad()
    def forward_functions(self, x, n_samples, seed=None, sample_offset=0, noise=None, relu=False):
        """The layer under ``n_samples`` posterior weight draws (those of ``sample_weights``): [S, B, n_out] with
        out[s] = x_s @ W_s^T + b_s, every input row of sample s through the same W_s, b_s.  x: [B, n_in], shared by the
        samples, or [S, B, n_in], one block per sample.  ``relu`` applies a ReLU in the GEMM's epilogue.  Exact fp32
        whatever ``precision`` says.  Row s * B + b of ``out.view(S * B, n_out)`` is sample s of input b, the layout of
        forward_mc."""
        ops.check_function_args(n_samples, sample_offset)
        x = ops.function_input(x, self.n_in, int(n_samples))
        return self._functions(x, int(n_samples), self._function_noise(noise, seed, x.device), int(sample_offset),
                               relu)

    def _functions(self, x, n_samples, noise, sample_offset, relu=False, affine=None, chunk=None):
        """forward_functions on a Noise: z of all samples in one draw, then chunk by chunk the weight image
        (mnf_linear_sample_weights) and the function GEMM.  Without a tape every chunk takes the same two stream ids
        for E and e, its Philox elements keyed by its global samples; a tape is consumed in one chunk.  affine: the
        folded batch norm of the GEMM's epilogue."""
        if noise.tape is not None:
            chunk = n_samples
        elif chunk is None:
            chunk = ops.function_chunk(self.n_out * (self.n_in + 1))
        z = ops.linear_function_z(self, n_samples, noise, sample_offset)
        out = torch.empty((n_samples, x.size(-2), self.n_out), device=x.device, dtype=torch.float32)
        weight_stream = noise.streams
        for c in range(0, n_samples, chunk):
            k = min(chunk, n_samples - c)
            noise.streams = weight_stream
            W, b = ops.linear_sample_weights(self, z[c:c + k], noise, sample_offset + c)
            ops.linear_function_forward(x[c:c + k] if x.dim() == 3 else x, W, b, relu, affine, out=out[c:c + k])
        return out

    def kl_div(self, noise=None):
        if _train.needs_grad(self):
            return _train.linear_kl_div(self, noise)
        return ops.kl_div(self, conv=False, tape=noise)
