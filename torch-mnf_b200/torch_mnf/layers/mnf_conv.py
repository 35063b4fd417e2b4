"""Multiplicative-normalizing-flow 2-D convolution (reference: layers/mnf_conv.py:10-133)."""

from collections.abc import Sequence

import torch
from torch import nn

from .. import _lib, flows
from .._program import state_without_caches
from . import _mnf_ops as ops
from . import _train


def _check_int(name, value, least):
    if not isinstance(value, int) or isinstance(value, bool):
        raise TypeError(f"MNFConv2d: {name} must be an int, got {value!r}")
    if value < least:
        raise ValueError(f"MNFConv2d: {name} must be >= {least}, got {value}")
    return value


class MNFConv2d(nn.Module):
    """Bayesian conv layer.  One z [n_out] per call, shared by the batch, scales the output channels
    of the mean path; out = conv(x, W_mean*z) + sqrt(conv(x^2, exp(W_log_var)) + exp(b_log_var)) * eps,
    computed as one implicit-GEMM CUDA kernel.  ``padding`` (zeros), ``stride``, ``dilation`` and
    ``groups`` mean what they mean for ``torch.nn.functional.conv2d``; the reference has none of them
    (padding=0, stride=1, dilation=1, groups=1).  Padding, stride and dilation are geometry, not
    parameters: the state_dict and kl_div do not depend on them.  ``groups`` splits the channels
    into groups that do not mix: W_mean / W_log_var are [n_out, n_in // groups, k, k].
    ``b_mean`` is a fixed zero tensor and not part of the state_dict, as in the reference."""

    __getstate__ = state_without_caches  # copy.deepcopy / pickle drop cached device scratch

    def __init__(self, n_in: int, n_out: int, kernel_size: int, n_flows_q: int = 2, n_flows_r: int = 2,
                 h_sizes: Sequence[int] = (50,), *, padding: int = 0, stride: int = 1, dilation: int = 1,
                 groups: int = 1) -> None:
        super().__init__()
        self.padding, self.stride = _check_int("padding", padding, 0), _check_int("stride", stride, 1)
        self.dilation, self.groups = _check_int("dilation", dilation, 1), _check_int("groups", groups, 1)
        if n_in % groups or n_out % groups:
            raise ValueError(f"MNFConv2d: groups={groups} must divide n_in={n_in} and n_out={n_out}")
        self.n_in, self.n_out, self.kernel_size = n_in, n_out, kernel_size
        shape = [n_out, n_in // groups, kernel_size, kernel_size]
        self.W_mean = nn.Parameter(0.1 * torch.randn(shape))
        self.W_log_var = nn.Parameter(-9 + 0.1 * torch.randn(shape))
        self.register_buffer("b_mean", torch.zeros(n_out), persistent=False)
        self.b_log_var = nn.Parameter(-9 + 0.1 * torch.randn(n_out))
        self.q0_mean = nn.Parameter(0.1 * torch.randn(n_out))
        self.q0_log_var = nn.Parameter(-9 + 0.1 * torch.randn(n_out))
        self.r0_c = nn.Parameter(0.1 * torch.randn(n_out))
        self.r0_b1 = nn.Parameter(0.1 * torch.randn(n_out))
        self.r0_b2 = nn.Parameter(0.1 * torch.randn(n_out))
        self.flow_q = flows.NormalizingFlow([flows.RNVP(n_out, h_sizes=h_sizes) for _ in range(n_flows_q)])
        self.flow_r = flows.NormalizingFlow([flows.RNVP(n_out, h_sizes=h_sizes) for _ in range(n_flows_r)])

    def extra_repr(self) -> str:
        s = f"{self.n_in}, {self.n_out}, kernel_size={self.kernel_size}, padding={self.padding}, stride={self.stride}"
        if self.dilation != 1:
            s += f", dilation={self.dilation}"
        if self.groups != 1:
            s += f", groups={self.groups}"
        return s

    def output_size(self, height: int, width: int) -> tuple[int, int]:
        """(OH, OW) of this layer on height x width inputs; ValueError when the output would be empty."""
        p, s = self.padding, self.stride
        k = self.dilation * (self.kernel_size - 1) + 1  # extent of the dilated filter
        if height + 2 * p < k or width + 2 * p < k:
            raise ValueError(f"MNFConv2d: kernel_size {self.kernel_size} (extent {k} at dilation {self.dilation}) "
                             f"is larger than the {height}x{width} input padded by {p}")
        return (height + 2 * p - k) // s + 1, (width + 2 * p - k) // s + 1

    def sample_z(self, noise=None):
        """-> (z [1, n_out], log_det_q)."""
        dev = self.W_mean.device
        if dev.type != "cuda":
            raise RuntimeError("torch_mnf (B200) runs only on CUDA parameters (no CPU fallback)")
        if _train.needs_grad(self):  # differentiable, like the reference's (mnf_conv.py:80-88 under autograd)
            z, ld = _train.sample_z(self, -1, _train._tape(noise, dev), self.n_out)
            return z, ld.squeeze()
        noise = noise if isinstance(noise, ops.Noise) else ops.Noise(noise, dev)
        # z is ONE draw shared by the whole call (mnf_conv.py:80-88): it must not depend on which shard of the
        # rows this rank owns, so it is drawn at row offset 0 whatever the caller's offset is
        keep, noise.row_offset = noise.row_offset, 0
        try:
            z = ops.sample_z0(self.q0_mean, self.q0_log_var, -1, noise)
            ld, _ = ops.rnvp_stack_inplace(list(self.flow_q.flows), z, noise)
        finally:
            noise.row_offset = keep
        return z, ld.squeeze()

    def forward(self, x, noise=None, row_offset=0, relu_pool=False, n_imgs=None):
        """relu_pool=True fuses the ReLU + MaxPool2d(2) that follow this layer in MNFLeNet;
        n_imgs > len(x) replicates the images (image r reads x[r % len(x)])."""
        if isinstance(x, torch.Tensor) and x.dim() == 4:
            self.output_size(x.size(2), x.size(3))  # argument errors before any device work
        if _train.needs_grad(self, x):  # training: differentiable exact-fp32 path (layers/_train.py)
            if n_imgs is not None and n_imgs != x.size(0):
                x = x.repeat(n_imgs // x.size(0), 1, 1, 1)
            return _train.conv_forward(self, x, noise, relu_pool)
        x = _lib.require_cuda_f32(x, "input")
        noise = noise if isinstance(noise, ops.Noise) else ops.Noise(noise, x.device, row_offset)
        z, _ = self.sample_z(noise)
        return ops.conv_forward(self, x, z, noise, n_imgs=n_imgs, relu_pool=relu_pool)

    def kl_div(self, noise=None):
        if _train.needs_grad(self):
            return _train.conv_kl_div(self, noise)
        return ops.kl_div(self, conv=True, tape=noise)
