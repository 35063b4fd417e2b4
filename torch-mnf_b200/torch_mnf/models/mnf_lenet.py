"""Bayesian LeNet built from MNF layers (reference: models/mnf_lenet.py:8-32)."""

from typing import Any

import torch
from torch import nn

from .. import _lib
from ..layers import MNFConv2d, MNFLinear
from ..layers import _mnf_ops as ops
from ..layers import _train
from .mnf_feed_forward import check_mc_args, uncertainty_from_sums


class MNFLeNet(nn.Sequential):
    """MNFConv2d(1,20,5) -> ReLU -> MaxPool2 -> MNFConv2d(20,50,5) -> ReLU -> MaxPool2 -> Flatten ->
    MNFLinear(800,50) -> ReLU -> MNFLinear(50,10) -> LogSoftmax, with the reference's Sequential
    indices (MNF layers at 0, 3, 7, 9) so its state_dict loads unchanged.

    ``forward`` runs the CUDA pipeline: each conv kernel applies its noise, ReLU and 2x2 max-pool in
    the epilogue (the un-pooled activations never reach HBM), the linear kernels fuse bias, noise and
    ReLU.  ``noise`` injects a tape (16 draws in the reference's order); ``n_samples`` evaluates
    ``forward(x.repeat(n_samples, 1, 1, 1))`` -- the Monte-Carlo prediction of mnf_mnist.ipynb:316-318
    -- without materialising the repeat."""

    def __init__(self, **kwargs: Any) -> None:
        super().__init__(
            MNFConv2d(1, 20, kernel_size=5, **kwargs), nn.ReLU(), nn.MaxPool2d(kernel_size=2),
            MNFConv2d(20, 50, kernel_size=5, **kwargs), nn.ReLU(), nn.MaxPool2d(kernel_size=2),
            nn.Flatten(),
            MNFLinear(50 * 16, 50, **kwargs), nn.ReLU(),
            MNFLinear(50, 10, **kwargs), nn.LogSoftmax(dim=-1),
        )

    #: "auto": batches of >= TC_MIN_ROWS rows take the Monte-Carlo pipeline (conv1 moments once per image, conv2 and
    #: fc1 on TF32 tensor cores; tolerance class 2e-3); "fp32": exact-fp32 kernels throughout
    precision = "auto"
    TC_MIN_ROWS = 512

    def forward(self, x, noise=None, n_samples: int = 1, row_offset: int = 0, seed=None,
                per_sample_conv_z: bool = False):
        """per_sample_conv_z (SURVEY 8f-4): every Monte-Carlo sample draws its own z for the two conv layers -- what
        ``n_samples`` separate reference calls would do (mnf_conv.py:80-88 draws one z per CALL) -- instead of sharing
        one z across the whole replicated batch as ``model(x.repeat(n_samples, 1, 1, 1))`` does.  Draw order in this
        mode, per conv layer: normal[S, n_out], one Bernoulli[S, n_out] per q-flow, normal[R, n_out, OH, OW]."""
        x = _lib.require_cuda_f32(x, "input")
        if per_sample_conv_z and not _train.needs_grad(self, x):
            return self._forward_per_sample_z(x, noise, n_samples, row_offset, seed)
        if _train.needs_grad(self, x):  # training: every layer takes its differentiable path, one shared tape
            tape = _train._tape(noise, x.device)
            h = x.repeat(n_samples, 1, 1, 1) if n_samples > 1 else x
            h = _train.conv_forward(self[0], h, tape, relu_pool=True)
            h = _train.conv_forward(self[3], h, tape, relu_pool=True)
            h = _train.linear_forward(self[7], h.flatten(1), tape, relu=True)
            return torch.log_softmax(_train.linear_forward(self[9], h, tape), dim=-1)
        R = x.size(0) * n_samples
        nz = ops.Noise(noise, x.device, row_offset, seed=seed)
        if self.precision != "fp32" and R >= self.TC_MIN_ROWS:
            z1, _ = self[0].sample_z(nz)
            h = ops.conv_mc_relu_pool(self[0], x, z1, nz, R)
            z2, _ = self[3].sample_z(nz)
            h = ops.conv_forward_tc(self[3], h, z2, nz)
        else:
            h = self[0].forward(x, nz, relu_pool=True, n_imgs=R)
            h = self[3].forward(h, nz, relu_pool=True)
        h = h.view(R, -1)
        prec = "fp32" if self.precision == "fp32" else None
        h = self[7].forward(h, nz, relu=True, precision=prec)
        h = self[9].forward(h, nz, precision=prec)
        return torch.log_softmax(h, dim=-1)

    def _forward_per_sample_z(self, x, noise, S, row_offset, seed, conv1=None):
        """conv1: conv_moments(self[0], x, None) when the caller already has them (they do not depend on the sample)."""
        B = x.size(0)
        R = B * S
        if row_offset % B:
            raise ValueError("per-sample conv z: row_offset must be a multiple of the image count (whole samples per shard)")
        nz = ops.Noise(noise, x.device, row_offset, seed=seed)
        s0 = row_offset // B  # global index of this shard's first Monte-Carlo sample
        # conv1: moments once per image with unit z (exact fp32), z[s, c] scales the mean in the noise / pool pass
        z1 = ops.conv_sample_z_rows(self[0], S, nz, s0)
        mean1, sd1 = conv1 if conv1 is not None else ops.conv_moments(self[0], x, None)
        h = ops.conv_noise_relu_pool(mean1, sd1, nz, R, z_rows=z1, rows_per_z=B)
        z2 = ops.conv_sample_z_rows(self[3], S, nz, s0)
        if self.precision != "fp32":
            h = ops.conv_forward_tc(self[3], h, None, nz, z_rows=z2, rows_per_z=B)
        else:  # exact fp32: one launch per sample, each with its own z and its slice of the noise draw
            c_out = self[3].n_out
            eps, sid = nz.normal((R, c_out, 8, 8))
            out = torch.empty((R, c_out, 4, 4), device=x.device, dtype=torch.float32)
            for s in range(S):
                ops.conv_forward(self[3], h[s * B:(s + 1) * B], z2[s], nz, relu_pool=True,
                                 drawn=(None if eps is None else eps[s * B:(s + 1) * B], sid, nz.row_offset + s * B),
                                 out=out[s * B:(s + 1) * B])
            h = out
        h = h.view(R, -1)
        prec = "fp32" if self.precision == "fp32" else None
        h = self[7].forward(h, nz, relu=True, precision=prec)
        h = self[9].forward(h, nz, precision=prec)
        return torch.log_softmax(h, dim=-1)

    @torch.no_grad()
    def predict(self, x, n_samples: int = 500, chunk: int = 25, seed=None, sample_range=None):
        """Monte-Carlo predictive class probabilities ``[B, 10]``: the mean over ``n_samples`` stochastic forward passes of
        ``softmax(model(x))`` -- ``model(img.repeat(500, 1, 1, 1))`` followed by the mean over the copies in
        examples/mnf_mnist.ipynb:316-318 -- without materialising the repeat.  As in that single reference call the two conv
        layers draw ONE z each for the whole prediction (mnf_conv.py:80-88), so their sample-independent parts (z, conv1's
        mean / variance maps) are evaluated once instead of once per chunk of samples; everything per-row is drawn with
        Philox keyed by the global row (sample s, image b), so the result does not depend on ``chunk`` or on how the samples
        are sharded.  ``sample_range=(lo, hi)``: only samples lo..hi-1 and the SUM of their probabilities is returned (a
        rank's share under MC-sample sharding: all-reduce the sums, divide by n_samples -- torch_mnf.distributed).
        Identical, draw for draw, to summing ``forward(x, n_samples=chunk, seed=seed, row_offset=c * B).exp()`` over the chunks."""
        x = _lib.require_cuda_f32(x, "input")
        B = x.size(0)
        lo, hi = (0, n_samples) if sample_range is None else sample_range
        if seed is None:
            seed = int(torch.randint(0, 2**62, (1,)).item())  # follows torch.manual_seed
        sums = torch.zeros(B, 10, device=x.device, dtype=torch.float32)
        for s_here, log_probs in self._mc_log_probs(x, chunk, seed, lo, hi):
            sums += log_probs.exp().view(s_here, B, 10).sum(0)
        return sums if sample_range is not None else sums / n_samples

    @torch.no_grad()
    def predict_uncertainty(self, x, n_samples: int = 500, chunk: int = 25, seed=None, sample_range=None,
                            per_sample_conv_z: bool = False):
        """Monte-Carlo predictive uncertainty: an MCUncertainty with the mean and variance of the class probabilities
        ``[B, 10]`` and, per image, the predictive entropy H[p_bar] (total), the expected entropy E_s H[p_s] (aleatoric)
        and their difference, the mutual information (epistemic; BALD).  The samples and draws are ``predict``'s; each
        chunk's log-probabilities are reduced on the device into fp64 sums of the probabilities, their squares and the
        per-sample entropies (mnf_mc_class_moments), so ``mean`` agrees with ``predict`` to fp32 rounding and the result
        does not depend on ``chunk`` beyond fp64 rounding.  ``sample_range=(lo, hi)``: the raw ``(sums [2, B, 10],
        entropy_sums [B])`` of samples lo..hi-1; all-reduce both and finish with ``uncertainty_from_sums``.

        ``per_sample_conv_z``: every sample draws its own conv z, as ``forward(..., per_sample_conv_z=True)`` does chunk
        by chunk (bit for bit).  ``predict``'s single z per conv layer leaves the conv layers' multiplicative posterior
        out of the spread across samples, so the mutual information undercounts their epistemic part; this mode
        includes it, at the cost of one z draw per sample."""
        lo, hi = check_mc_args(n_samples, chunk, sample_range)
        x = _lib.require_cuda_f32(x, "input")
        B = x.size(0)
        if seed is None:
            seed = int(torch.randint(0, 2**62, (1,)).item())  # follows torch.manual_seed
        sums = torch.zeros((2, B, 10), device=x.device, dtype=torch.float64)
        entropy_sums = torch.zeros(B, device=x.device, dtype=torch.float64)
        for s_here, log_probs in self._mc_log_probs(x, chunk, seed, lo, hi, per_sample_conv_z):
            ops.mc_moments(log_probs, B, s_here, sums, softmax=True, entropy_sums=entropy_sums)
        if sample_range is not None:
            return sums, entropy_sums
        return uncertainty_from_sums(sums, entropy_sums, n_samples)

    def _mc_log_probs(self, x, chunk, seed, lo, hi, per_sample_conv_z=False):
        """Yields (s_here, log-probabilities [s_here * B, 10]) chunk by chunk for samples lo..hi-1: the draws of
        ``forward(x, n_samples=s_here, seed=seed, row_offset=c * B, per_sample_conv_z=...)`` per chunk c."""
        B = x.size(0)
        if per_sample_conv_z:  # conv1's unit-z moments do not depend on the sample: once per prediction
            conv1 = ops.conv_moments(self[0], x, None)
            for c in range(lo, hi, chunk):
                s_here = min(chunk, hi - c)
                yield s_here, self._forward_per_sample_z(x, None, s_here, c * B, seed, conv1=conv1)
            return
        if self.precision == "fp32" or B * min(chunk, max(hi - lo, 1)) < self.TC_MIN_ROWS:
            for c in range(lo, hi, chunk):  # exact-fp32 pipeline: nothing sample-independent to share across chunks
                s_here = min(chunk, hi - c)
                yield s_here, self.forward(x, n_samples=s_here, seed=seed, row_offset=c * B)
            return
        # the call's two conv z draws (row offset 0 on every rank) and conv1's moments: once
        nz0 = ops.Noise(None, x.device, 0, seed=seed)
        z1, _ = self[0].sample_z(nz0)
        mean1, sd1 = ops.conv_moments(self[0], x, z1)
        nz0._next_stream()  # conv1's noise draw (per chunk below)
        z2, _ = self[3].sample_z(nz0)
        n_z = 1 + len(self[0].flow_q.flows)  # noise streams one conv sample_z consumes: z0 + one mask per q-flow
        for c in range(lo, hi, chunk):
            s_here = min(chunk, hi - c)
            R = B * s_here
            nz = ops.Noise(None, x.device, c * B, seed=seed)
            nz.streams += n_z  # conv1's z: drawn above
            h = ops.conv_noise_relu_pool(mean1, sd1, nz, R)
            nz.streams += 1 + len(self[3].flow_q.flows)  # conv2's z: drawn above
            h = ops.conv_forward_tc(self[3], h, z2, nz)
            h = self[7].forward(h.view(R, -1), nz, relu=True)
            h = self[9].forward(h, nz)
            yield s_here, torch.log_softmax(h, dim=-1)

    def kl_div(self, noise=None):
        """Sum of the MNF layers' KL estimates (mnf_lenet.py:28-32).  Without an injected tape and outside autograd the
        four layers go through ONE call of three launches (mnf_kl_div_fused_multi: the layers are independent and each
        one's flow kernel is latency-bound, so they run side by side) -- same draws and values as the loop."""
        layers = [layer for layer in self if hasattr(layer, "kl_div")]
        if noise is None and not _train.needs_grad(self):
            total = ops.kl_div_multi(layers)
            if total is not None:
                return total
        return sum(layer.kl_div(noise) for layer in layers)
