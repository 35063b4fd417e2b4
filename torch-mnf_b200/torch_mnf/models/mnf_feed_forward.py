"""Feed-forward net of MNFLinear layers (reference: models/mnf_feed_forward.py:14-38)."""

from collections.abc import Sequence
from typing import Any, NamedTuple

import torch
from torch import nn

from .. import _lib
from .._program import state_without_caches
from ..layers import MNFLinear
from ..layers import _mnf_ops as ops
from ..layers import _train


def fold_batch_norm(bn: nn.BatchNorm1d) -> tuple[torch.Tensor, torch.Tensor]:
    """The eval-mode ``bn`` as a per-column affine map ``y = scale * h + shift``: scale = weight / sqrt(running_var + eps),
    shift = bias - running_mean * scale (weight 1 and bias 0 without ``affine``) -- the folded coefficients of
    inference batch norm.  fp32, contiguous, on the buffers' device."""
    with torch.no_grad():
        var, mean = bn.running_var.float(), bn.running_mean.float()
        w = bn.weight.detach().float() if bn.weight is not None else torch.ones_like(var)
        b = bn.bias.detach().float() if bn.bias is not None else torch.zeros_like(mean)
        scale = w / torch.sqrt(var + bn.eps)
        return scale.contiguous(), (b - mean * scale).contiguous()


def moments_from_sums(sums: torch.Tensor, n_samples: int) -> tuple[torch.Tensor, torch.Tensor]:
    """(mean, var) [B, n_out] fp32 from the fp64 sums [2, B, n_out] of ``MNFFeedForward.predict(sample_range=...)``
    (all ranks' shares added): mean = S1 / S, population variance = S2 / S - mean^2, clamped at 0 (rounding can leave
    a tiny negative value where all samples agree)."""
    mean = sums[0] / n_samples
    var = (sums[1] / n_samples - mean * mean).clamp_min_(0.0)
    return mean.float(), var.float()


class MCUncertainty(NamedTuple):
    """Monte-Carlo predictive uncertainty of a classifier over S samples p_s = softmax(model(x)) (natural log units):
    ``mean``, ``var`` [B, C] fp32: mean and population variance of the class probabilities;
    ``predictive_entropy`` [B]: H[p_bar], the total uncertainty;
    ``expected_entropy`` [B]: E_s H[p_s], the aleatoric part;
    ``mutual_information`` [B]: H[p_bar] - E_s H[p_s] (BALD), the epistemic part."""

    mean: torch.Tensor
    var: torch.Tensor
    predictive_entropy: torch.Tensor
    expected_entropy: torch.Tensor
    mutual_information: torch.Tensor


def check_mc_args(n_samples: int, chunk: int | None, sample_range) -> tuple[int, int]:
    """(lo, hi) of a Monte-Carlo prediction's samples; ValueError for n_samples < 1, chunk < 1 or a sample_range
    outside [0, n_samples] -- before any device work."""
    if n_samples < 1:
        raise ValueError(f"n_samples must be positive, got {n_samples}")
    if chunk is not None and chunk < 1:
        raise ValueError(f"chunk must be positive, got {chunk}")
    lo, hi = (0, n_samples) if sample_range is None else sample_range
    if not 0 <= lo <= hi <= n_samples:
        raise ValueError(f"sample_range {sample_range} outside [0, {n_samples}]")
    return lo, hi


def uncertainty_from_sums(sums: torch.Tensor, entropy_sums: torch.Tensor, n_samples: int) -> MCUncertainty:
    """MCUncertainty from the fp64 probability sums [2, B, C] and entropy sums [B] of ``predict_uncertainty(...,
    sample_range=...)`` (all ranks' shares added).  mean / var as moments_from_sums; H[p_bar] = -sum_c p_bar log p_bar in
    fp64 with 0 log 0 = 0; E_s H[p_s] = entropy_sums / S; the mutual information is clamped at 0 (rounding can leave a
    tiny negative value where all samples agree)."""
    mean, var = moments_from_sums(sums, n_samples)
    p_bar = sums[0] / n_samples
    predictive = -torch.special.xlogy(p_bar, p_bar).sum(-1)
    expected = entropy_sums / n_samples
    mutual = (predictive - expected).clamp_min_(0.0)
    return MCUncertainty(mean, var, predictive.float(), expected.float(), mutual.float())


class MNFFeedForward(nn.Sequential):
    """MNFLinear -> activation -> BatchNorm1d blocks; the final activation and batch norm are dropped.

    ``forward(x)`` is the plain ``nn.Sequential`` call.  ``forward_mc(x, n_samples)`` evaluates the model on
    ``x.repeat(n_samples, 1)`` without materialising the repeat, with ReLU and an eval-mode BatchNorm1d applied in the
    MNFLinear kernels' epilogues; ``predict(x, n_samples)`` reduces such samples to the predictive mean and variance."""

    __getstate__ = state_without_caches  # copy.deepcopy / pickle drop the folded batch-norm coefficients

    #: rows * widest layer per forward_mc chunk of predict() when ``chunk`` is not given (512 MB of fp32 activations per
    #: layer output): few, large chunks keep the layer GEMMs efficient, each chunk costs a full pass of launches
    CHUNK_FLOATS = 1 << 27

    def __init__(self, layer_sizes: Sequence[int], activation: type[nn.Module] = nn.ReLU, **kwargs: Any) -> None:
        mods = []
        for n_in, n_out in zip(layer_sizes[:-1], layer_sizes[1:]):
            mods += [MNFLinear(n_in, n_out, **kwargs), activation(), nn.BatchNorm1d(n_out)]
        super().__init__(*mods[:-2])

    def kl_div(self):
        return sum(layer.kl_div() for layer in self if hasattr(layer, "kl_div"))

    def _blocks(self):
        """(MNFLinear, activation or None, BatchNorm or None) per layer."""
        mods = list(self)
        return [(mods[i], *(mods[i + 1:i + 3] if i + 3 <= len(mods) else (None, None))) for i in range(0, len(mods), 3)]

    @staticmethod
    def _uses_running_stats(bn) -> bool:
        return not bn.training and bn.running_mean is not None and bn.running_var is not None

    def _folded(self, i, bn, dev):
        """fold_batch_norm(bn) on dev, cached while its parameters and buffers keep their storage and version."""
        tensors = [t for t in (bn.weight, bn.bias, bn.running_mean, bn.running_var) if t is not None]
        key = (str(dev), bn.eps, tuple((t.data_ptr(), t._version) for t in tensors))
        cache = self.__dict__.setdefault("_bn_fold", {})
        hit = cache.get(i)
        if hit is not None and hit[0] == key:
            return hit[1]
        if any(t.device != dev for t in tensors):
            raise RuntimeError(f"BatchNorm1d at block {i} is on {tensors[0].device} but the input is on {dev}")
        folded = fold_batch_norm(bn)
        cache[i] = (key, folded)
        return folded

    def forward_mc(self, x, n_samples: int, noise=None, seed=None, row_offset: int = 0):
        """== the model on ``x.repeat(n_samples, 1)`` (row s * B + b is sample s of input b), without the repeat.

        One noise source is shared by all layers; each layer draws as ``MNFLinear.forward`` on R = B * n_samples rows
        (normal[R, n_in], one Bernoulli[R, n_in] per q-flow, normal[R, n_out]), from the tape ``noise`` or from Philox
        keyed by ``(seed, row_offset + row)``, so calls on consecutive row blocks reproduce one call.  Hidden blocks with
        ``nn.ReLU`` and an eval-mode BatchNorm1d run both in the layer's kernel epilogue (the first layer reads ``x``
        through its B distinct rows).  Other activations, and batch norms that use batch statistics (training mode or no
        running stats), are applied by their modules after the layer -- a training-mode BatchNorm therefore normalises
        over all B * n_samples rows and updates its running stats, as the repeated call would.  With grad enabled and
        trainable parameters every layer takes its differentiable path (draws from the tape or torch's generator; ``seed``
        does not apply)."""
        x = _lib.require_cuda_f32(x, "input")
        if n_samples < 1:
            raise ValueError(f"n_samples must be positive, got {n_samples}")
        R = x.size(0) * n_samples
        if _train.needs_grad(self, x):
            tape = _train._tape(noise, x.device)
            h = x.repeat(n_samples, 1)
            for lin, act, bn in self._blocks():
                h = lin(h, noise=tape)
                if act is not None:
                    h = bn(act(h))
            return h
        nz = ops.Noise(noise, x.device, row_offset, seed=seed)
        h = x
        for i, (lin, act, bn) in enumerate(self._blocks()):
            relu = type(act) is nn.ReLU
            affine = self._folded(i, bn, x.device) if relu and self._uses_running_stats(bn) else None
            h = lin._forward_rows(h, R, nz, relu=relu, affine=affine)
            if act is not None and affine is None:
                h = bn(h if relu else act(h))
        return h

    @torch.no_grad()
    def predict(self, x, n_samples: int = 500, chunk: int | None = None, seed=None, sample_range=None,
                softmax: bool = False):
        """Monte-Carlo predictive moments over ``n_samples`` stochastic passes: ``(mean, var)``, each [B, n_out] fp32,
        of the outputs -- or, with ``softmax``, of the class probabilities ``softmax(model(x))``.  ``var`` is the
        population variance over the samples: the model's predictive uncertainty.

        Samples run ``chunk`` at a time through ``forward_mc`` (default: about CHUNK_FLOATS activations per chunk) with
        Philox keyed by ``(seed, global row)``, and each chunk is reduced on the device into fp64 sums of the values and
        their squares.  So the result does not depend on ``chunk`` beyond fp64 rounding.  ``sample_range=(lo, hi)``: only
        samples lo..hi-1, and the raw fp64 sums [2, B, n_out] are returned -- a rank's share under sample sharding;
        all-reduce the shares and finish them with ``moments_from_sums(sums, n_samples)``, the formula this call uses.
        Shares that each hold one chunk, added in sample order, give the bits of the unsharded sums.

        Needs every BatchNorm1d in eval mode with running statistics: batch statistics of a chunk are not those of the
        whole replicated batch."""
        sums, _ = self._mc_sums(x, n_samples, chunk, seed, sample_range, softmax, entropy=False)
        if sample_range is not None:
            return sums
        return moments_from_sums(sums, n_samples)

    @torch.no_grad()
    def predict_uncertainty(self, x, n_samples: int = 500, chunk: int | None = None, seed=None, sample_range=None):
        """Monte-Carlo predictive uncertainty of the classifier ``softmax(model(x))``: an MCUncertainty with the mean and
        variance of the class probabilities (the bits of ``predict(..., softmax=True)`` for the same seed and chunk) and
        the predictive entropy, expected entropy and mutual information per input.  Same chunking, draws and batch-norm
        requirement as ``predict``; each chunk's per-sample entropies are summed in fp64 on the device in the same pass
        as the probabilities (mnf_mc_class_moments).  ``sample_range=(lo, hi)``: the raw ``(sums [2, B, C],
        entropy_sums [B])`` of samples lo..hi-1; all-reduce both and finish with ``uncertainty_from_sums``."""
        check_mc_args(n_samples, chunk, sample_range)
        sums, entropy_sums = self._mc_sums(x, n_samples, chunk, seed, sample_range, True, entropy=True)
        if sample_range is not None:
            return sums, entropy_sums
        return uncertainty_from_sums(sums, entropy_sums, n_samples)

    def _require_running_stats(self):
        for m in self:
            if isinstance(m, nn.modules.batchnorm._BatchNorm) and not self._uses_running_stats(m):
                raise RuntimeError("MNFFeedForward.predict needs every BatchNorm1d in eval mode with running statistics "
                                   "(call model.eval()): batch statistics of a chunk of samples are not those of the "
                                   "whole replicated batch")

    @torch.no_grad()
    def forward_functions(self, x, n_samples: int, seed=None, sample_offset: int = 0, chunk: int | None = None,
                          noise=None):
        """The network under ``n_samples`` posterior function draws: [S, B, n_out_last], out[s] = f_s(x) with every layer
        evaluated on its weights of sample s (MNFLinear.sample_weights), shared by all rows of x [B, n_in] (or of its
        block x[s] when x is [S, B, n_in]).

        One noise source is shared by the layers, which draw in layer order as ``MNFLinear.forward_functions`` does
        (1 + n_flows_q + 2 draws each), from the tape ``noise`` or from Philox keyed by ``(seed, sample_offset + s)``:
        the result does not depend on x, the batch size, ``chunk`` or a split of the samples between calls.  The layers
        run one after the other over all samples; in each, the weight images are drawn and applied ``chunk`` samples at
        a time (default: about ops.FUNCTION_IMAGE_BYTES of weights; a tape runs as one chunk).  Blocks with ``nn.ReLU``
        and an eval-mode BatchNorm1d run both in the function GEMM's epilogue, other activations are applied by their
        modules.  Needs every BatchNorm1d in eval mode with running statistics, as ``predict`` does: batch statistics
        would mix the samples."""
        ops.check_function_args(n_samples, sample_offset, chunk)
        self._require_running_stats()
        blocks = self._blocks()
        n_samples, sample_offset = int(n_samples), int(sample_offset)
        x = ops.function_input(x, blocks[0][0].n_in, n_samples)
        nz = noise if isinstance(noise, ops.Noise) else ops.Noise(noise, x.device, seed=seed)
        h = x
        for i, (lin, act, bn) in enumerate(blocks):
            relu = type(act) is nn.ReLU
            affine = self._folded(i, bn, x.device) if relu else None
            h = lin._functions(h, n_samples, nz, sample_offset, relu=relu, affine=affine, chunk=chunk)
            if act is not None and affine is None:
                h = bn(act(h.view(-1, h.size(-1)))).view(h.shape)
        return h

    def _mc_sums(self, x, n_samples, chunk, seed, sample_range, softmax, entropy):
        """The chunk loop of predict / predict_uncertainty: fp64 sums [2, B, n_out] and, with ``entropy``, the entropy
        sums [B] (else None) of samples lo..hi-1."""
        self._require_running_stats()
        x = _lib.require_cuda_f32(x, "input")
        B = x.size(0)
        lo, hi = (0, n_samples) if sample_range is None else sample_range
        if not 0 <= lo <= hi <= n_samples:
            raise ValueError(f"sample_range {sample_range} outside [0, {n_samples}]")
        if chunk is None:
            widest = max(max(lin.n_in, lin.n_out) for lin, _, _ in self._blocks())
            chunk = max(1, self.CHUNK_FLOATS // (B * widest))
        if chunk < 1:
            raise ValueError(f"chunk must be positive, got {chunk}")
        if seed is None:
            seed = int(torch.randint(0, 2**62, (1,)).item())  # follows torch.manual_seed
        n_out = self._blocks()[-1][0].n_out
        sums = torch.zeros((2, B, n_out), device=x.device, dtype=torch.float64)
        entropy_sums = torch.zeros(B, device=x.device, dtype=torch.float64) if entropy else None
        for c in range(lo, hi, chunk):
            s_here = min(chunk, hi - c)
            y = self.forward_mc(x, s_here, seed=seed, row_offset=c * B)
            ops.mc_moments(y, B, s_here, sums, softmax=softmax, entropy_sums=entropy_sums)
        return sums, entropy_sums
