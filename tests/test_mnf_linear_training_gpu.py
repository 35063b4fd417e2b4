"""Gradients of MNFLinear (forward and kl_div) and MNFFeedForward on the training path (csrc/mnf_train.cu through
torch_mnf/layers/_train.py) against fp64 autograd over the oracle, under the same noise, at shapes beyond the golden
fixtures: batches past the mnf_colsum row split (8 192 rows) and the elementwise grid-stride loop (606 208 elements),
2 100 output rows past the mnf_kl_rows_backward row split, one-unit layers, deeper conditioner nets (the LeakyReLU
between two Linears), layers without q- or r-flows, and a fused ReLU.

Noise: a RecordingTape hands the oracle draws from a seeded generator and keeps them; the CUDA module then replays
them through NoiseTape, which checks the kind and shape of every draw, so a change in draw order fails loudly.  The
layers get W_log_var + 4, so the noise branch carries weight in the gradients.

Tolerances:
* fewer than 4 097 rows: |err| <= 2e-4 max |ref| + 1e-7 per tensor, the class of tests/test_mnf_autograd_gpu.py;
* 4 097 rows and more: the forward part of a parameter gradient is a sum over rows, and its fp32 rounding grows with
  the sum of the absolute values of the summed terms, not with the (partly cancelled) result.  The oracle runs the
  rows in chunks of 1 024 and forms S = sum over chunks |chunk gradient| in fp64; the bound is
  (8 + 4 sqrt(R)) u S + 16 u max S + 2e-4 max |kl_div gradient|, u = 2^-24.  The first term covers the reductions over
  R rows, as in tests/test_mnf_train_primitives_gpu.py; the second, per-row rounding in the flow chain, which scales
  with the largest terms rather than an element's own; the third, the kl_div part, whose size does not depend on R and
  which keeps the small-batch class.  S over chunks is at most the sum over single rows, so this is stricter than the
  per-row bound.  The input gradient is per row and keeps the 2e-4 max |ref| class at every size."""

import copy
import math

import pytest
import torch
import torch.nn.functional as F
from torch import nn

from oracle import mnf_cpu
from oracle.noise import NoiseTape

pytestmark = pytest.mark.gpu

DEV = "cuda"
U = 2.0**-24
LARGE_R = 4097
CHUNK = 1024


class RecordingTape:
    """Draws from a seeded CPU generator when asked and records every draw (kind, tensor) in order."""

    def __init__(self, seed):
        self.g = torch.Generator().manual_seed(seed)
        self.draws = []

    def normal(self, shape):
        t = torch.randn(tuple(shape), generator=self.g)
        self.draws.append(("normal", t))
        return t

    def bernoulli(self, shape):
        t = torch.bernoulli(torch.full(tuple(shape), 0.5), generator=self.g)
        self.draws.append(("bernoulli", t))
        return t


def _layer(n_in, n_out, seed=0, **kw):
    from torch_mnf.layers import MNFLinear

    torch.manual_seed(seed)
    layer = MNFLinear(n_in, n_out, **kw)
    with torch.no_grad():
        layer.W_log_var.add_(4.0)
    return layer


def _sd64(module):
    return {k: v.detach().cpu().double().requires_grad_() for k, v in module.state_dict().items()}


def _grads(sd64):
    return {k: (v.grad.clone() if v.grad is not None else torch.zeros_like(v)) for k, v in sd64.items()}


def _oracle_linear(layer, x, w, seed, relu=False, kl=True):
    """fp64 gradients of sum(w * y) [+ kl_div] over the oracle, rows in chunks of CHUNK.  Returns (forward draws,
    kl draws, {name: grad}, {name: (S, kl_div gradient)}, grad x, kl value)."""
    R = x.size(0)
    rec = RecordingTape(seed)
    ref, S, gx, chunk_draws = None, None, [], []
    for r0 in range(0, R, CHUNK):
        p = _sd64(layer)
        xr = x[r0:r0 + CHUNK].double().requires_grad_()
        n0 = len(rec.draws)
        y = mnf_cpu.linear_forward(p, xr, rec)
        y = torch.relu(y) if relu else y
        (y * w[r0:r0 + CHUNK].double()).sum().backward()
        g = _grads(p)
        ref = g if ref is None else {k: ref[k] + g[k] for k in g}
        S = {k: v.abs() for k, v in g.items()} if S is None else {k: S[k] + g[k].abs() for k in g}
        gx.append(xr.grad)
        chunk_draws.append(rec.draws[n0:])
    fwd = [(kind, torch.cat([c[i][1] for c in chunk_draws])) for i, (kind, _) in enumerate(chunk_draws[0])]
    kl_draws, kl_value, g = None, None, {k: torch.zeros_like(v) for k, v in ref.items()}
    if kl:
        rec_kl = RecordingTape(seed + 1)
        p = _sd64(layer)
        kl_value = mnf_cpu.linear_kl_div(p, rec_kl)
        kl_value.backward()
        g = _grads(p)
        ref = {k: ref[k] + g[k] for k in g}
        kl_draws = rec_kl.draws
    return fwd, kl_draws, ref, {k: (S[k], g[k]) for k in S}, torch.cat(gx), kl_value


def _check(got, ref, S, R, what):
    if got is None:
        got = torch.zeros_like(ref)
    err = (got.detach().cpu().double() - ref).abs()
    if R < LARGE_R:
        bound = 2e-4 * float(ref.abs().max()) + 1e-7
    else:
        S, g_kl = S
        bound = (8 + 4 * math.sqrt(R)) * U * S + 16 * U * float(S.max()) + 2e-4 * float(g_kl.abs().max())
    bad = ~(err <= bound)  # NaN fails
    assert not bool(bad.any()), (f"{what}: {int(bad.sum())} elements outside the bound, max err {float(err.max()):.3e}, "
                                 f"worst excess {float((err - bound).max()):.3e} (max |ref| {float(ref.abs().max()):.3e})")


def _check_module(module, ref, S, R, what):
    checked = 0
    for k, p in module.named_parameters():
        _check(p.grad, ref[k], S[k], R, f"{what} {k}")
        checked += 1
    assert checked >= 8


def _run_linear(n_in, n_out, R, seed, relu=False, **kw):
    layer = _layer(n_in, n_out, seed, **kw)
    g = torch.Generator().manual_seed(seed + 7)
    x = torch.randn(R, n_in, generator=g)
    w = torch.randn(R, n_out, generator=g)  # fp32 loss weights, exact in the fp64 oracle too
    fwd, kl_draws, ref, S, gx_ref, kl_ref = _oracle_linear(layer, x, w, seed + 11, relu=relu)
    layer.cuda()
    xg = x.cuda().requires_grad_()
    ft, kt = NoiseTape(fwd), NoiseTape(kl_draws)
    y = layer(xg, noise=ft, relu=relu)
    kl = layer.kl_div(noise=kt)
    assert ft.pos == len(ft.draws) and kt.pos == len(kt.draws), "draws left on the tape"
    torch.testing.assert_close(kl.detach().cpu().double(), kl_ref.detach(), rtol=2e-5, atol=1e-4)
    ((y * w.cuda()).sum() + kl).backward()
    what = f"MNFLinear({n_in}, {n_out}, {kw}) R={R} relu={relu}"
    _check_module(layer, ref, S, R, what)
    _check(xg.grad, gx_ref, gx_ref.abs(), 0, what + " x")  # per row: the max-relative class at every R
    return layer, kl_draws, kl_ref


SHAPES = [(1, 1, 1), (17, 65, 1), (64, 64, 64), (65, 129, 130), (300, 33, 4097), (130, 2100, 16), (64, 10, 65536)]


@pytest.mark.parametrize("n_in,n_out,R", SHAPES)
def test_linear_forward_and_kl_div_gradients(n_in, n_out, R):
    """loss = sum(w * y) + kl_div: the gradient of every parameter and of x against fp64 autograd."""
    _run_linear(n_in, n_out, R, seed=n_in + n_out + R)


@pytest.mark.parametrize("kw,relu", [({"h_sizes": (16, 8)}, False), ({"n_flows_q": 0}, False),
                                     ({"n_flows_r": 0}, False), ({"n_flows_q": 0, "n_flows_r": 0}, False),
                                     ({}, True), ({"h_sizes": (16, 8)}, True)])
@pytest.mark.parametrize("n_in,n_out,R", [(33, 20, 70), (65, 129, 4097)])
def test_linear_gradients_flow_variants_and_relu(n_in, n_out, R, kw, relu):
    """Deeper conditioner nets (LeakyFn between two LinearFns), no q- or r-flows (a zero log-det stands in), and the
    fused ReLU of forward(relu=True)."""
    _run_linear(n_in, n_out, R, seed=3 * n_in + R, relu=relu, **kw)


@pytest.mark.parametrize("n_in,n_out", [(n_in, n_out) for n_in, n_out, _ in SHAPES])
def test_kl_div_grad_path_matches_the_fused_kernel(n_in, n_out):
    """The grad-mode kl_div (_train.linear_kl_div) and the no-grad one (ops.kl_div, csrc/mnf_kl.cu) on the same tape
    agree with each other and with the fp64 oracle."""
    layer = _layer(n_in, n_out, seed=5 + n_in)
    rec = RecordingTape(99)
    ref = mnf_cpu.linear_kl_div({k: v.double() for k, v in layer.state_dict().items()}, rec)
    layer.cuda()
    grad_kl = layer.kl_div(noise=NoiseTape(rec.draws))
    assert grad_kl.requires_grad
    with torch.no_grad():
        fused = layer.kl_div(noise=NoiseTape(rec.draws))
    torch.testing.assert_close(grad_kl.detach().cpu().double(), ref, rtol=2e-5, atol=1e-4)
    torch.testing.assert_close(fused.cpu().double(), ref, rtol=2e-5, atol=1e-4)
    torch.testing.assert_close(fused, grad_kl.detach(), rtol=2e-5, atol=1e-4)


# ---- partial gradients ------------------------------------------------------------------------------------------------
def _partial_case(seed=21, n_in=17, n_out=30, R=33):
    """Small enough that no reduction splits over blocks (R <= 64 rows, n_out <= 32): the gradients are deterministic."""
    layer = _layer(n_in, n_out, seed)
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(R, n_in, generator=g)
    w = torch.randn(R, n_out, generator=g)  # fp32 loss weights, exact in the fp64 oracle too
    fwd, kl_draws, ref, S, gx_ref, _ = _oracle_linear(layer, x, w, seed)
    return layer.cuda(), x, w.cuda(), fwd, kl_draws, ref, S, gx_ref


def _step(layer, x, w, fwd, kl_draws):
    y = layer(x, noise=NoiseTape(fwd))
    loss = (y * w).sum()
    if kl_draws is not None:
        loss = loss + layer.kl_div(noise=NoiseTape(kl_draws))
    loss.backward()


def test_frozen_parameters_give_only_the_input_gradient():
    layer, x, w, fwd, _, _, _, _ = _partial_case()
    x64 = x.double().requires_grad_()
    y_ref = mnf_cpu.linear_forward({k: v.detach().cpu().double() for k, v in layer.state_dict().items()}, x64,
                                   NoiseTape(fwd))
    (y_ref * w.cpu().double()).sum().backward()
    for p in layer.parameters():
        p.requires_grad_(False)
    xg = x.cuda().requires_grad_()
    _step(layer, xg, w, fwd, None)
    assert all(p.grad is None for p in layer.parameters())
    _check(xg.grad, x64.grad, None, 0, "frozen layer: x")


def test_input_without_grad_leaves_the_parameter_gradients_unchanged():
    layer, x, w, fwd, kl_draws, ref, S, _ = _partial_case()
    twin = copy.deepcopy(layer)
    xg = x.cuda().requires_grad_()
    _step(layer, xg, w, fwd, kl_draws)
    xn = x.cuda()
    _step(twin, xn, w, fwd, kl_draws)
    assert xn.grad is None and xg.grad is not None
    for (k, a), (_, b) in zip(layer.named_parameters(), twin.named_parameters()):
        assert torch.equal(a.grad, b.grad), k
    _check_module(twin, ref, S, x.size(0), "x without grad")


def test_non_contiguous_input_gives_the_contiguous_gradients():
    layer, x, w, fwd, kl_draws, _, _, gx_ref = _partial_case()
    twin = copy.deepcopy(layer)
    xc = x.cuda().requires_grad_()
    _step(layer, xc, w, fwd, kl_draws)
    xt = x.t().contiguous().cuda().t().requires_grad_()  # the same values in a transposed layout
    assert not xt.is_contiguous() and xt.is_leaf
    _step(twin, xt, w, fwd, kl_draws)
    assert torch.equal(xt.grad, xc.grad)
    for (k, a), (_, b) in zip(layer.named_parameters(), twin.named_parameters()):
        assert torch.equal(a.grad, b.grad), k
    _check(xt.grad, gx_ref, None, 0, "transposed x")


# ---- MNFFeedForward ---------------------------------------------------------------------------------------------------
def _ff_model(sizes, seed):
    from torch_mnf.models import MNFFeedForward

    torch.manual_seed(seed)
    model = MNFFeedForward(sizes)
    g = torch.Generator().manual_seed(seed + 100)
    for i in range(2, len(model), 3):
        bn, n = model[i], model[i].num_features
        with torch.no_grad():
            bn.running_mean.copy_(0.05 * torch.randn(n, generator=g))
            bn.running_var.copy_(0.01 * (0.2 + torch.rand(n, generator=g)) ** 2)
            bn.weight.copy_(1 + 0.5 * torch.randn(n, generator=g))
            bn.bias.copy_(0.3 * torch.randn(n, generator=g))
    for m in model:
        if hasattr(m, "kl_div"):
            with torch.no_grad():
                m.W_log_var.add_(4.0)
    return model


def _ff_oracle(model, x, w, S, seed, training):
    """fp64 composition mnf_cpu.linear_forward -> relu -> F.batch_norm(training=...) on x.repeat(S, 1); returns the
    draws, the gradients by parameter name and the input gradient."""
    rec = RecordingTape(seed)
    params = {k: v.detach().double().requires_grad_() for k, v in model.named_parameters()}
    h = x.double().requires_grad_()
    x64 = h
    h = h.repeat(S, 1)
    for i, (lin, act, bn) in enumerate(model._blocks()):
        li = 3 * i
        p = {k: params[f"{li}.{k}"] for k, _ in lin.named_parameters()}
        h = mnf_cpu.linear_forward(p, h, rec)
        if act is not None:
            rm, rv = (None, None) if training else (bn.running_mean.double(), bn.running_var.double())
            h = F.batch_norm(torch.relu(h), rm, rv, params[f"{li + 2}.weight"], params[f"{li + 2}.bias"],
                             training=training, eps=bn.eps)
    (h * w.double()).sum().backward()
    return rec.draws, {k: v.grad for k, v in params.items()}, x64.grad


@pytest.mark.parametrize("sizes", [[16, 65, 33, 3], [130, 64, 10]])
@pytest.mark.parametrize("training", [True, False])
@pytest.mark.parametrize("S", [1, 4])
def test_feed_forward_gradients_match_fp64(sizes, training, S):
    """forward_mc(x, S) under grad -- every MNFLinear on its differentiable path, nn.ReLU, and BatchNorm1d with batch
    statistics over all B * S rows (training) or running statistics (eval) -- against the fp64 composition: the
    gradient of every MNFLinear and BatchNorm parameter, and of x."""
    model = _ff_model(sizes, seed=len(sizes) + sizes[0])
    model.train(training)
    B = 37
    g = torch.Generator().manual_seed(S)
    x = torch.randn(B, sizes[0], generator=g)
    w = torch.randn(B * S, sizes[-1], generator=g)
    draws, ref, gx_ref = _ff_oracle(model, x, w, S, seed=31 + S, training=training)
    model.to(DEV)
    tape = NoiseTape(draws)
    xg = x.to(DEV).requires_grad_()
    y = model.forward_mc(xg, S, noise=tape)
    assert y.requires_grad and tape.pos == len(tape.draws)
    (y * w.to(DEV)).sum().backward()
    what = f"MNFFeedForward({sizes}) training={training} S={S}"
    n_bn = 0
    for k, p in model.named_parameters():
        if ref[k] is None:  # kl_div's auxiliary posterior (r0_*, flow_r) is not part of the forward pass
            assert p.grad is None or not p.grad.any(), f"{what}: unexpected gradient on {k}"
            continue
        _check(p.grad, ref[k], None, 0, f"{what} {k}")
        n_bn += isinstance(model[int(k.split(".")[0])], nn.BatchNorm1d)
    assert n_bn == 2 * (len(sizes) - 2)
    _check(xg.grad, gx_ref, None, 0, what + " x")
