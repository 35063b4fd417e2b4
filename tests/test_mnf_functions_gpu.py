"""Posterior function samples of MNFLinear / MNFFeedForward on the GPU: the weight draw against the restated Philox
generator, parity with an fp64 composition under a noise tape, the function GEMM against the weights it was given,
coherence (one network per sample), sharding and chunking, agreement of the marginals with forward_mc's local
reparameterisation, and the MNFFeedForward composition.

Tolerances: fp64 compositions under a tape, rtol 1e-4 (the exact-fp32 MNF class of BASELINE.md 5); the function GEMM
against fp64 on its own weights, the worst-case bound (K + 2) u sum_k |x_k W_k| of a K-term fp32 sum; draws, check_draw's
bound plus the rounding of W = W_mean z + sd E.  The function GEMM runs its tiled form for every batch size, so the
coherence, sharding and chunking checks are bitwise."""

import numpy as np
import pytest
import torch
import torch.nn.functional as F
from torch import nn

from oracle import mnf_cpu
from oracle.noise import NoiseTape
from tests.helpers import golden_sd, load_golden, t
from tests.test_flow_sample_gpu import philox_normal_np

pytestmark = pytest.mark.gpu

DEV = "cuda"
U = 2.0**-24


def _layer(n_in, n_out, seed=0, **kw):
    from torch_mnf.layers import MNFLinear

    torch.manual_seed(seed)
    layer = MNFLinear(n_in, n_out, **kw)
    with torch.no_grad():
        layer.W_log_var.add_(4.0)  # weight noise large enough to matter
        layer.b_log_var.add_(4.0)
        layer.b_mean.normal_(0, 0.1)
    layer.precision = "fp32"
    return layer.requires_grad_(False).to(DEV)


def _model(sizes, seed=0, bn_affine=True, activation=nn.ReLU):
    from torch_mnf.models import MNFFeedForward

    torch.manual_seed(seed)
    model = MNFFeedForward(sizes, activation=activation)
    g = torch.Generator().manual_seed(seed + 100)
    for i in range(2, len(model), 3):
        n = model[i].num_features
        if not bn_affine:
            model[i] = nn.BatchNorm1d(n, affine=False)
        bn = model[i]
        with torch.no_grad():
            bn.running_mean.copy_(0.05 * torch.randn(n, generator=g))
            bn.running_var.copy_(0.01 * (0.2 + torch.rand(n, generator=g)) ** 2)
            if bn_affine:
                bn.weight.copy_(1 + 0.5 * torch.randn(n, generator=g))
                bn.bias.copy_(0.3 * torch.randn(n, generator=g))
    for lin in _linears(model):
        lin.precision = "fp32"
        with torch.no_grad():
            lin.W_log_var.add_(4.0)
    return model.requires_grad_(False).to(DEV).eval()


def _linears(model):
    return [m for m in model if hasattr(m, "kl_div")]


def _x(B, n_in, seed=1):
    return torch.randn(B, n_in, generator=torch.Generator().manual_seed(seed)).to(DEV)


def _noise(seed, row_offset=0):
    from torch_mnf.layers import _mnf_ops as ops

    return ops.Noise(None, DEV, row_offset=row_offset, seed=seed)


def _function_tape(layers, S, seed):
    """Draws of a function call over S samples for each layer in order: z0, the q-flow masks, E, e."""
    g = torch.Generator().manual_seed(seed)
    draws = []
    for lin in layers:
        draws.append(("normal", torch.randn(S, lin.n_in, generator=g)))
        for _ in lin.flow_q.flows:
            draws.append(("bernoulli", torch.bernoulli(torch.full((S, lin.n_in), 0.5), generator=g)))
        draws.append(("normal", torch.randn(S, lin.n_out, lin.n_in, generator=g)))
        draws.append(("normal", torch.randn(S, lin.n_out, generator=g)))
    return NoiseTape(draws)


def _sd64(layer):
    return {k: v.detach().double().cpu() for k, v in layer.state_dict().items()}


def _ref_functions(sd, x, S, tape):
    """fp64: z_s from oracle.mnf_cpu.linear_sample_z, W_s = W_mean z_s + exp(W_log_var / 2) E_s, b_s likewise, and
    x_s @ W_s^T + b_s for x [B, n_in] (shared) or [S, B, n_in]."""
    n_out, n_in = sd["W_mean"].shape
    z, _ = mnf_cpu.linear_sample_z(sd, S, tape)
    E, e = tape.normal((S, n_out, n_in)).double(), tape.normal((S, n_out)).double()
    W = sd["W_mean"] * z[:, None, :] + (0.5 * sd["W_log_var"]).exp() * E
    b = sd["b_mean"] + (0.5 * sd["b_log_var"]).exp() * e
    return x.double() @ W.transpose(1, 2) + b[:, None, :]


def _close(got, ref, what, rtol=1e-4):
    ref = ref.double().cpu()
    atol = 1e-5 * max(1.0, float(ref.abs().mean()))
    torch.testing.assert_close(got.double().cpu(), ref, rtol=rtol, atol=atol, msg=lambda m: f"{what}: {m}")


# ---------------------------------------------------------------------------------------------------------------------
# 1. draws
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_in,n_out,S,offset", [(20, 7, 5, 0), (33, 9, 6, 3), (64, 48, 3, (1 << 32) // (64 * 48) + 1),
                                                 (300, 4, 7, 2)])
def test_sample_weights_match_restated_philox(n_in, n_out, S, offset):
    """E and e are philox_normal of their global elements ((offset + s) * n_out + o) * n_in + i and (offset + s) * n_out
    + o on streams 1 + n_flows_q and 2 + n_flows_q; z is sample_z(S) at row_offset = offset, bit for bit.  The last
    case puts the weight elements past 2^32; (33, 9) starts and ends the image inside a Philox block."""
    from torch_mnf.layers import _mnf_ops as ops

    layer = _layer(n_in, n_out, seed=n_in)
    seed = 0x1234_5678_9ABC
    noise = _noise(seed)
    z = ops.linear_function_z(layer, S, noise, offset)
    W, b = ops.linear_sample_weights(layer, z, noise, offset)
    assert noise.streams == len(layer.flow_q.flows) + 3
    z_ref, _ = layer.sample_z(S, noise=_noise(seed, row_offset=offset))
    assert torch.equal(z, z_ref)
    W2, b2 = layer.sample_weights(S, seed=seed, sample_offset=offset)
    assert torch.equal(W, W2) and torch.equal(b, b2)
    assert W.shape == (S, n_out, n_in) and b.shape == (S, n_out) and W.is_contiguous()
    nq = len(layer.flow_q.flows)
    if n_in == 64:
        assert offset * n_out * n_in > 1 << 32

    sd = _sd64(layer)
    z64 = z.double().cpu()
    Wg, bg = W.double().cpu().numpy(), b.double().cpu().numpy()
    mz = (sd["W_mean"] * z64[:, None, :]).numpy()
    sdw = (0.5 * sd["W_log_var"]).exp().numpy()
    el = ((np.arange(S, dtype=np.uint64)[:, None, None] + np.uint64(offset)) * np.uint64(n_out)
          + np.arange(n_out, dtype=np.uint64)[None, :, None]) * np.uint64(n_in) + np.arange(n_in, dtype=np.uint64)
    for got, ref_el, stream, scale, ulp in (
            ((Wg - mz) / sdw, el, nq + 1, sdw, np.abs(Wg) + np.abs(mz)),
            ((bg - sd["b_mean"].numpy()) / (0.5 * sd["b_log_var"]).exp().numpy(),
             (np.arange(S, dtype=np.uint64)[:, None] + np.uint64(offset)) * np.uint64(n_out)
             + np.arange(n_out, dtype=np.uint64), nq + 2, (0.5 * sd["b_log_var"]).exp().numpy(),
             np.abs(bg) + np.abs(sd["b_mean"].numpy()))):
        ref, r = philox_normal_np(ref_el, stream, seed)
        # check_draw's bound, expf's error on the scale, and the fp32 rounding of the stored weight over the scale
        tol = 1e-6 + 2e-6 * r + 2e-7 / r + 4e-7 * np.abs(ref) + 2 * U * ulp / scale
        bad = np.abs(got - ref) > tol
        assert not bad.any(), f"{int(bad.sum())} draws off, worst {float(np.abs(got - ref).max()):.3e}"


# ---------------------------------------------------------------------------------------------------------------------
# 2. tape parity
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,n_in,n_out,kw", [("mnf_linear_20x7", 20, 7, {}),
                                                ("mnf_linear_256x128", 256, 128, {"n_flows_r": 1})])
def test_linear_functions_match_fp64_under_a_tape(name, n_in, n_out, kw):
    from torch_mnf.layers import MNFLinear

    g = load_golden(name)
    layer = MNFLinear(n_in, n_out, **kw)
    layer.load_state_dict(golden_sd(g))
    layer.to(DEV)
    x, S = t(g, "x"), 4
    tape = _function_tape([layer], S, seed=3)
    y = layer.forward_functions(x.to(DEV), S, noise=tape)
    assert tape.pos == len(tape.draws)
    assert y.shape == (S, x.size(0), n_out) and y.is_contiguous()
    _close(y, _ref_functions(golden_sd(g), x.double(), S, _function_tape([layer], S, seed=3)), name)
    tape = _function_tape([layer], S, seed=3)
    y = layer.forward_functions(x.to(DEV), S, noise=tape, relu=True)
    _close(y, torch.relu(_ref_functions(golden_sd(g), x.double(), S, _function_tape([layer], S, seed=3))), name + " relu")


@pytest.mark.parametrize("bn_affine", [True, False])
def test_feed_forward_functions_match_fp64_under_a_tape(bn_affine):
    model = _model([20, 32, 7], seed=2, bn_affine=bn_affine)
    x, S = _x(9, 20, seed=4), 5
    tape = _function_tape(_linears(model), S, seed=6)
    y = model.forward_functions(x, S, noise=tape)
    assert tape.pos == len(tape.draws) and y.shape == (S, 9, 7)
    ref_tape = _function_tape(_linears(model), S, seed=6)
    h = x.double().cpu()
    for lin, act, bn in model._blocks():
        h = _ref_functions(_sd64(lin), h, S, ref_tape)
        if act is not None:
            d = lambda v: None if v is None else v.detach().double().cpu()  # noqa: E731
            h = F.batch_norm(torch.relu(h).reshape(-1, h.size(-1)), d(bn.running_mean), d(bn.running_var), d(bn.weight),
                             d(bn.bias), training=False, eps=bn.eps).view(h.shape)
    _close(y, h, "MNFFeedForward")


# ---------------------------------------------------------------------------------------------------------------------
# 3. the function GEMM against its weights
# ---------------------------------------------------------------------------------------------------------------------
def _gemm_bound_check(y, x, W, b, relu=False):
    x64, W64, b64 = x.double().cpu(), W.double().cpu(), b.double().cpu()
    ref = x64 @ W64.transpose(1, 2) + b64[:, None, :]
    absum = x64.abs() @ W64.abs().transpose(1, 2) + b64.abs()[:, None, :]
    if relu:
        ref = ref.clamp_min(0)
    K = W.size(2)
    err = (y.double().cpu() - ref).abs()
    bound = 1.01 * (K + 2) * U * absum + 1e-30
    assert bool((err <= bound).all()), f"worst error / bound {float((err / bound).max()):.3f}"


@pytest.mark.parametrize("n_in,n_out", [(37, 45), (130, 70), (300, 5), (64, 128)])
@pytest.mark.parametrize("B", [1, 3, 5, 64, 200])
def test_function_gemm_matches_fp64_on_its_weights(n_in, n_out, B):
    layer = _layer(n_in, n_out, seed=B)
    S, seed = 3, 77 + B
    W, b = layer.sample_weights(S, seed=seed)
    x = _x(B, n_in, seed=B)
    y = layer.forward_functions(x, S, seed=seed)
    assert y.shape == (S, B, n_out)
    _gemm_bound_check(y, x.unsqueeze(0).expand(S, B, n_in), W, b)
    x3 = torch.randn(S, B, n_in, generator=torch.Generator().manual_seed(B + 1)).to(DEV)
    y3 = layer.forward_functions(x3, S, seed=seed, relu=True)
    _gemm_bound_check(y3, x3, W, b, relu=True)


# ---------------------------------------------------------------------------------------------------------------------
# 4. coherence: one network per sample
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_in", [20, 300])
def test_duplicated_rows_get_identical_outputs(n_in):
    layer = _layer(n_in, 6, seed=5)
    x = _x(6, n_in, seed=2)
    x[4] = x[1]
    y = layer.forward_functions(x, 8, seed=11)
    assert torch.equal(y[:, 4], y[:, 1])
    assert not torch.equal(y[0], y[1])  # the samples are different networks
    mc = layer.forward_mc(x, 8).view(8, 6, -1)  # local reparameterisation: a fresh z and eps per row
    assert not torch.equal(mc[:, 4], mc[:, 1])

    model = _model([n_in, 16, 3], seed=1)
    y = model.forward_functions(x, 8, seed=12)
    assert torch.equal(y[:, 4], y[:, 1])
    mc = model.forward_mc(x, 8, seed=12).view(8, 6, -1)
    assert not torch.equal(mc[:, 4], mc[:, 1])


@pytest.mark.parametrize("n_in", [20, 300])
def test_functions_do_not_depend_on_the_rest_of_the_batch(n_in):
    layer = _layer(n_in, 9, seed=6)
    x1, x2 = _x(5, n_in, seed=3), _x(3, n_in, seed=4)
    both = layer.forward_functions(torch.cat([x1, x2]), 6, seed=21)
    sep = torch.cat([layer.forward_functions(x1, 6, seed=21), layer.forward_functions(x2, 6, seed=21)], dim=1)
    assert torch.equal(both, sep)
    one = layer.forward_functions(x2[1:2], 6, seed=21)
    assert torch.equal(one[:, 0], both[:, 6])


# ---------------------------------------------------------------------------------------------------------------------
# 5. sharding and chunking
# ---------------------------------------------------------------------------------------------------------------------
def test_sample_offset_shards_reproduce_one_call():
    layer = _layer(33, 10, seed=7)
    x, S = _x(7, 33), 12
    full = layer.forward_functions(x, S, seed=5)
    halves = torch.cat([layer.forward_functions(x, S // 2, seed=5),
                        layer.forward_functions(x, S // 2, seed=5, sample_offset=S // 2)])
    assert torch.equal(full, halves)
    W, b = layer.sample_weights(S, seed=5)
    W2, b2 = layer.sample_weights(S - 5, seed=5, sample_offset=5)
    assert torch.equal(W[5:], W2) and torch.equal(b[5:], b2)

    model = _model([33, 24, 4], seed=3)
    full = model.forward_functions(x, S, seed=8)
    halves = torch.cat([model.forward_functions(x, S // 2, seed=8),
                        model.forward_functions(x, S // 2, seed=8, sample_offset=S // 2)])
    assert torch.equal(full, halves)


@pytest.mark.parametrize("activation", [nn.ReLU, nn.Tanh])
def test_feed_forward_chunking_gives_the_same_bits(activation):
    model = _model([20, 32, 16, 5], seed=4, activation=activation)
    x, S = _x(11, 20), 16
    ref = model.forward_functions(x, S, seed=9, chunk=S)
    for chunk in (1, 7, None):
        assert torch.equal(model.forward_functions(x, S, seed=9, chunk=chunk), ref), chunk


def test_layer_chunks_of_the_weight_image_give_the_same_bits(monkeypatch):
    from torch_mnf.layers import _mnf_ops as ops

    layer = _layer(40, 24, seed=8)
    x = _x(5, 40)
    ref = layer.forward_functions(x, 9, seed=3)
    monkeypatch.setattr(ops, "FUNCTION_IMAGE_BYTES", 4 * 24 * 41 * 2)  # two samples per chunk
    assert ops.function_chunk(24 * 41) == 2
    assert torch.equal(layer.forward_functions(x, 9, seed=3), ref)


# ---------------------------------------------------------------------------------------------------------------------
# 6. marginals agree with the local reparameterisation
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("seed", [1, 2, 3])
def test_marginals_match_forward_mc(seed):
    """Per row, f_s(x) and forward(x) have the same distribution.  With S = 4096 the means agree within 6 standard
    errors and the variances within [0.8, 1.25] (about 7 standard deviations of the ratio of two sample variances)."""
    layer = _layer(16, 5, seed=10)
    with torch.no_grad():
        layer.q0_log_var.fill_(-2.0)  # z varies too
    x, S = _x(8, 16, seed=seed), 4096
    torch.manual_seed(seed)
    f = layer.forward_functions(x, S).double()
    m = layer.forward_mc(x, S).view(S, 8, 5).double()
    se = ((f.var(0) + m.var(0)) / S).sqrt()
    assert bool(((f.mean(0) - m.mean(0)).abs() <= 6 * se).all())
    ratio = f.var(0) / m.var(0)
    assert bool(((ratio >= 0.8) & (ratio <= 1.25)).all()), ratio


# ---------------------------------------------------------------------------------------------------------------------
# 7. MNFFeedForward composition
# ---------------------------------------------------------------------------------------------------------------------
def _chain(model, x, S, seed):
    """MNFLinear.forward_functions layer by layer on one shared Noise; activation and batch norm through the modules."""
    nz = _noise(seed)
    h = x
    for lin, act, bn in model._blocks():
        h = lin.forward_functions(h, S, noise=nz)
        if act is not None:
            h = bn(act(h.view(-1, h.size(-1)))).view(h.shape)
    return h


def test_feed_forward_equals_the_layer_chain():
    model = _model([20, 32, 16, 7], seed=5)
    x, S = _x(13, 20), 6
    y = model.forward_functions(x, S, seed=31)
    ref = _chain(model, x, S, 31)
    torch.testing.assert_close(y, ref, rtol=1e-4, atol=1e-5 * float(ref.abs().max()))
    tanh = _model([20, 32, 7], seed=5, activation=nn.Tanh)
    assert torch.equal(tanh.forward_functions(x, S, seed=31), _chain(tanh, x, S, 31))


def test_feed_forward_rejects_batch_statistics():
    model = _model([20, 32, 7], seed=5).train()
    with pytest.raises(RuntimeError, match="eval mode"):
        model.forward_functions(_x(4, 20), 3, seed=1)
