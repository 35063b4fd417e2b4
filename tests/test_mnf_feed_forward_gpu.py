"""MNFFeedForward.forward_mc / predict on the GPU: oracle parity with injected noise, the same draws as an unfused layer
loop, bitwise invariance of the plain MNFLinear entry points, sharding, the Monte-Carlo moments, and the fallbacks.

Tolerances: exact-fp32 kernels rtol 1e-4 against the fp64 oracle; tensor-core (TF32) layers the 2e-3 class of
BASELINE.json.  Fused vs unfused runs of the same kernels differ only by the folded batch norm: fp32 rounding."""

import copy

import pytest
import torch
import torch.nn.functional as F
from torch import nn

from oracle import mnf_cpu
from oracle.noise import NoiseTape

pytestmark = pytest.mark.gpu

DEV = "cuda"


def _model(sizes, seed=0, bn_affine=True, activation=nn.ReLU, precision=None):
    from torch_mnf.models import MNFFeedForward

    torch.manual_seed(seed)
    model = MNFFeedForward(sizes, activation=activation)
    g = torch.Generator().manual_seed(seed + 100)
    for i in range(2, len(model), 3):  # trained-looking batch norms: non-zero running mean, non-unit running variance
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
        lin.precision = precision or lin.precision
        with torch.no_grad():
            lin.W_log_var.add_(4.0)  # noise large enough to matter
    return model.to(DEV).eval()


def _linears(model):
    return [m for m in model if hasattr(m, "kl_div")]


def _blocks(model):
    return model._blocks()


def _tape(model, R, seed):
    g = torch.Generator().manual_seed(seed)
    draws = []
    for lin in _linears(model):
        draws.append(("normal", torch.randn(R, lin.n_in, generator=g)))
        for _ in lin.flow_q.flows:
            draws.append(("bernoulli", torch.bernoulli(torch.full((R, lin.n_in), 0.5), generator=g)))
        draws.append(("normal", torch.randn(R, lin.n_out, generator=g)))
    return NoiseTape(draws)


def _oracle(model, x, S, tape, act=torch.relu):
    """fp64 composition: oracle.mnf_cpu.linear_forward + activation + F.batch_norm(training=False)."""
    h = x.double().cpu().repeat(S, 1)
    for lin, a, bn in _blocks(model):
        sd = {k: v.detach().double().cpu() for k, v in lin.state_dict().items()}
        h = mnf_cpu.linear_forward(sd, h, tape)
        if a is not None:
            d = lambda t: None if t is None else t.detach().double().cpu()  # noqa: E731
            h = F.batch_norm(act(h), d(bn.running_mean), d(bn.running_var), d(bn.weight), d(bn.bias), training=False,
                             eps=bn.eps)
    return h


def _unfused(model, x, S, seed, row_offset=0):
    """Hand-written layer loop: one shared Noise, plain layer kernels, then the activation and BatchNorm modules."""
    from torch_mnf.layers import _mnf_ops as ops

    nz = ops.Noise(None, x.device, row_offset, seed=seed)
    h = x
    for lin, a, bn in _blocks(model):
        h = lin._forward_rows(h, x.size(0) * S, nz, relu=False)
        if a is not None:
            h = bn(a(h))
    return h


def _close_tc(got, ref):
    ref = ref.float()
    torch.testing.assert_close(got.cpu(), ref, rtol=2e-3, atol=2e-3 * float(ref.pow(2).mean().sqrt()))


# ---- 1. parity with the oracle ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("bn_affine", [True, False])
def test_forward_mc_matches_oracle_exact_fp32(bn_affine):
    model = _model([16, 32, 3], seed=1, bn_affine=bn_affine, precision="fp32")
    B, S = 7, 5
    x = torch.randn(B, 16, generator=torch.Generator().manual_seed(2))
    tape = _tape(model, B * S, seed=3)
    got = model.forward_mc(x.to(DEV), S, noise=tape)
    assert tape.pos == len(tape.draws)
    ref = _oracle(model, x, S, tape.rewind())
    torch.testing.assert_close(got.cpu().double(), ref, rtol=1e-4, atol=1e-5 * max(1.0, float(ref.abs().mean())))


@pytest.mark.parametrize("sizes,bn_affine", [([256, 256, 10], True), ([256, 256, 10], False), ([128, 72, 12], True)])
def test_forward_mc_matches_oracle_tensor_cores(sizes, bn_affine):
    """Every layer on the tcgen05 path; hidden width 72 also runs the epilogue's ragged column chunk."""
    model = _model(sizes, seed=4, bn_affine=bn_affine, precision="tf32")
    B, S = 32, 8
    x = torch.randn(B, sizes[0], generator=torch.Generator().manual_seed(5))
    tape = _tape(model, B * S, seed=6)
    got = model.forward_mc(x.to(DEV), S, noise=tape)
    _close_tc(got, _oracle(model, x, S, tape.rewind()))


# ---- 2. same draws as the unfused path ----------------------------------------------------------------------------------
@pytest.mark.parametrize("sizes,B,S", [([16, 32, 3], 9, 11), ([256, 256, 10], 64, 8), ([784, 1024, 1024, 10], 16, 4)])
def test_forward_mc_matches_unfused_layer_loop(sizes, B, S):
    model = _model(sizes, seed=7)
    x = torch.randn(B, sizes[0], device=DEV)
    got = model.forward_mc(x, S, seed=1234)
    ref = _unfused(model, x, S, seed=1234)
    scale = float(ref.abs().mean())
    torch.testing.assert_close(got, ref, rtol=2e-5, atol=2e-5 * scale)
    # the folded coefficients follow an in-place update of the buffers
    with torch.no_grad():
        model[2].running_mean.add_(0.01)
        model[2].weight.mul_(1.5)
    got = model.forward_mc(x, S, seed=1234)
    ref = _unfused(model, x, S, seed=1234)
    torch.testing.assert_close(got, ref, rtol=2e-5, atol=2e-5 * scale)


# ---- 3. the plain entry points are unchanged ------------------------------------------------------------------------------
@pytest.mark.parametrize("tc", [False, True])
def test_plain_linear_entry_points_are_bitwise_unchanged(tc):
    from torch_mnf import _lib
    from torch_mnf.layers import MNFLinear
    from torch_mnf.layers import _mnf_ops as ops

    torch.manual_seed(8)
    n_in, n_out, x_rows, R = (256, 200, 64, 512) if tc else (24, 13, 5, 40)
    layer = MNFLinear(n_in, n_out).to(DEV)
    x = torch.randn(x_rows, n_in, device=DEV)
    z = 1 + 0.1 * torch.randn(R, n_in, device=DEV)
    lib = _lib.lib()
    args = [layer.W_mean, layer.W_log_var, layer.b_mean, layer.b_log_var]
    st = _lib.stream_ptr(x.device)

    def run(fn, *affine):
        out = torch.empty(R, n_out, device=DEV)
        common = [x.data_ptr(), x_rows, z.data_ptr(), *(a.data_ptr() for a in args), None, 77, 3, 5, out.data_ptr(), R,
                  n_in, n_out, 1]
        if tc:
            ws = torch.empty(lib.mnf_linear_tc_workspace(x_rows, R, n_in, n_out), device=DEV)
            rc = fn(*common, *affine, ws.data_ptr(), st)
        else:
            rc = fn(*common, *affine, st)
        _lib.check(rc, "linear")
        return out

    plain = run(lib.mnf_linear_forward_tc if tc else lib.mnf_linear_forward)
    null = run(lib.mnf_linear_forward_tc_affine if tc else lib.mnf_linear_forward_affine, None, None)
    ones, zeros = torch.ones(n_out, device=DEV), torch.zeros(n_out, device=DEV)
    unit = run(lib.mnf_linear_forward_tc_affine if tc else lib.mnf_linear_forward_affine, ones.data_ptr(), zeros.data_ptr())
    scale, shift = torch.randn(n_out, device=DEV), torch.randn(n_out, device=DEV)
    aff = run(lib.mnf_linear_forward_tc_affine if tc else lib.mnf_linear_forward_affine, scale.data_ptr(), shift.data_ptr())
    assert torch.equal(plain.view(torch.int32), null.view(torch.int32))
    assert torch.equal(plain, unit)  # 1 * v + 0 == v (up to the sign of a zero)
    torch.testing.assert_close(aff, torch.addcmul(shift, scale, plain), rtol=1e-6, atol=1e-6)
    # the module path (which now calls the _affine entry points with NULL) gives the same bits as before
    nz = ops.Noise(None, x.device, 5, seed=77)
    nz.streams = 3
    mod = ops.linear_forward(layer, x, z, nz, x_rows=x_rows, relu=True, precision="tf32" if tc else "fp32")
    assert torch.equal(mod.view(torch.int32), plain.view(torch.int32))


# ---- 4. sharding ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("precision", ["fp32", "tf32"])
def test_forward_mc_split_at_a_sample_boundary_is_bitwise(precision):
    model = _model([64, 96, 16], seed=9, precision=precision)
    B, S, s0 = 24, 10, 3
    x = torch.randn(B, 64, device=DEV)
    whole = model.forward_mc(x, S, seed=55)
    a = model.forward_mc(x, s0, seed=55)
    b = model.forward_mc(x, S - s0, seed=55, row_offset=s0 * B)
    assert torch.equal(torch.cat([a, b]).view(torch.int32), whole.view(torch.int32))


def test_predict_shares_and_chunks():
    model = _model([16, 32, 3], seed=10)
    B, S, chunk = 13, 12, 4
    x = torch.randn(B, 16, device=DEV)
    full = model.predict(x, S, chunk=chunk, seed=9, sample_range=(0, S))
    assert full.dtype == torch.float64 and full.shape == (2, B, 3)
    total = torch.zeros_like(full)
    for lo in range(0, S, chunk):  # one chunk per share, added in sample order: the bits of the unsharded sums
        total += model.predict(x, S, chunk=chunk, seed=9, sample_range=(lo, lo + chunk))
    assert torch.equal(total, full)
    for other in (1, 5, S):  # other chunkings: same sums up to fp64 rounding
        torch.testing.assert_close(model.predict(x, S, chunk=other, seed=9, sample_range=(0, S)), full, rtol=1e-12,
                                   atol=1e-12)
    from torch_mnf.models.mnf_feed_forward import moments_from_sums

    mean, var = model.predict(x, S, chunk=chunk, seed=9)
    m2, v2 = moments_from_sums(total, S)
    assert torch.equal(mean, m2) and torch.equal(var, v2)


# ---- 5. moments -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("sizes,B,S", [([16, 32, 3], 17, 40), ([256, 256, 10], 64, 12), ([8, 50, 50, 1], 300, 33),
                                       ([24, 40, 300], 5, 9)])
@pytest.mark.parametrize("softmax", [False, True])
def test_predict_moments_match_stacked_samples(sizes, B, S, softmax):
    model = _model(sizes, seed=11)
    x = torch.randn(B, sizes[0], device=DEV)
    y = model.forward_mc(x, S, seed=21).double().view(S, B, -1)
    if softmax:
        y = torch.softmax(y, dim=-1)
    mean, var = model.predict(x, S, seed=21, softmax=softmax)  # one chunk: the very samples stacked above
    assert mean.shape == var.shape == (B, sizes[-1]) and mean.dtype == var.dtype == torch.float32
    torch.testing.assert_close(mean.double(), y.mean(0), rtol=1e-6, atol=1e-7)
    torch.testing.assert_close(var.double(), y.var(0, unbiased=False), rtol=1e-5, atol=1e-9)
    m7, v7 = model.predict(x, S, chunk=7, seed=21, softmax=softmax)  # same draws, sums in another association
    torch.testing.assert_close(m7, mean, rtol=1e-6, atol=1e-7)
    torch.testing.assert_close(v7, var, rtol=1e-5, atol=1e-9)
    if softmax:
        torch.testing.assert_close(mean.sum(-1), torch.ones(B, device=DEV), rtol=1e-5, atol=1e-5)


# ---- 6. fallbacks -----------------------------------------------------------------------------------------------------
def test_tanh_activation_falls_back_with_the_same_draws():
    model = _model([16, 32, 3], seed=12, activation=nn.Tanh, precision="fp32")
    B, S = 6, 4
    x = torch.randn(B, 16, generator=torch.Generator().manual_seed(13))
    tape = _tape(model, B * S, seed=14)
    got = model.forward_mc(x.to(DEV), S, noise=tape)
    assert tape.pos == len(tape.draws)
    ref = _oracle(model, x, S, tape.rewind(), act=torch.tanh)
    torch.testing.assert_close(got.cpu().double(), ref, rtol=1e-4, atol=1e-5 * max(1.0, float(ref.abs().mean())))
    xd = x.to(DEV)
    torch.testing.assert_close(model.forward_mc(xd, S, seed=3), _unfused(model, xd, S, seed=3), rtol=0, atol=0)


def test_training_mode_batch_norm_uses_statistics_of_all_rows():
    model = _model([16, 32, 3], seed=15)
    model.train()
    twin = copy.deepcopy(model)
    B, S = 10, 6
    x = torch.randn(B, 16, device=DEV)
    got = model.forward_mc(x, S, seed=8)
    ref = _unfused(twin, x, S, seed=8)  # BatchNorm1d module in training mode over all B * S rows
    torch.testing.assert_close(got, ref, rtol=0, atol=0)
    torch.testing.assert_close(model[2].running_mean, twin[2].running_mean, rtol=0, atol=0)
    torch.testing.assert_close(model[2].running_var, twin[2].running_var, rtol=0, atol=0)
    with pytest.raises(RuntimeError, match="eval mode"):
        model.predict(x, 4)


def test_grad_enabled_takes_the_differentiable_path():
    model = _model([16, 32, 3], seed=16)
    B, S = 5, 3
    x = torch.randn(B, 16, generator=torch.Generator().manual_seed(17))
    tape = _tape(model, B * S, seed=18)
    with torch.enable_grad():
        y = model.forward_mc(x.to(DEV), S, noise=tape)
        assert y.requires_grad
        (y * torch.randn_like(y)).sum().backward()
    ref = _oracle(model, x, S, tape.rewind())
    torch.testing.assert_close(y.detach().cpu().double(), ref, rtol=1e-4, atol=1e-5 * max(1.0, float(ref.abs().mean())))
    for lin in _linears(model):
        for name, p in lin.named_parameters():
            if name.startswith(("r0_", "flow_r.")):  # kl_div's auxiliary posterior: not part of the forward pass
                continue
            assert p.grad is not None and torch.isfinite(p.grad).all() and p.grad.abs().sum() > 0, name
    bn = model[2]
    for p in (bn.weight, bn.bias):
        assert p.grad is not None and p.grad.abs().sum() > 0
