"""Monte-Carlo predictive uncertainty on the GPU: the entropy sums of mnf_mc_class_moments against fp64 torch, and
MNFFeedForward / MNFLeNet.predict_uncertainty against predict, the stacked samples, re-chunking and sharding.

Tolerances: the kernel forms each sample's softmax in fp32 and its entropy in fp64, so per-row mean entropies are held
to 1e-5 absolute of fp64 torch on the same fp32 input.  Sums of the same samples in another chunking differ by fp64
rounding only; predict sums in fp32, so its mean is compared at rtol 1e-6."""

import math

import pytest
import torch

from tests.helpers import golden_sd, load_golden, t
from tests.test_mnf_feed_forward_gpu import _model

pytestmark = pytest.mark.gpu

DEV = "cuda"


def _lib():
    import torch_mnf.layers  # noqa: F401  (registers the MNF entry points)
    from torch_mnf import _lib

    return _lib.lib()


def _entropy64(logits):
    """fp64 entropy of softmax over the last dim, 0 log 0 = 0."""
    logp = torch.log_softmax(logits.double(), dim=-1)
    return -torch.where(logp > -math.inf, logp.exp() * logp, torch.zeros_like(logp)).sum(-1)


def _class_moments(y, n_unique, n_samples, sums=None, ent=None):
    n_cols = y.size(1)
    sums = torch.zeros(2, n_unique, n_cols, device=DEV, dtype=torch.float64) if sums is None else sums
    ent = torch.zeros(n_unique, device=DEV, dtype=torch.float64) if ent is None else ent
    rc = _lib().mnf_mc_class_moments(y.data_ptr(), n_unique, n_samples, n_cols, sums.data_ptr(), ent.data_ptr(), None)
    assert rc == 0, _lib().mnf_last_error()
    return sums, ent


def _logits(S, B, C, seed):
    g = torch.Generator().manual_seed(seed)
    y = torch.randn(S, B, C, generator=g) * 3
    y[:, 0] = 0.0  # uniform rows: log C
    if C > 1:
        y[:, 1, :] = -2.0
        y[:, 1, C // 2] = 1e4  # one-hot gap: every other exp underflows to 0, entropy 0
        y[:, 2, ::2] = -math.inf  # -inf columns add nothing (not NaN)
        y[::2, 3, 1:] = -math.inf  # -inf everywhere but column 0 in every other sample
    return y.view(S * B, C).contiguous()


@pytest.mark.parametrize("n_cols", [1, 10, 128, 129, 300])
def test_class_moments_entropy_matches_fp64(n_cols):
    S, B = 9, 37
    y = _logits(S, B, n_cols, seed=n_cols).to(DEV)
    sums, ent = _class_moments(y, B, S)
    ref = _entropy64(y.view(S, B, n_cols)).mean(0)
    assert not torch.isnan(ent).any()
    torch.testing.assert_close((ent / S).cpu(), ref.cpu(), rtol=0, atol=1e-5)
    torch.testing.assert_close((ent[0] / S).cpu(), torch.tensor(math.log(n_cols), dtype=torch.float64), rtol=0, atol=1e-6)
    if n_cols > 1:
        assert float(ent[1]) == 0.0
    # the probability sums are bitwise those of mnf_mc_moments(softmax = 1)
    plain = torch.zeros_like(sums)
    assert _lib().mnf_mc_moments(y.data_ptr(), B, S, n_cols, 1, plain.data_ptr(), None) == 0
    assert torch.equal(sums, plain)
    p = torch.softmax(y.view(S, B, n_cols).double(), dim=-1)
    torch.testing.assert_close(sums[0].cpu(), p.sum(0).cpu(), rtol=1e-6, atol=1e-6)


def test_class_moments_consecutive_chunks_add_once():
    """Calls over consecutive sample chunks into one buffer give the bits of per-chunk sums formed from zero and added
    in order; a call with no samples changes nothing."""
    S, B, C = 12, 50, 129
    y = _logits(S, B, C, seed=3).to(DEV)
    sums, ent = _class_moments(y, B, 0)
    assert not sums.any() and not ent.any()
    want_s, want_e = torch.zeros_like(sums), torch.zeros_like(ent)
    for lo, hi in ((0, 5), (5, 7), (7, 12)):
        part = y[lo * B:hi * B]
        _class_moments(part, B, hi - lo, sums, ent)
        s, e = _class_moments(part, B, hi - lo)
        want_s += s
        want_e += e
    assert torch.equal(sums, want_s) and torch.equal(ent, want_e)
    one_s, one_e = _class_moments(y, B, S)
    torch.testing.assert_close(ent, one_e, rtol=1e-12, atol=0)
    torch.testing.assert_close(sums, one_s, rtol=1e-12, atol=1e-15)


def _check_identities(u, C):
    tol = 1e-6
    h, e, mi = u.predictive_entropy, u.expected_entropy, u.mutual_information
    assert (mi >= 0).all()
    assert (mi <= h + tol).all() and (h <= math.log(C) + tol).all() and (e <= h + tol).all() and (e >= -tol).all()


@pytest.mark.parametrize("sizes,B,S,chunk,precision", [([16, 32, 10], 33, 12, 5, "fp32"),
                                                       ([64, 256, 256, 10], 64, 24, 10, None)])
def test_feed_forward_predict_uncertainty(sizes, B, S, chunk, precision):
    from torch_mnf.models import uncertainty_from_sums

    model = _model(sizes, seed=5, precision=precision)
    x = torch.randn(B, sizes[0], device=DEV, generator=torch.Generator(device=DEV).manual_seed(6))
    u = model.predict_uncertainty(x, S, chunk=chunk, seed=31)
    mean, var = model.predict(x, S, chunk=chunk, seed=31, softmax=True)
    assert torch.equal(u.mean, mean) and torch.equal(u.var, var)
    assert u.predictive_entropy.shape == u.expected_entropy.shape == u.mutual_information.shape == (B,)
    # against fp64 from the stacked samples (forward_mc in one call: the same draws, keyed by global row)
    y = model.forward_mc(x, S, seed=31).view(S, B, -1)
    p = torch.softmax(y.double(), dim=-1)
    p_bar = p.mean(0)
    h_ref = -torch.special.xlogy(p_bar, p_bar).sum(-1)
    e_ref = _entropy64(y).mean(0)
    torch.testing.assert_close(u.predictive_entropy.double(), h_ref, rtol=0, atol=1e-5)
    torch.testing.assert_close(u.expected_entropy.double(), e_ref, rtol=0, atol=1e-5)
    torch.testing.assert_close(u.mutual_information.double(), (h_ref - e_ref).clamp_min(0), rtol=0, atol=1e-5)
    _check_identities(u, sizes[-1])
    # shares of one chunk each, added in sample order: the unsharded bits
    shares = [model.predict_uncertainty(x, S, chunk=chunk, seed=31, sample_range=(lo, min(lo + chunk, S)))
              for lo in range(0, S, chunk)]
    sums, ent = shares[0]
    for s, e in shares[1:]:
        sums, ent = sums + s, ent + e
    whole = uncertainty_from_sums(sums, ent, S)
    assert all(torch.equal(a, b) for a, b in zip(whole, u))


def _lenet(precision):
    from torch_mnf.models import MNFLeNet

    g = load_golden("mnf_lenet")
    net = MNFLeNet()
    net.load_state_dict(golden_sd(g))
    net.precision = precision
    gen = torch.Generator().manual_seed(8)
    labels = torch.randint(0, 10, (64,), generator=gen)
    x = (t(g, "templates")[labels] + 0.3 * torch.randn(64, 1, 28, 28, generator=gen)).clamp(0, 1)
    x[48:] = torch.rand(16, 1, 28, 28, generator=gen)  # noise images: off the training distribution
    return net.cuda(), x.cuda()


def _reduce(chunks, B):
    sums = torch.zeros(2, B, 10, device=DEV, dtype=torch.float64)
    ent = torch.zeros(B, device=DEV, dtype=torch.float64)
    from torch_mnf.layers import _mnf_ops as ops

    for s_here, lp in chunks:
        ops.mc_moments(lp, B, s_here, sums, softmax=True, entropy_sums=ent)
    return sums, ent


@pytest.mark.parametrize("precision", ["fp32", "auto"])
def test_lenet_predict_uncertainty(precision):
    from torch_mnf.models import uncertainty_from_sums

    net, x = _lenet(precision)
    B, S, chunk, seed = 64, 24, 8, 77  # 512 rows per chunk: the tensor-core branch under "auto"
    u = net.predict_uncertainty(x, n_samples=S, chunk=chunk, seed=seed)
    torch.testing.assert_close(u.mean, net.predict(x, n_samples=S, chunk=chunk, seed=seed), rtol=1e-6, atol=1e-7)
    # entropies against fp64 from the chunked forward log-probs (predict's draws)
    lp = torch.cat([net(x, n_samples=chunk, seed=seed, row_offset=c * B) for c in range(0, S, chunk)]).view(S, B, 10)
    p_bar = torch.softmax(lp.double(), dim=-1).mean(0)
    h_ref = -torch.special.xlogy(p_bar, p_bar).sum(-1)
    e_ref = _entropy64(lp).mean(0)
    torch.testing.assert_close(u.predictive_entropy.double(), h_ref, rtol=0, atol=1e-5)
    torch.testing.assert_close(u.expected_entropy.double(), e_ref, rtol=0, atol=1e-5)
    torch.testing.assert_close(u.mutual_information.double(), (h_ref - e_ref).clamp_min(0), rtol=0, atol=1e-5)
    _check_identities(u, 10)
    # chunk size: fp64 rounding only
    u12 = net.predict_uncertainty(x, n_samples=S, chunk=12, seed=seed)
    for a, b in zip(u12, u):
        torch.testing.assert_close(a, b, rtol=1e-6, atol=1e-7)
    # sharding: shares added in sample order give the unsharded bits
    s1, e1 = net.predict_uncertainty(x, n_samples=S, chunk=chunk, seed=seed, sample_range=(0, 16))
    s2, e2 = net.predict_uncertainty(x, n_samples=S, chunk=chunk, seed=seed, sample_range=(16, 24))
    assert all(torch.equal(a, b) for a, b in zip(uncertainty_from_sums(s1 + s2, e1 + e2, S), u))

    # one conv z per sample: the reduction of per-chunk forward(..., per_sample_conv_z=True), bit for bit
    per = net.predict_uncertainty(x, n_samples=S, chunk=chunk, seed=seed, per_sample_conv_z=True)
    sums, ent = _reduce(((chunk, net(x, n_samples=chunk, seed=seed, row_offset=c * B, per_sample_conv_z=True))
                         for c in range(0, S, chunk)), B)
    assert all(torch.equal(a, b) for a, b in zip(uncertainty_from_sums(sums, ent, S), per))
    s1, e1 = net.predict_uncertainty(x, n_samples=S, chunk=chunk, seed=seed, sample_range=(0, 16), per_sample_conv_z=True)
    s2, e2 = net.predict_uncertainty(x, n_samples=S, chunk=chunk, seed=seed, sample_range=(16, 24),
                                     per_sample_conv_z=True)
    assert torch.equal(s1 + s2, sums) and torch.equal(e1 + e2, ent)
    _check_identities(per, 10)
    assert not torch.equal(per.mean, u.mean) and not torch.equal(per.mutual_information, u.mutual_information)
