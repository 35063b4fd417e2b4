"""Monte-Carlo predictive uncertainty without a GPU: argument checks of mnf_mc_class_moments and of the ops.mc_moments
wrapper's entropy_sums, the finishing formula of uncertainty_from_sums against fp64 torch, the argument errors of both
models' predict_uncertainty."""

import ctypes
import math

import pytest
import torch

from tests.test_mnf_feed_forward_host import FAKE, _handle


def test_class_moments_symbol_is_declared_and_bound():
    from torch_mnf import _lib

    lib = _handle()
    assert "mnf_mc_class_moments" in _lib.declared_symbols()
    fn = lib.mnf_mc_class_moments
    assert len(fn.argtypes) == 7 and fn.restype is ctypes.c_int


def test_class_moments_argument_errors():
    lib = _handle()

    def call(y=FAKE, n_unique=4, n_samples=3, n_cols=10, sums=FAKE, entropy_sums=FAKE):
        return lib.mnf_mc_class_moments(y, n_unique, n_samples, n_cols, sums, entropy_sums, None)

    assert call(y=None) == -1 and b"NULL" in lib.mnf_last_error()
    assert call(sums=None) == -1 and b"NULL" in lib.mnf_last_error()
    assert call(entropy_sums=None) == -1 and b"NULL" in lib.mnf_last_error()
    assert call(n_unique=0) == -2 and b"bad shape" in lib.mnf_last_error()
    assert call(n_cols=0) == -2 and b"bad shape" in lib.mnf_last_error()
    assert call(n_samples=-1) == -2 and b"bad shape" in lib.mnf_last_error()
    assert call(n_unique=1 << 40, n_samples=1 << 20) == -2 and b"too many" in lib.mnf_last_error()


def test_class_moments_without_samples_leaves_both_buffers_untouched():
    lib = _handle()
    sums = (ctypes.c_double * 8)(*[float(i) + 0.5 for i in range(8)])
    ent = (ctypes.c_double * 2)(7.25, -3.5)
    y = (ctypes.c_float * 8)()
    rc = lib.mnf_mc_class_moments(ctypes.addressof(y), 2, 0, 2, ctypes.addressof(sums), ctypes.addressof(ent), None)
    assert rc == 0
    assert list(sums) == [float(i) + 0.5 for i in range(8)] and list(ent) == [7.25, -3.5]


def test_mc_moments_wrapper_checks_entropy_sums_before_launching():
    from torch_mnf.layers import _mnf_ops as ops

    y = torch.zeros(12, 5)
    sums = torch.zeros(2, 4, 5, dtype=torch.float64)
    with pytest.raises(ValueError, match="softmax"):
        ops.mc_moments(y, 4, 3, sums, entropy_sums=torch.zeros(4, dtype=torch.float64))
    for bad in (torch.zeros(5, dtype=torch.float64), torch.zeros(4, 1, dtype=torch.float64), torch.zeros(4),
                torch.zeros(8, dtype=torch.float64)[::2]):
        with pytest.raises(ValueError, match="entropy_sums"):
            ops.mc_moments(y, 4, 3, sums, softmax=True, entropy_sums=bad)


def _reference(p):
    """fp64 (mean, var, H[p_bar], E_s H[p_s], MI) from stacked probabilities p [S, B, C]."""
    p_bar = p.mean(0)
    h_bar = -torch.special.xlogy(p_bar, p_bar).sum(-1)
    h_s = -torch.special.xlogy(p, p).sum(-1).mean(0)
    return p_bar, p.var(0, unbiased=False), h_bar, h_s, h_bar - h_s


def _sums(p):
    return torch.stack([p.sum(0), (p * p).sum(0)]), (-torch.special.xlogy(p, p).sum(-1)).sum(0)


def test_uncertainty_from_sums_matches_fp64_reference():
    from torch_mnf.models import MCUncertainty, uncertainty_from_sums

    S, C = 6, 5
    g = torch.Generator().manual_seed(11)
    p = torch.softmax(torch.randn(S, 5, C, generator=g, dtype=torch.float64) * 3, dim=-1)
    p[:, 0] = torch.nn.functional.one_hot(torch.tensor(2), C).double()  # one-hot: every entropy 0
    p[:, 1] = 1.0 / C  # uniform: log C everywhere, nothing epistemic
    p[:, 2, 4] = 0.0  # a class no sample gives probability to
    p[:, 2] /= p[:, 2].sum(-1, keepdim=True)
    sums, ent = _sums(p)
    got = uncertainty_from_sums(sums, ent, S)
    assert isinstance(got, MCUncertainty)
    assert got.mean.shape == got.var.shape == (5, C) and got.predictive_entropy.shape == (5,)
    assert all(t.dtype == torch.float32 for t in got)
    mean, var, h_bar, h_s, mi = _reference(p)
    torch.testing.assert_close(got.mean, mean.float())
    torch.testing.assert_close(got.var, var.float(), rtol=1e-6, atol=1e-7)
    torch.testing.assert_close(got.predictive_entropy, h_bar.float())
    torch.testing.assert_close(got.expected_entropy, h_s.float())
    torch.testing.assert_close(got.mutual_information, mi.clamp_min(0).float(), rtol=1e-6, atol=1e-7)
    assert torch.equal(got.predictive_entropy[0], torch.tensor(0.0)) and got.expected_entropy[0] == 0
    assert got.mutual_information[0] == 0
    torch.testing.assert_close(got.predictive_entropy[1], torch.tensor(math.log(C), dtype=torch.float32))
    torch.testing.assert_close(got.expected_entropy[1], torch.tensor(math.log(C), dtype=torch.float32))
    assert not torch.isnan(got.predictive_entropy).any() and not torch.isnan(got.expected_entropy).any()
    assert (got.mutual_information >= 0).all()
    assert (got.mutual_information[3:] > 1e-3).all()  # random rows disagree across samples


def test_uncertainty_from_sums_agreeing_samples_give_exactly_zero_information():
    """All samples equal: H[p_bar] and E_s H[p_s] agree up to rounding, and the mutual information is exactly 0 -- never
    a rounding-negative value."""
    from torch_mnf.models import uncertainty_from_sums

    g = torch.Generator().manual_seed(5)
    row = torch.softmax(torch.randn(7, 10, generator=g, dtype=torch.float64), dim=-1)
    for S in (2, 3, 7):
        p = row.expand(S, 7, 10).clone()
        sums, ent = _sums(p)
        got = uncertainty_from_sums(sums, ent, S)
        exact = -torch.special.xlogy(sums[0] / S, sums[0] / S).sum(-1) - ent / S  # what the clamp sees
        assert (got.mutual_information >= 0).all()
        assert torch.equal(got.mutual_information, exact.clamp_min(0).float())
        assert float(got.mutual_information.max()) < 1e-12
        if S == 2:  # sums of two equal values and their halves are exact: the two entropies are the same bits
            assert torch.equal(got.mutual_information, torch.zeros(7))
        torch.testing.assert_close(got.predictive_entropy, got.expected_entropy, rtol=1e-7, atol=0)


def test_predict_uncertainty_argument_errors_need_no_device():
    from torch_mnf.models import MNFFeedForward, MNFLeNet

    ff = MNFFeedForward([6, 5, 3]).eval()
    lenet = MNFLeNet()
    for model, x in ((ff, torch.zeros(2, 6)), (lenet, torch.zeros(2, 1, 28, 28))):
        with pytest.raises(ValueError, match="n_samples"):
            model.predict_uncertainty(x, n_samples=0)
        with pytest.raises(ValueError, match="chunk"):
            model.predict_uncertainty(x, n_samples=4, chunk=0)
        for rng in ((-1, 2), (3, 2), (0, 5)):
            with pytest.raises(ValueError, match="sample_range"):
                model.predict_uncertainty(x, n_samples=4, sample_range=rng)
        with pytest.raises(RuntimeError, match="CUDA"):  # valid arguments: the CPU input is refused, no fallback
            model.predict_uncertainty(x, n_samples=4)
    with pytest.raises(RuntimeError, match="eval mode"):
        MNFFeedForward([6, 5, 3]).predict_uncertainty(torch.zeros(2, 6), n_samples=4)

