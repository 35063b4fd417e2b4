"""MNFFeedForward's Monte-Carlo entry points without a GPU: argument checks of mnf_linear_forward_affine,
mnf_linear_forward_tc_affine and mnf_mc_moments, the batch-norm folding arithmetic, the moments formula, and the
compiler's report for the new kernels."""

import ctypes
import os
import re

import pytest
import torch
import torch.nn.functional as F
from torch import nn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FAKE = 1 << 20  # a non-NULL, 16-byte aligned address: every call below fails its argument checks before any use


def _handle():
    import torch_mnf.layers  # noqa: F401  (registers the MNF entry points)
    from torch_mnf import _lib

    return _lib.lib()


def _affine(tc, x=FAKE, scale=None, shift=None, n_rows=8, n_in=32, n_out=16, x_rows=8):
    lib = _handle()
    args = [x, x_rows, FAKE, FAKE, FAKE, FAKE, FAKE, None, 0, 0, 0, FAKE, n_rows, n_in, n_out, 1, scale, shift]
    if tc:
        return lib.mnf_linear_forward_tc_affine(*args, FAKE, None)
    return lib.mnf_linear_forward_affine(*args, None)


def test_new_symbols_are_declared_and_bound():
    from torch_mnf import _lib

    lib = _handle()
    for name, n_args in (("mnf_linear_forward_affine", 19), ("mnf_linear_forward_tc_affine", 20), ("mnf_mc_moments", 7)):
        assert name in _lib.declared_symbols()
        fn = getattr(lib, name)
        assert len(fn.argtypes) == n_args and fn.restype is ctypes.c_int


@pytest.mark.parametrize("tc", [False, True])
def test_linear_affine_argument_errors(tc):
    lib = _handle()
    assert _affine(tc, x=None) == -1 and b"NULL" in lib.mnf_last_error()
    assert _affine(tc, scale=FAKE) == -1 and b"col_scale and col_shift" in lib.mnf_last_error()
    assert _affine(tc, shift=FAKE) == -1 and b"col_scale and col_shift" in lib.mnf_last_error()
    if tc:
        assert _affine(tc, scale=FAKE + 4, shift=FAKE) == -3 and b"16-byte" in lib.mnf_last_error()
        assert _affine(tc, scale=FAKE, shift=FAKE, n_in=30) == -2 and b"n_in" in lib.mnf_last_error()
        assert _affine(tc, scale=FAKE, shift=FAKE, x_rows=0) == -1
    else:
        assert _affine(tc, scale=FAKE, shift=FAKE, n_out=0) == -1 and b"bad shape" in lib.mnf_last_error()
        assert _affine(tc, scale=FAKE, shift=FAKE, n_rows=1 << 30) == -2
    assert _affine(tc, scale=FAKE, shift=FAKE, n_rows=0, x_rows=1) == 0  # an empty batch is a no-op


def test_mc_moments_argument_errors():
    lib = _handle()

    def call(y=FAKE, n_unique=4, n_samples=3, n_cols=10, softmax=0, sums=FAKE):
        return lib.mnf_mc_moments(y, n_unique, n_samples, n_cols, softmax, sums, None)

    assert call(y=None) == -1 and b"NULL" in lib.mnf_last_error()
    assert call(sums=None) == -1 and b"NULL" in lib.mnf_last_error()
    assert call(softmax=2) == -1 and b"softmax" in lib.mnf_last_error()
    assert call(n_unique=0) == -2 and b"bad shape" in lib.mnf_last_error()
    assert call(n_cols=0) == -2 and b"bad shape" in lib.mnf_last_error()
    assert call(n_samples=-1) == -2 and b"bad shape" in lib.mnf_last_error()
    assert call(n_unique=1 << 40, n_samples=1 << 20) == -2 and b"too many" in lib.mnf_last_error()
    assert call(n_samples=0) == 0  # no samples: the sums stay as they are


def test_mc_moments_wrapper_checks_shapes_before_launching():
    from torch_mnf.layers import _mnf_ops as ops

    y = torch.zeros(12, 5)
    with pytest.raises(ValueError, match="do not match"):
        ops.mc_moments(y, 4, 2, torch.zeros(2, 4, 5, dtype=torch.float64))
    with pytest.raises(ValueError, match="float64"):
        ops.mc_moments(y, 4, 3, torch.zeros(2, 4, 5))


def _trained_bn(n, affine, seed):
    g = torch.Generator().manual_seed(seed)
    bn = nn.BatchNorm1d(n, affine=affine, eps=1e-3 if affine else 1e-5)
    with torch.no_grad():
        bn.running_mean.copy_(torch.randn(n, generator=g) * 2)
        bn.running_var.copy_(torch.rand(n, generator=g) * 5 + 0.05)
        if affine:
            bn.weight.copy_(torch.randn(n, generator=g))
            bn.bias.copy_(torch.randn(n, generator=g))
    return bn.eval()


@pytest.mark.parametrize("affine", [True, False])
def test_batch_norm_folding_matches_inference_batch_norm(affine):
    from torch_mnf.models.mnf_feed_forward import fold_batch_norm

    bn = _trained_bn(37, affine, seed=3)
    h = torch.relu(torch.randn(64, 37, generator=torch.Generator().manual_seed(4)) * 3)
    scale, shift = fold_batch_norm(bn)
    assert scale.shape == shift.shape == (37,) and scale.dtype == torch.float32 and scale.is_contiguous()
    ref = F.batch_norm(h.double(), bn.running_mean.double(), bn.running_var.double(),
                       None if bn.weight is None else bn.weight.double(), None if bn.bias is None else bn.bias.double(),
                       training=False, eps=bn.eps)
    got = torch.addcmul(shift, scale, h)  # the epilogue's fmaf(scale, h, shift), up to the fma's single rounding
    torch.testing.assert_close(got.double(), ref, rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(got, bn(h), rtol=1e-5, atol=1e-5)
    if not affine:
        torch.testing.assert_close(scale, 1 / torch.sqrt(bn.running_var + bn.eps))


def test_moments_from_sums():
    from torch_mnf.models.mnf_feed_forward import moments_from_sums

    y = torch.randn(7, 3, 4, dtype=torch.float64)
    y[:, 0, 0] = 0.1  # every sample equal: the variance must come out as 0, not a rounding-negative value
    sums = torch.stack([y.sum(0), (y * y).sum(0)])
    mean, var = moments_from_sums(sums, 7)
    assert mean.dtype == var.dtype == torch.float32
    torch.testing.assert_close(mean, y.mean(0).float())
    torch.testing.assert_close(var, y.var(0, unbiased=False).float(), rtol=1e-6, atol=1e-7)
    assert var[0, 0] >= 0


def test_predict_rejects_batch_statistics_before_touching_the_device():
    from torch_mnf.models import MNFFeedForward

    model = MNFFeedForward([6, 5, 2])  # a fresh model is in training mode
    with pytest.raises(RuntimeError, match="eval mode"):
        model.predict(torch.zeros(3, 6), n_samples=4)


def _ptxas_report(src):
    log = os.path.join(ROOT, "torch-mnf_b200", "build", src + ".ptxas.log")
    if not os.path.exists(log):
        pytest.skip("no compiler report: build the library first (python torch-mnf_b200/build.py)")
    out, cur = {}, None
    for line in open(log):
        m = re.search(r"Compiling entry function '(\w+)'", line)
        if m:
            cur = m.group(1)
            continue
        m = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if cur and m:
            out[cur] = (int(m.group(1)), int(m.group(2)))
            cur = None
    return out


def test_simt_linear_and_moments_kernels_do_not_spill():
    lin = {k: v for k, v in _ptxas_report("mnf_layers").items() if "MnfLinearProb" in k}
    assert len(lin) == 2 and all(v == (0, 0) for v in lin.values()), lin
    mom = _ptxas_report("mnf_moments")
    assert len(mom) == 2 and all(v == (0, 0) for v in mom.values()), mom
