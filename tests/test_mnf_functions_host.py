"""Posterior function samples without a GPU: the header documents and the binding declares mnf_linear_sample_weights and
mnf_linear_function_forward, both check their arguments before any device use, the Python methods raise their argument
errors before touching the device, and the new kernels do not spill."""

import ctypes
import os
import re

import pytest
import torch
from torch import nn

from tests.test_mnf_feed_forward_host import FAKE, _handle, _ptxas_report

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_new_symbols_are_declared_and_bound():
    from torch_mnf import _lib

    lib = _handle()
    for name, n_args in (("mnf_linear_sample_weights", 17), ("mnf_linear_function_forward", 13)):
        assert name in _lib.declared_symbols()
        fn = getattr(lib, name)
        assert len(fn.argtypes) == n_args and fn.restype is ctypes.c_int


def test_header_documents_both_entry_points():
    src = open(os.path.join(ROOT, "include", "mnf_b200.h")).read()
    for name, words in (("mnf_linear_sample_weights", ("sample_offset", "NULL", "w_noise_stream", "64-bit")),
                        ("mnf_linear_function_forward", ("x_per_sample", "65535", "col_scale"))):
        m = re.search(r"/\*((?:(?!\*/).)*)\*/\s*int " + name + r"\(", src, flags=re.S)
        assert m, f"{name} has no comment directly above its declaration"
        assert all(w in m.group(1) for w in words), name


def _weights(W_out=FAKE, b_out=FAKE, z=FAKE, sample_offset=0, n_samples=4, n_in=8, n_out=3):
    return _handle().mnf_linear_sample_weights(FAKE, FAKE, FAKE, FAKE, z, None, None, 1, 3, 4, sample_offset, W_out,
                                               b_out, n_samples, n_in, n_out, None)


def test_sample_weights_argument_errors():
    lib = _handle()
    for kw in ({"W_out": None}, {"b_out": None}, {"z": None}):
        assert _weights(**kw) == -1 and b"NULL" in lib.mnf_last_error()
    for kw in ({"n_samples": -1}, {"n_in": 0}, {"n_out": 0}):
        assert _weights(**kw) == -1 and b"bad shape" in lib.mnf_last_error()
    assert _weights(n_samples=1 << 40, n_in=1 << 20, n_out=1 << 10) == -2 and b"too large" in lib.mnf_last_error()
    assert _weights(sample_offset=1 << 62) == -2 and b"sample_offset" in lib.mnf_last_error()
    assert _weights(n_samples=0) == 0  # nothing to draw


def _gemm(x=FAKE, out=FAKE, x_per_sample=0, n_samples=4, batch=5, n_in=8, n_out=3, scale=None, shift=None):
    return _handle().mnf_linear_function_forward(x, x_per_sample, FAKE, FAKE, out, n_samples, batch, n_in, n_out, 1,
                                                 scale, shift, None)


def test_function_forward_argument_errors():
    lib = _handle()
    assert _gemm(x=None) == -1 and b"NULL" in lib.mnf_last_error()
    assert _gemm(out=None) == -1 and b"NULL" in lib.mnf_last_error()
    assert _gemm(scale=FAKE) == -1 and b"col_scale and col_shift" in lib.mnf_last_error()
    assert _gemm(shift=FAKE) == -1 and b"col_scale and col_shift" in lib.mnf_last_error()
    assert _gemm(x_per_sample=2) == -1 and b"x_per_sample" in lib.mnf_last_error()
    for kw in ({"n_samples": -1}, {"batch": -1}, {"n_in": 0}, {"n_out": 0}):
        assert _gemm(**kw) == -1 and b"bad shape" in lib.mnf_last_error()
    assert _gemm(n_samples=65536) == -2 and b"65535" in lib.mnf_last_error()
    assert _gemm(batch=1 << 31) == -2 and b"too large" in lib.mnf_last_error()
    assert _gemm(n_samples=0) == 0 and _gemm(batch=0) == 0  # an empty call is a no-op


def test_linear_methods_raise_argument_errors_before_device_work():
    from torch_mnf.layers import MNFLinear

    layer = MNFLinear(6, 3)  # CPU parameters: any device work would fail with the CUDA error instead
    for kw in ({"n_samples": 0}, {"n_samples": 2, "sample_offset": -1}):
        with pytest.raises(ValueError, match="n_samples|sample_offset"):
            layer.sample_weights(**kw)
        with pytest.raises(ValueError, match="n_samples|sample_offset"):
            layer.forward_functions(torch.zeros(2, 6), **kw)
    for x in (torch.zeros(2, 5), torch.zeros(3, 2, 6), torch.zeros(2, 2, 5), torch.zeros(6)):
        with pytest.raises(ValueError, match="expected"):
            layer.forward_functions(x, 2)
    with pytest.raises(TypeError):
        layer.forward_functions([[0.0] * 6], 2)
    with pytest.raises(RuntimeError, match="CUDA"):
        layer.sample_weights(2)
    with pytest.raises(RuntimeError, match="CUDA"):  # valid arguments: the CPU input is refused, no fallback
        layer.forward_functions(torch.zeros(2, 2, 6), 2)


def test_feed_forward_raises_argument_errors_before_device_work():
    from torch_mnf.models import MNFFeedForward

    model = MNFFeedForward([6, 5, 3]).eval()
    x = torch.zeros(2, 6)
    for kw, what in (({"n_samples": 0}, "n_samples"), ({"n_samples": 2, "chunk": 0}, "chunk"),
                     ({"n_samples": 2, "sample_offset": -3}, "sample_offset")):
        with pytest.raises(ValueError, match=what):
            model.forward_functions(x, **kw)
    with pytest.raises(ValueError, match="expected"):
        model.forward_functions(torch.zeros(2, 5), 2)
    with pytest.raises(RuntimeError, match="CUDA"):
        model.forward_functions(x, 2)
    with pytest.raises(RuntimeError, match="eval mode"):
        MNFFeedForward([6, 5, 3]).forward_functions(x, 2)
    no_stats = MNFFeedForward([6, 5, 3]).eval()
    no_stats[2] = nn.BatchNorm1d(5, track_running_stats=False)
    with pytest.raises(RuntimeError, match="eval mode"):
        no_stats.forward_functions(x, 2)


def test_function_chunk_budget():
    from torch_mnf.layers import _mnf_ops as ops

    assert ops.function_chunk(4096 * 4097) == 1  # one sample's image is over the budget: still one per chunk
    assert ops.function_chunk(1024 * 1025) == ops.FUNCTION_IMAGE_BYTES // (4 * 1024 * 1025)
    assert ops.function_chunk(8) == 65535  # at most one function GEMM launch


def test_function_kernels_do_not_spill():
    rep = _ptxas_report("mnf_functions")
    new = {k: v for k, v in rep.items() if "function_weights_kernel" in k or "MnfFunctionProb" in k}
    assert len(new) >= 2 and all(v == (0, 0) for v in new.values()), new
