"""Argument checks of the MNF training primitives (csrc/mnf_train.cu) without a GPU: every call below returns its
documented error code, or 0 for an empty problem, before any device work; and the ctypes binding of each primitive
matches its declaration in include/mnf_b200.h argument for argument."""

import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FAKE = 1 << 20  # a non-NULL, 16-byte aligned address: every call below returns before it is dereferenced
E_ARG, E_SHAPE = -1, -2
PRIMITIVES = ("mnf_gemm_f32", "mnf_gemm_f32_batched", "mnf_ew", "mnf_colsum", "mnf_rowsum", "mnf_swap01",
              "mnf_rnvp_gate_forward", "mnf_rnvp_gate_backward", "mnf_kl_rows_forward", "mnf_kl_rows_backward")


def _handle():
    import torch_mnf.layers  # noqa: F401  (registers the training entry points)
    from torch_mnf import _lib

    return _lib.lib()


def _header_args(name):
    src = open(os.path.join(ROOT, "include", "mnf_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    m = re.search(r"\bint\s+" + name + r"\s*\(([^)]*)\)\s*;", src)
    assert m, f"{name} is not declared in the header"
    return [a.strip() for a in m.group(1).split(",") if a.strip()]


def _ctype(decl):
    if "*" in decl:
        return ctypes.c_void_p
    if decl.startswith("int64_t"):
        return ctypes.c_int64
    if decl.startswith("float"):
        return ctypes.c_float
    assert decl.startswith("int "), decl
    return ctypes.c_int


@pytest.mark.parametrize("name", PRIMITIVES)
def test_binding_matches_the_header(name):
    from torch_mnf import _lib

    fn = getattr(_handle(), name)
    assert name in _lib.declared_symbols()
    assert fn.restype is ctypes.c_int
    want = [_ctype(a) for a in _header_args(name)]
    assert list(fn.argtypes) == want, f"{name}: bound {fn.argtypes}, declared {_header_args(name)}"


def _gemm(lib, M=4, N=4, K=4, A=FAKE):
    return lib.mnf_gemm_f32(0, 0, M, N, K, A, 4, FAKE, 4, None, 0.0, FAKE, 4, None)


def _batched(lib, batch=2, M=4, N=4, K=4):
    return lib.mnf_gemm_f32_batched(1, 1, batch, M, N, K, FAKE, 4, 16, FAKE, 4, 16, None, 0.0, FAKE, 4, 16, None)


def test_gemm_argument_errors():
    lib = _handle()
    for kw in ({"M": -1}, {"N": -1}, {"K": -1}):
        assert _gemm(lib, **kw) == E_ARG and b"negative" in lib.mnf_last_error(), kw
        assert _batched(lib, **kw) == E_ARG and b"negative" in lib.mnf_last_error(), kw
    assert _gemm(lib, A=None) == E_ARG and b"NULL" in lib.mnf_last_error()
    assert _batched(lib, batch=65536) == E_ARG and b"batch" in lib.mnf_last_error()
    assert _batched(lib, batch=-1) == E_ARG and b"batch" in lib.mnf_last_error()
    # one launch covers at most 65535 row tiles of 64
    assert _batched(lib, M=65535 * 64 + 1) == E_SHAPE and b"too large" in lib.mnf_last_error()
    assert _gemm(lib, M=65535 * 64 + 1) == E_SHAPE and b"too large" in lib.mnf_last_error()
    # empty products: nothing launched
    assert _gemm(lib, M=0) == 0 and _gemm(lib, N=0) == 0 and _batched(lib, batch=0) == 0


def test_ew_argument_errors():
    lib = _handle()

    def call(op=1, n=8, ncols=1, a=FAKE, out=FAKE):
        return lib.mnf_ew(op, a, FAKE, FAKE, FAKE, out, FAKE, n, ncols, None)

    for op in (0, 17, -1):
        assert call(op=op) == E_ARG and b"unknown elementwise op" in lib.mnf_last_error(), op
    for ncols in (0, -3):
        assert call(ncols=ncols) == E_ARG, ncols
    assert call(n=-1) == E_ARG
    assert call(a=None) == E_ARG and call(out=None) == E_ARG
    assert call(n=0) == 0  # empty: nothing launched


def test_colsum_argument_errors():
    lib = _handle()
    for N in (0, -1):
        assert lib.mnf_colsum(FAKE, None, 10, N, FAKE, None) == E_ARG, N
    assert lib.mnf_colsum(FAKE, FAKE, -1, 4, FAKE, None) == E_ARG
    assert lib.mnf_colsum(None, None, 10, 4, FAKE, None) == E_ARG
    assert lib.mnf_colsum(FAKE, None, 10, 4, None, None) == E_ARG


def test_swap01_rowsum_and_rnvp_gate_argument_errors():
    lib = _handle()
    assert lib.mnf_swap01(FAKE, FAKE, 2, 3, 4, None) == E_ARG and b"aliased" in lib.mnf_last_error()
    assert lib.mnf_swap01(None, FAKE, 2, 3, 4, None) == E_ARG
    assert lib.mnf_swap01(FAKE, FAKE + 4096, 0, 3, 4, None) == 0
    assert lib.mnf_rowsum(None, 4, 4, FAKE, None) == E_ARG
    assert lib.mnf_rowsum(FAKE, 0, 4, FAKE, None) == 0
    assert lib.mnf_rnvp_gate_forward(FAKE, FAKE, FAKE, None, FAKE, FAKE, 4, 4, None) == E_ARG
    assert lib.mnf_rnvp_gate_forward(FAKE, FAKE, FAKE, FAKE, FAKE, FAKE, 0, 4, None) == 0
    # grad_out / grad_log_det may be NULL, the outputs may not
    assert lib.mnf_rnvp_gate_backward(FAKE, FAKE, FAKE, FAKE, None, None, FAKE, FAKE, None, 4, 4, None) == E_ARG
    assert lib.mnf_rnvp_gate_backward(FAKE, FAKE, FAKE, FAKE, None, None, FAKE, FAKE, FAKE, 0, 4, None) == 0


def _kl_fwd(lib, n_out, n_in, z=FAKE):
    return lib.mnf_kl_rows_forward(z, FAKE, FAKE, FAKE, FAKE, FAKE, FAKE, n_out, n_in, None)


def _kl_bwd(lib, n_out, n_in, z=FAKE):
    return lib.mnf_kl_rows_backward(z, *([FAKE] * 10), n_out, n_in, None)


def test_kl_rows_refuse_negative_sizes():
    lib = _handle()
    for n_out, n_in in ((-1, 4), (4, -1), (-5, -5)):
        assert _kl_fwd(lib, n_out, n_in) == E_ARG and b"negative size" in lib.mnf_last_error(), (n_out, n_in)
        assert _kl_bwd(lib, n_out, n_in) == E_ARG and b"negative size" in lib.mnf_last_error(), (n_out, n_in)
    assert _kl_fwd(lib, 4, 4, z=None) == E_ARG and b"NULL" in lib.mnf_last_error()
    assert _kl_bwd(lib, 4, 4, z=None) == E_ARG and b"NULL" in lib.mnf_last_error()


def test_kl_rows_empty_problems_return_before_device_work():
    lib = _handle()
    assert _kl_fwd(lib, 0, 4) == 0 and _kl_fwd(lib, 0, 0) == 0  # no rows to write
    assert _kl_bwd(lib, 4, 0) == 0 and _kl_bwd(lib, 0, 0) == 0  # no columns to write
