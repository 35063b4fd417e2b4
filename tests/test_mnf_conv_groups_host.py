"""MNFConv2d dilation and groups without a GPU: argument errors of the module and of the new C entry points, output
sizes against torch's conv2d, extra_repr, deepcopy / pickle, state_dict shapes and cross-loading, and the ctypes
binding of the new symbols against include/mnf_b200.h."""

import copy
import ctypes
import os
import pickle
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FAKE = 1 << 20  # a non-NULL, 16-byte aligned address: every call below fails its argument checks before any use
# new symbol -> (the symbol it extends, number of added arguments)
NEW_SYMBOLS = {"mnf_conv2d_forward_geom": ("mnf_conv2d_forward_ps", 2),
               "mnf_conv2d_moments_geom": ("mnf_conv2d_moments_ps", 2),
               "mnf_im2col_t_geom": ("mnf_im2col_t_ps", 1),
               "mnf_col2im_t_geom": ("mnf_col2im_t_ps", 1),
               "mnf_gemm_f32_batched": ("mnf_gemm_f32", 4)}


def _conv(*args, **kw):
    from torch_mnf.layers import MNFConv2d

    return MNFConv2d(*args, **kw)


def _handle():
    import torch_mnf.layers  # noqa: F401  (registers the MNF entry points)
    from torch_mnf import _lib

    return _lib.lib()


@pytest.mark.parametrize("kw,err", [({"dilation": 0}, ValueError), ({"dilation": -1}, ValueError),
                                    ({"groups": 0}, ValueError), ({"groups": -2}, ValueError),
                                    ({"dilation": 2.0}, TypeError), ({"groups": 2.0}, TypeError),
                                    ({"dilation": True}, TypeError), ({"groups": True}, TypeError),
                                    ({"dilation": (2, 2)}, TypeError), ({"groups": (2,)}, TypeError),
                                    ({"dilation": "2"}, TypeError),
                                    ({"groups": 3}, ValueError),   # divides neither 4 nor 6
                                    ({"groups": 4}, ValueError),   # divides n_in = 4, not n_out = 6
                                    ({"groups": 6}, ValueError)])  # divides n_out = 6, not n_in = 4
def test_constructor_argument_errors(kw, err):
    with pytest.raises(err):
        _conv(4, 6, 3, **kw)


def test_groups_error_names_both_channel_counts():
    with pytest.raises(ValueError, match="n_in=4 and n_out=6"):
        _conv(4, 6, 3, groups=4)


def test_dilation_and_groups_are_keyword_only():
    with pytest.raises(TypeError):
        _conv(4, 4, 3, 2, 2, (50,), 0, 1, 2)
    with pytest.raises(TypeError):
        _conv(4, 4, 3, 2, 2, (50,), 0, 1, 1, 2)
    layer = _conv(4, 4, 3, dilation=2, groups=2)
    assert (layer.dilation, layer.groups) == (2, 2)


def test_output_size_matches_torch_conv2d_with_dilation():
    for k in (1, 2, 3, 5):
        for d in (1, 2, 3):
            for p in (0, 1, 2):
                for s in (1, 2, 3):
                    layer = _conv(2, 4, k, padding=p, stride=s, dilation=d, groups=2)
                    for h, w in ((5, 5), (7, 6), (9, 12), (13, 4)):
                        if h + 2 * p < d * (k - 1) + 1 or w + 2 * p < d * (k - 1) + 1:
                            with pytest.raises(ValueError, match="larger than"):
                                layer.output_size(h, w)
                            continue
                        ref = torch.nn.functional.conv2d(torch.zeros(1, 2, h, w), torch.zeros(4, 1, k, k), padding=p,
                                                         stride=s, dilation=d, groups=2)
                        assert layer.output_size(h, w) == tuple(ref.shape[2:]), (k, d, p, s, h, w)


def test_dilated_empty_output_is_refused_before_device_work():
    layer = _conv(3, 3, 3, dilation=3, groups=3)  # extent 7
    assert layer.output_size(7, 7) == (1, 1)
    with pytest.raises(ValueError, match="larger than"):
        layer(torch.zeros(1, 3, 6, 9))
    with torch.enable_grad(), pytest.raises(ValueError, match="larger than"):
        layer(torch.zeros(1, 3, 9, 6))


def test_extra_repr():
    assert _conv(3, 4, 3).extra_repr() == "3, 4, kernel_size=3, padding=0, stride=1"
    assert _conv(3, 4, 3, padding=1, stride=2).extra_repr() == "3, 4, kernel_size=3, padding=1, stride=2"
    assert _conv(3, 4, 3, dilation=2).extra_repr() == "3, 4, kernel_size=3, padding=0, stride=1, dilation=2"
    assert _conv(4, 8, 3, groups=4).extra_repr() == "4, 8, kernel_size=3, padding=0, stride=1, groups=4"
    assert (_conv(4, 8, 3, padding=2, dilation=2, groups=2).extra_repr()
            == "4, 8, kernel_size=3, padding=2, stride=1, dilation=2, groups=2")


def test_deepcopy_and_pickle_keep_the_geometry():
    layer = _conv(6, 12, 3, padding=2, stride=2, dilation=3, groups=3)
    for other in (copy.deepcopy(layer), pickle.loads(pickle.dumps(layer))):
        assert (other.padding, other.stride, other.dilation, other.groups) == (2, 2, 3, 3)
        assert other.extra_repr() == layer.extra_repr()
        assert other.W_mean.shape == (12, 2, 3, 3)
        for k, v in layer.state_dict().items():
            assert torch.equal(other.state_dict()[k], v)


def test_groups_one_draws_the_parameters_of_the_plain_layer():
    torch.manual_seed(3)
    plain = _conv(4, 6, 3)
    torch.manual_seed(3)
    same = _conv(4, 6, 3, dilation=1, groups=1)
    for k, v in plain.state_dict().items():
        assert torch.equal(same.state_dict()[k], v), k


def test_state_dict_shapes_and_cross_loading():
    torch.manual_seed(0)
    plain = _conv(8, 16, 3)
    grouped = _conv(8, 16, 3, groups=4)
    depthwise = _conv(8, 8, 3, groups=8)
    assert list(grouped.state_dict().keys()) == list(plain.state_dict().keys())
    assert not any("dilation" in k or "groups" in k for k in grouped.state_dict())
    for k, v in plain.state_dict().items():
        want = (16, 2, 3, 3) if k in ("W_mean", "W_log_var") else v.shape
        assert grouped.state_dict()[k].shape == want, k
    assert depthwise.W_mean.shape == depthwise.W_log_var.shape == (8, 1, 3, 3)
    # dilation is geometry only: a dilated layer loads an undilated state dict of the same shape and keeps its dilation
    dilated = _conv(8, 16, 3, dilation=2, padding=2)
    dilated.load_state_dict(plain.state_dict(), strict=True)
    assert (dilated.dilation, dilated.padding) == (2, 2)
    for k, v in plain.state_dict().items():
        assert torch.equal(dilated.state_dict()[k], v)
    dg = _conv(8, 16, 3, dilation=3, groups=4)
    dg.load_state_dict(grouped.state_dict(), strict=True)
    assert (dg.dilation, dg.groups) == (3, 4)
    # across different groups the weight shapes differ: load_state_dict names them and keeps the layer's weights
    keep = grouped.W_mean.detach().clone(), grouped.W_log_var.detach().clone()
    with pytest.raises(RuntimeError, match="size mismatch for W_mean"):
        grouped.load_state_dict(plain.state_dict())
    with pytest.raises(RuntimeError, match="size mismatch for W_log_var"):
        plain.load_state_dict(_conv(8, 16, 3, groups=2).state_dict())
    assert grouped.groups == 4
    assert torch.equal(grouped.W_mean, keep[0]) and torch.equal(grouped.W_log_var, keep[1])


def _header_arity(name):
    src = open(os.path.join(ROOT, "include", "mnf_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    m = re.search(r"\b" + name + r"\s*\(([^)]*)\)\s*;", src)
    assert m, f"{name} is not declared in the header"
    return len([a for a in m.group(1).split(",") if a.strip()])


@pytest.mark.parametrize("name", sorted(NEW_SYMBOLS))
def test_new_symbols_are_declared_bound_and_exported(name):
    from torch_mnf import _lib

    lib = _handle()
    assert name in _lib.declared_symbols()
    fn = getattr(lib, name)
    assert fn.restype is ctypes.c_int
    assert len(fn.argtypes) == _header_arity(name)
    old, added = NEW_SYMBOLS[name]
    assert len(fn.argtypes) == len(getattr(lib, old).argtypes) + added
    assert lib.mnf_abi_version() == _lib.ABI_VERSION == 1


def _forward(lib, pad=0, stride=1, dil=1, groups=1, H=8, W=8, ks=3, c_in=4, c_out=6, relu_pool=0, x=FAKE):
    return lib.mnf_conv2d_forward_geom(x, 1, FAKE, FAKE, FAKE, FAKE, None, 0, 0, 0, FAKE, 1, c_in, H, W, c_out, ks,
                                       relu_pool, pad, stride, dil, groups, None)


def test_forward_geom_argument_errors():
    lib = _handle()
    assert _forward(lib, dil=0) == -1 and b"dilation" in lib.mnf_last_error()
    assert _forward(lib, dil=-3) == -1 and b"dilation" in lib.mnf_last_error()
    assert _forward(lib, dil=40000) == -1 and b"dilation" in lib.mnf_last_error()  # tap offsets past the table's range
    assert _forward(lib, groups=0) == -1 and b"groups" in lib.mnf_last_error()
    assert _forward(lib, groups=4) == -1 and b"groups 4 must divide c_in 4 and c_out 6" in lib.mnf_last_error()
    assert _forward(lib, groups=3) == -1 and b"groups" in lib.mnf_last_error()
    assert _forward(lib, pad=-1, dil=2) == -1 and b"padding" in lib.mnf_last_error()
    # 8 x 8 input, k 3, dilation 4: extent 9 > 8, nothing to compute
    assert _forward(lib, dil=4) == -2 and b"larger than" in lib.mnf_last_error()
    # dilation 2, padding 1: OH = (9 + 2 - 5) // 1 + 1 = 7 is odd, so the fused pool is refused
    assert _forward(lib, H=9, W=8, pad=1, dil=2, relu_pool=1) == -2 and b"even" in lib.mnf_last_error()
    assert _forward(lib, dil=2, groups=2, x=None) == -1 and b"NULL" in lib.mnf_last_error()


def test_moments_geom_argument_errors():
    lib = _handle()

    def call(dil=1, groups=1, H=8, n=1):
        return lib.mnf_conv2d_moments_geom(FAKE, None, FAKE, FAKE, FAKE, FAKE, FAKE, n, 4, H, 8, 6, 3, 0, 1, dil, groups,
                                           None)

    assert call(dil=0) == -1 and b"dilation" in lib.mnf_last_error()
    assert call(groups=0) == -1 and b"groups" in lib.mnf_last_error()
    assert call(groups=4) == -1 and b"must divide" in lib.mnf_last_error()
    assert call(dil=4) == -2 and b"bad shape" in lib.mnf_last_error()
    # nothing to do for zero images: success without a launch (and without a device)
    assert call(dil=2, groups=2, n=0) == 0


def test_im2col_col2im_geom_argument_errors():
    lib = _handle()
    for fn in (lib.mnf_im2col_t_geom, lib.mnf_col2im_t_geom):
        assert fn(FAKE, FAKE, 1, 2, 8, 8, 3, 0, 1, 0, None) == -1 and b"dilation" in lib.mnf_last_error()
        assert fn(FAKE, FAKE, 1, 2, 8, 8, 3, -1, 1, 2, None) == -1 and b"padding" in lib.mnf_last_error()
        assert fn(FAKE, FAKE, 1, 2, 8, 8, 3, 0, 1, 4, None) == -2 and b"larger than" in lib.mnf_last_error()
        assert fn(None, FAKE, 1, 2, 8, 8, 3, 1, 1, 2, None) == -1 and b"NULL" in lib.mnf_last_error()
        assert fn(FAKE, FAKE, 0, 2, 8, 8, 3, 1, 2, 3, None) == 0  # empty: nothing launched


def test_gemm_batched_argument_errors():
    lib = _handle()

    def call(batch=2, M=4, A=FAKE):
        return lib.mnf_gemm_f32_batched(0, 0, batch, M, 4, 4, A, 4, 16, FAKE, 4, 16, None, 0.0, FAKE, 4, 16, None)

    assert call(batch=-1) == -1 and b"batch" in lib.mnf_last_error()
    assert call(batch=70000) == -1 and b"batch" in lib.mnf_last_error()
    assert call(M=-1) == -1 and b"negative" in lib.mnf_last_error()
    assert call(A=None) == -1 and b"NULL" in lib.mnf_last_error()
    assert call(batch=0) == 0 and call(M=0) == 0  # empty: nothing launched


def test_tensor_core_conv_refuses_dilation_and_groups():
    from torch_mnf.layers import _mnf_ops as ops

    for kw in ({"dilation": 2}, {"groups": 2}):
        layer = _conv(4, 4, 3, **kw)
        with pytest.raises(ValueError, match="dilation=1, groups=1"):
            ops.conv_forward_tc(layer, torch.zeros(1, 4, 8, 8), None, None)
