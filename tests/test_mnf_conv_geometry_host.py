"""MNFConv2d padding and stride without a GPU: argument errors of the module and of the new C entry points, extra_repr,
deepcopy / pickle, state_dict keys and cross-loading between geometries, and the ctypes arity of the new symbols
against include/mnf_b200.h."""

import copy
import ctypes
import os
import pickle
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FAKE = 1 << 20  # a non-NULL, 16-byte aligned address: every call below fails its argument checks before any use
NEW_SYMBOLS = ("mnf_conv2d_forward_ps", "mnf_conv2d_moments_ps", "mnf_im2col_t_ps", "mnf_col2im_t_ps")


def _conv(*args, **kw):
    from torch_mnf.layers import MNFConv2d

    return MNFConv2d(*args, **kw)


def _handle():
    import torch_mnf.layers  # noqa: F401  (registers the MNF entry points)
    from torch_mnf import _lib

    return _lib.lib()


@pytest.mark.parametrize("kw,err", [({"padding": -1}, ValueError), ({"stride": 0}, ValueError),
                                    ({"stride": -2}, ValueError), ({"padding": 1.0}, TypeError),
                                    ({"padding": "same"}, TypeError), ({"stride": (2, 2)}, TypeError),
                                    ({"padding": True}, TypeError)])
def test_constructor_argument_errors(kw, err):
    with pytest.raises(err):
        _conv(3, 4, 3, **kw)


def test_geometry_is_keyword_only():
    with pytest.raises(TypeError):
        _conv(3, 4, 3, 2, 2, (50,), 1)


def test_empty_output_is_refused_before_device_work():
    layer = _conv(3, 4, 5, padding=1)
    assert layer.output_size(3, 3) == (1, 1)
    with pytest.raises(ValueError, match="larger than"):
        layer.output_size(2, 7)
    # a CPU tensor would hit the "CUDA only" error on any device path: the ValueError comes first
    with pytest.raises(ValueError, match="larger than"):
        layer(torch.zeros(1, 3, 2, 2))
    with torch.enable_grad(), pytest.raises(ValueError, match="larger than"):
        layer(torch.zeros(1, 3, 2, 2))


def test_output_size_matches_torch_conv2d():
    for k in (1, 3, 5):
        for p in (0, 1, 2, 4):
            for s in (1, 2, 3):
                layer = _conv(2, 3, k, padding=p, stride=s)
                for h, w in ((5, 5), (7, 6), (9, 12)):
                    if h + 2 * p < k or w + 2 * p < k:
                        continue
                    ref = torch.nn.functional.conv2d(torch.zeros(1, 2, h, w), torch.zeros(3, 2, k, k), padding=p, stride=s)
                    assert layer.output_size(h, w) == tuple(ref.shape[2:]), (k, p, s, h, w)


def test_extra_repr():
    assert _conv(3, 4, 3, padding=1, stride=2).extra_repr() == "3, 4, kernel_size=3, padding=1, stride=2"
    assert _conv(3, 4, 5).extra_repr() == "3, 4, kernel_size=5, padding=0, stride=1"
    assert "1, 2, kernel_size=3, padding=2, stride=3" in repr(_conv(1, 2, 3, padding=2, stride=3)).splitlines()[1]


def test_deepcopy_and_pickle_keep_the_geometry():
    layer = _conv(3, 4, 3, padding=2, stride=3)
    for other in (copy.deepcopy(layer), pickle.loads(pickle.dumps(layer))):
        assert (other.padding, other.stride, other.kernel_size) == (2, 3, 3)
        assert other.extra_repr() == layer.extra_repr()
        for k, v in layer.state_dict().items():
            assert torch.equal(other.state_dict()[k], v)


def test_state_dict_keys_and_cross_loading():
    torch.manual_seed(0)
    plain = _conv(3, 4, 3)
    torch.manual_seed(1)
    geo = _conv(3, 4, 3, padding=1, stride=2)
    assert list(geo.state_dict().keys()) == list(plain.state_dict().keys())
    assert not any("padding" in k or "stride" in k for k in geo.state_dict())
    geo.load_state_dict(plain.state_dict(), strict=True)
    assert (geo.padding, geo.stride) == (1, 2)
    for k, v in plain.state_dict().items():
        assert torch.equal(geo.state_dict()[k], v)
    other = _conv(3, 4, 3)
    other.load_state_dict(geo.state_dict(), strict=True)
    assert (other.padding, other.stride) == (0, 1)


def _header_arity(name):
    src = open(os.path.join(ROOT, "include", "mnf_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    m = re.search(r"\b" + name + r"\s*\(([^)]*)\)\s*;", src)
    assert m, f"{name} is not declared in the header"
    return len([a for a in m.group(1).split(",") if a.strip()])


@pytest.mark.parametrize("name", NEW_SYMBOLS)
def test_new_symbols_are_declared_bound_and_exported(name):
    from torch_mnf import _lib

    lib = _handle()
    assert name in _lib.declared_symbols()
    fn = getattr(lib, name)
    assert fn.restype is ctypes.c_int
    assert len(fn.argtypes) == _header_arity(name)
    old = name[: -len("_ps")]
    assert len(fn.argtypes) == len(getattr(lib, old).argtypes) + 2  # the old argument list plus pad and stride
    assert lib.mnf_abi_version() == _lib.ABI_VERSION == 1


def test_forward_ps_argument_errors():
    lib = _handle()

    def call(pad=0, stride=1, H=8, W=8, ks=3, relu_pool=0):
        return lib.mnf_conv2d_forward_ps(FAKE, 1, FAKE, FAKE, FAKE, FAKE, None, 0, 0, 0, FAKE, 1, 2, H, W, 3, ks,
                                         relu_pool, pad, stride, None)

    assert call(pad=-1) == -1 and b"padding" in lib.mnf_last_error()
    assert call(stride=0) == -1 and b"stride" in lib.mnf_last_error()
    assert call(H=2, ks=5, pad=1) == -2 and b"larger than" in lib.mnf_last_error()
    # 9 x 8 input, padding 1, stride 2: OH = (9 + 2 - 3) // 2 + 1 = 5 is odd, so the fused pool is refused
    assert call(H=9, W=8, pad=1, stride=2, relu_pool=1) == -2 and b"even" in lib.mnf_last_error()
    assert lib.mnf_conv2d_forward_ps(None, 1, FAKE, FAKE, FAKE, FAKE, None, 0, 0, 0, FAKE, 1, 2, 8, 8, 3, 3, 0, 1, 2,
                                     None) == -1 and b"NULL" in lib.mnf_last_error()


def test_moments_ps_argument_errors():
    lib = _handle()

    def call(pad=0, stride=1, H=8, ks=3):
        return lib.mnf_conv2d_moments_ps(FAKE, None, FAKE, FAKE, FAKE, FAKE, FAKE, 1, 2, H, 8, 3, ks, pad, stride, None)

    assert call(pad=-1) == -1 and b"padding" in lib.mnf_last_error()
    assert call(stride=0) == -1 and b"stride" in lib.mnf_last_error()
    assert call(H=1, ks=5, pad=1) == -2 and b"bad shape" in lib.mnf_last_error()
    # nothing to do for zero images: success without a launch (and without a device)
    assert lib.mnf_conv2d_moments_ps(FAKE, None, FAKE, FAKE, FAKE, FAKE, FAKE, 0, 2, 8, 8, 3, 3, 1, 2, None) == 0


def test_im2col_col2im_ps_argument_errors():
    lib = _handle()
    for fn in (lib.mnf_im2col_t_ps, lib.mnf_col2im_t_ps):
        assert fn(FAKE, FAKE, 1, 2, 8, 8, 3, -1, 1, None) == -1 and b"padding" in lib.mnf_last_error()
        assert fn(FAKE, FAKE, 1, 2, 8, 8, 3, 0, 0, None) == -1 and b"stride" in lib.mnf_last_error()
        assert fn(FAKE, FAKE, 1, 2, 2, 8, 5, 1, 1, None) == -2 and b"larger than" in lib.mnf_last_error()
        assert fn(None, FAKE, 1, 2, 8, 8, 3, 1, 1, None) == -1 and b"NULL" in lib.mnf_last_error()
        assert fn(FAKE, FAKE, 0, 2, 8, 8, 3, 1, 2, None) == 0  # empty: nothing launched
