"""MNFConv2d with dilation and channel groups on the GPU, against an fp64 CPU restatement of the layer built here from
torch.nn.functional.conv2d(..., padding, stride, dilation, groups) and fed the same injected noise: forward on both sides
of the direct / grouped-GEMM dispatch (fused ReLU + pool, image replication, the arithmetic tap path), the moments entry
point, Philox sharding, bitwise equality of the new entry points with the old ones at dilation 1 / one group, dilated
im2col / col2im, gradients of the training path, kl_div of grouped layers, the launch count of a grouped training step
and a short training run of a depthwise-separable network."""

import pytest
import torch
import torch.nn.functional as F

from oracle import mnf_cpu
from oracle.noise import NoiseTape

pytestmark = pytest.mark.gpu

DIRECT_MAX_NG, DIRECT_MAX_TAPS = 8, 4096  # the library's dispatch rule (mnf_layers.cu, run_conv_gemm)


def _layer(c_in, c_out, k, pad=0, stride=1, dil=1, groups=1, seed=0):
    from torch_mnf.layers import MNFConv2d

    torch.manual_seed(seed)
    layer = MNFConv2d(c_in, c_out, k, padding=pad, stride=stride, dilation=dil, groups=groups)
    with torch.no_grad():
        layer.W_log_var.add_(5.0)  # a variance path of the same order as the mean path
        layer.b_log_var.add_(5.0)
    return layer


def _direct(layer):
    """True when the library runs this layer's forward on the grouped direct kernel."""
    ng, taps = layer.n_out // layer.groups, (layer.n_in // layer.groups) * layer.kernel_size**2
    return layer.groups > 1 and ng <= DIRECT_MAX_NG and taps <= DIRECT_MAX_TAPS


def _sd(layer, dtype=torch.float32):
    return {k: v.detach().cpu().clone().to(dtype) for k, v in layer.state_dict().items()}


def _draws(c_out, n_flows_q, out_shape, seed):
    g = torch.Generator().manual_seed(seed)
    d = [("normal", torch.randn(c_out, generator=g))]
    d += [("bernoulli", torch.bernoulli(torch.full((1, c_out), 0.5), generator=g)) for _ in range(n_flows_q)]
    d.append(("normal", torch.randn(out_shape, generator=g)))
    return d


def _geom(layer):
    return dict(padding=layer.padding, stride=layer.stride, dilation=layer.dilation, groups=layer.groups)


def ref_forward(sd, x, tape, geom):
    """MNFConv2d.forward (mnf_conv.py:67-78) with torch's padding, stride, dilation and groups."""
    z, _ = mnf_cpu.conv_sample_z(sd, tape)
    W_mean = sd["W_mean"] * z.reshape(-1, 1, 1, 1)
    mean = F.conv2d(x, W_mean, **geom)
    var = F.conv2d(x**2, sd["W_log_var"].exp(), bias=sd["b_log_var"].exp(), **geom)
    eps = tape.normal(var.shape)
    return mean + var.sqrt() * eps


def close(a, b, what, rtol=1e-4, atol_scale=1e-5):
    a = a.detach().double().cpu()
    b = b.detach().double()
    scale = max(1.0, float(b.abs().mean()))
    torch.testing.assert_close(a, b, rtol=rtol, atol=atol_scale * scale, msg=lambda m: f"{what}: {m}")


def _oshape(layer, x, R=None):
    OH, OW = layer.output_size(x.size(2), x.size(3))
    return (R or x.size(0), layer.n_out, OH, OW)


# (c_in, c_out, groups): one group; 16 channels per group (grouped GEMM); 4 and 2 per group and depthwise with channel
# multiplier 2 and 1 (direct kernel)
GROUPINGS = [(8, 16, 1), (8, 32, 2), (8, 16, 4), (8, 16, 8), (8, 8, 8)]
FORWARD_CASES = [(c_in, c_out, g, d, pad, stride)
                 for (c_in, c_out, g) in GROUPINGS
                 for (d, pad, stride) in ((1, 1, 2), (2, 2, 1), (3, 1, 2))]


@pytest.mark.parametrize("c_in,c_out,groups,dil,pad,stride", FORWARD_CASES)
def test_forward_matches_fp64_conv2d(c_in, c_out, groups, dil, pad, stride):
    layer = _layer(c_in, c_out, 3, pad, stride, dil, groups, seed=groups * 10 + dil)
    sd = _sd(layer, torch.float64)
    x = torch.rand(3, c_in, 15, 11, generator=torch.Generator().manual_seed(dil + 7 * pad + 13 * stride))
    draws = _draws(c_out, 2, _oshape(layer, x), seed=5)
    ref = ref_forward(sd, x.double(), NoiseTape(draws), _geom(layer))
    tape = NoiseTape(draws)
    got = layer.cuda()(x.cuda(), noise=tape)
    assert tape.pos == len(draws)
    assert got.shape == ref.shape == torch.Size(_oshape(layer, x))
    close(got, ref, f"g{groups} d{dil} p{pad} s{stride}")


@pytest.mark.parametrize("c_in,c_out,k,groups,dil,pad,H,W", [
    (4, 140, 3, 2, 2, 2, 9, 10),     # 70 output channels per group: two column tiles of the grouped GEMM
    (400, 40, 3, 2, 2, 1, 7, 6),     # 1800 taps per group on the grouped GEMM: the arithmetic tap path
    (400, 4, 3, 2, 3, 3, 6, 7),      # 1800 taps per group on the direct kernel
    (6, 6, 5, 6, 2, 4, 9, 13),       # depthwise 5x5, "same" at dilation 2
    (12, 24, 1, 3, 3, 0, 5, 4),      # 1x1 grouped: dilation changes nothing
])
def test_wide_and_odd_shapes(c_in, c_out, k, groups, dil, pad, H, W):
    layer = _layer(c_in, c_out, k, pad, 1, dil, groups, seed=c_in)
    sd = _sd(layer, torch.float64)
    x = torch.rand(2, c_in, H, W, generator=torch.Generator().manual_seed(1))
    draws = _draws(c_out, 2, _oshape(layer, x), seed=3)
    ref = ref_forward(sd, x.double(), NoiseTape(draws), _geom(layer))
    close(layer.cuda()(x.cuda(), noise=NoiseTape(draws)), ref, f"{c_in}->{c_out} k{k} g{groups} d{dil}")


def test_dispatch_covers_both_kernels():
    """The cases above run both the direct kernel and the grouped GEMM (the rule the library applies)."""
    kinds = {_direct(_layer(c_in, c_out, 3, groups=g)) for (c_in, c_out, g) in GROUPINGS if g > 1}
    assert kinds == {True, False}


@pytest.mark.parametrize("c_in,c_out,groups,dil,pad,stride", [(8, 32, 2, 2, 2, 1), (8, 8, 8, 2, 2, 1),
                                                              (6, 12, 6, 3, 3, 2), (6, 30, 3, 1, 1, 1)])
def test_fused_relu_pool_and_image_replication(c_in, c_out, groups, dil, pad, stride):
    layer = _layer(c_in, c_out, 3, pad, stride, dil, groups, seed=dil)
    sd = _sd(layer, torch.float64)
    geom = _geom(layer)
    x = torch.rand(3, c_in, 12, 16, generator=torch.Generator().manual_seed(2))
    assert all(v % 2 == 0 for v in layer.output_size(12, 16))
    draws = _draws(c_out, 2, _oshape(layer, x), seed=4)
    ref = F.max_pool2d(torch.relu(ref_forward(sd, x.double(), NoiseTape(draws), geom)), 2)
    close(layer.cuda()(x.cuda(), noise=NoiseTape(draws), relu_pool=True), ref, "relu_pool")
    R = 9
    xr = x.double().repeat(R // 3, 1, 1, 1)
    draws = _draws(c_out, 2, _oshape(layer, x, R), seed=6)
    close(layer(x.cuda(), noise=NoiseTape(draws), n_imgs=R), ref_forward(sd, xr, NoiseTape(draws), geom), "n_imgs")
    draws = _draws(c_out, 2, _oshape(layer, x, R), seed=7)
    ref_pool = F.max_pool2d(torch.relu(ref_forward(sd, xr, NoiseTape(draws), geom)), 2)
    close(layer(x.cuda(), noise=NoiseTape(draws), n_imgs=R, relu_pool=True), ref_pool, "n_imgs relu_pool")


@pytest.mark.parametrize("c_in,c_out,groups,dil,pad", [(8, 32, 2, 2, 1), (8, 8, 8, 3, 3), (8, 16, 4, 1, 0),
                                                       (8, 16, 1, 2, 0)])
def test_moments_match_fp64(c_in, c_out, groups, dil, pad):
    from torch_mnf.layers import _mnf_ops as ops

    layer = _layer(c_in, c_out, 3, pad, 1, dil, groups, seed=11).cuda()
    sd = _sd(layer, torch.float64)
    x = torch.rand(5, c_in, 14, 13, generator=torch.Generator().manual_seed(8))
    z = torch.rand(c_out, generator=torch.Generator().manual_seed(9)) + 0.5
    geom = _geom(layer)
    x64 = x.double()
    ref_m = F.conv2d(x64, sd["W_mean"] * z.double().view(-1, 1, 1, 1), **geom)
    ref_v = F.conv2d(x64**2, sd["W_log_var"].exp(), bias=sd["b_log_var"].exp(), **geom)
    for zz, scale in ((z.cuda(), 1.0), (None, None)):
        mean, s = ops.conv_moments(layer, x.cuda(), zz)
        want = ref_m if scale else F.conv2d(x64, sd["W_mean"], **geom)
        close(mean, want, "moments mean")
        close(s, ref_v.sqrt(), "moments sd")


@pytest.mark.parametrize("c_in,c_out,groups,dil", [(8, 32, 2, 2), (8, 8, 8, 2), (8, 16, 4, 3)])
def test_philox_rows_split_by_row_offset_equal_one_call(c_in, c_out, groups, dil):
    from torch_mnf.layers._mnf_ops import Noise

    layer = _layer(c_in, c_out, 3, dil, 1, dil, groups, seed=4).cuda()
    x = torch.rand(10, c_in, 12, 13, device="cuda")
    dev = x.device
    for relu_pool in (False, True):
        x_ = x[..., :12] if relu_pool else x
        full = layer(x_, noise=Noise(None, dev, 0, seed=1234), relu_pool=relu_pool)
        assert torch.equal(full, layer(x_, noise=Noise(None, dev, 0, seed=1234), relu_pool=relu_pool))
        lo = layer(x_[:4], noise=Noise(None, dev, 0, seed=1234), relu_pool=relu_pool)
        hi = layer(x_[4:], noise=Noise(None, dev, 4, seed=1234), relu_pool=relu_pool)
        assert torch.equal(torch.cat([lo, hi]), full)
        assert not torch.equal(layer(x_, noise=Noise(None, dev, 0, seed=99), relu_pool=relu_pool), full)
    full = layer(x[:2], noise=Noise(None, dev, 0, seed=7), n_imgs=8)
    lo = layer(x[:2], noise=Noise(None, dev, 0, seed=7), n_imgs=4)
    hi = layer(x[:2], noise=Noise(None, dev, 4, seed=7), n_imgs=4)
    assert torch.equal(torch.cat([lo, hi]), full)


def test_direct_kernel_equals_grouped_gemm_bitwise():
    """The direct kernel sums the same products in the same order as the tiled grouped GEMM: a grouped layer with 4
    output channels per group (direct) gives the bits of the same weights run as 16 channels per group with the extra
    channels on the GEMM, channel by channel.  (396 output pixels: the tiled form, not the GEMV form of M <= 4.)"""
    from torch_mnf.layers import _mnf_ops as ops

    small = _layer(8, 8, 3, 2, 1, 2, 2, seed=1).cuda()     # 4 per group: direct
    wide = _layer(8, 32, 3, 2, 1, 2, 2, seed=2).cuda()     # 16 per group: grouped GEMM
    assert _direct(small) and not _direct(wide)
    with torch.no_grad():
        for name in ("W_mean", "W_log_var", "b_log_var"):
            w = getattr(wide, name)
            w.view(2, 16, *w.shape[1:])[:, :4] = getattr(small, name).view(2, 4, *w.shape[1:])
    x = torch.rand(3, 8, 11, 12, device="cuda")
    z = torch.rand(32, device="cuda") + 0.5
    ms, ss = ops.conv_moments(small, x, z.view(2, 16)[:, :4].reshape(8).contiguous())
    mw, sw = ops.conv_moments(wide, x, z)
    assert torch.equal(ms.view(3, 2, 4, 11, 12), mw.view(3, 2, 16, 11, 12)[:, :, :4])
    assert torch.equal(ss.view(3, 2, 4, 11, 12), sw.view(3, 2, 16, 11, 12)[:, :, :4])


def _raw_forward(fn, layer, x, z, eps, out, R, relu_pool, seed, extra):
    from torch_mnf import _lib

    c_in, H, W = x.shape[1:]
    args = [x.data_ptr(), x.size(0), z.data_ptr(), layer.W_mean.data_ptr(), layer.W_log_var.data_ptr(),
            layer.b_log_var.data_ptr(), eps.data_ptr() if eps is not None else None, seed, 3, 0, out.data_ptr(), R,
            c_in, H, W, layer.n_out, layer.kernel_size, int(relu_pool)]
    rc = fn(*args, *extra, _lib.stream_ptr(x.device))
    _lib.check(rc, "conv forward")


@pytest.mark.parametrize("c_in,c_out,k,H,pad,stride", [(1, 20, 5, 28, 0, 1), (20, 50, 5, 12, 0, 1),
                                                       (200, 8, 3, 6, 1, 1), (3, 70, 3, 9, 2, 2), (4, 6, 3, 11, 1, 2)])
def test_geom_entry_points_at_dilation_one_and_one_group_equal_ps_bitwise(c_in, c_out, k, H, pad, stride):
    from torch_mnf import _lib
    from torch_mnf.layers import _train

    lib = _lib.lib()
    layer = _layer(c_in, c_out, k, pad, stride, seed=c_in).cuda()
    R = 6
    x = torch.rand(3, c_in, H, H, device="cuda")
    z = torch.rand(c_out, device="cuda") + 0.5
    O = layer.output_size(H, H)[0]
    for eps in (None, torch.randn(R, c_out, O, O, device="cuda")):
        for relu_pool in ((False, True) if O % 2 == 0 else (False,)):
            shape = (R, c_out, O // 2, O // 2) if relu_pool else (R, c_out, O, O)
            a, b = torch.empty(shape, device="cuda"), torch.empty(shape, device="cuda")
            _raw_forward(lib.mnf_conv2d_forward_ps, layer, x, z, eps, a, R, relu_pool, 321, (pad, stride))
            _raw_forward(lib.mnf_conv2d_forward_geom, layer, x, z, eps, b, R, relu_pool, 321, (pad, stride, 1, 1))
            assert torch.equal(a, b)
    ma, sa, mb, sb = (torch.empty(3, c_out, O, O, device="cuda") for _ in range(4))
    common = (x.data_ptr(), z.data_ptr(), layer.W_mean.data_ptr(), layer.W_log_var.data_ptr(),
              layer.b_log_var.data_ptr())
    st = _lib.stream_ptr(x.device)
    _lib.check(lib.mnf_conv2d_moments_ps(*common, ma.data_ptr(), sa.data_ptr(), 3, c_in, H, H, c_out, k, pad, stride,
                                         st), "moments_ps")
    _lib.check(lib.mnf_conv2d_moments_geom(*common, mb.data_ptr(), sb.data_ptr(), 3, c_in, H, H, c_out, k, pad, stride,
                                           1, 1, st), "moments_geom")
    assert torch.equal(ma, mb) and torch.equal(sa, sb)
    cols_ps = _train.im2col_t(x, k, pad, stride)
    cols_geom = torch.empty_like(cols_ps)
    _train._call("mnf_im2col_t_geom", x.data_ptr(), cols_geom.data_ptr(), 3, c_in, H, H, k, pad, stride, 1,
                 device=x.device)
    assert torch.equal(cols_ps, cols_geom)
    g = torch.randn_like(cols_ps)
    gx_geom = torch.empty_like(x)
    _train._call("mnf_col2im_t_geom", g.data_ptr(), gx_geom.data_ptr(), 3, c_in, H, H, k, pad, stride, 1,
                 device=x.device)
    assert torch.equal(_train.col2im_t(g, tuple(x.shape), k, pad, stride), gx_geom)


def test_dilated_im2col_col2im_match_unfold_fold_and_are_adjoint():
    from torch_mnf.layers import _train

    gen = torch.Generator(device="cuda").manual_seed(0)
    for (k, pad, stride, dil, H, W) in ((3, 2, 1, 2, 7, 9), (3, 1, 2, 2, 9, 8), (5, 4, 2, 2, 11, 10),
                                         (3, 3, 1, 3, 5, 6), (2, 0, 1, 4, 6, 5), (3, 0, 3, 2, 13, 12)):
        x = torch.randn(2, 3, H, W, device="cuda", generator=gen)
        cols = _train.im2col_t(x, k, pad, stride, dil)
        ref = F.unfold(x.double(), k, dilation=dil, padding=pad, stride=stride)  # [R, C*k*k, L]
        assert torch.equal(cols.double(), ref.permute(1, 0, 2).reshape(cols.shape))
        g = torch.randn(cols.shape, device="cuda", generator=gen)
        gx = _train.col2im_t(g, tuple(x.shape), k, pad, stride, dil)
        ref_gx = F.fold(g.double().reshape(cols.size(0), 2, -1).permute(1, 0, 2), (H, W), k, dilation=dil, padding=pad,
                        stride=stride)
        torch.testing.assert_close(gx.double(), ref_gx, rtol=1e-6, atol=1e-5)
        lhs = float((cols.double() * g.double()).sum())
        rhs = float((x.double() * gx.double()).sum())
        assert abs(lhs - rhs) <= 1e-4 * max(1.0, abs(lhs)), (lhs, rhs)


def test_gemm_batched_matches_per_block_products():
    from torch_mnf.layers import _train

    gen = torch.Generator(device="cuda").manual_seed(1)
    G, M, K, N = 5, 7, 70, 33
    for ta, tb in ((False, False), (True, False), (False, True)):
        A = torch.randn(G * (K if ta else M), M if ta else K, device="cuda", generator=gen)
        B = torch.randn(G * (N if tb else K), K if tb else N, device="cuda", generator=gen)
        got = _train.gemm_grouped(A, B, G, trans_a=ta, trans_b=tb)
        for g, (a, b) in enumerate(zip(A.chunk(G), B.chunk(G))):
            want = _train.gemm(a.contiguous(), b.contiguous(), trans_a=ta, trans_b=tb)
            assert torch.equal(got[g * M:(g + 1) * M], want), (ta, tb, g)


def _sd64(sd):
    return {k: (v.double().requires_grad_() if v.is_floating_point() else v) for k, v in sd.items()}


def _kl_draws(c_out, fan, seed):
    g = torch.Generator().manual_seed(seed)
    # kl_div: z0 eps, flow_q masks, eps_w [fan], eps_b (), flow_r masks (mnf_conv.py:90-133)
    return ([("normal", torch.randn(c_out, generator=g))]
            + [("bernoulli", torch.bernoulli(torch.full((1, c_out), 0.5), generator=g)) for _ in range(2)]
            + [("normal", torch.randn(fan, generator=g)), ("normal", torch.randn((), generator=g))]
            + [("bernoulli", torch.bernoulli(torch.full((1, c_out), 0.5), generator=g)) for _ in range(2)])


@pytest.mark.parametrize("c_in,c_out,k,groups,dil,pad,stride", [
    (4, 32, 3, 2, 1, 1, 1),   # 16 per group (training runs batched GEMMs at any grouping)
    (6, 6, 3, 6, 1, 1, 2),    # depthwise
    (6, 12, 3, 6, 2, 2, 1),   # depthwise, multiplier 2, dilated
    (3, 4, 3, 1, 2, 1, 1),    # dilated, one group
    (4, 4, 5, 2, 3, 4, 2),    # dilated, grouped, strided
])
def test_gradients_match_fp64_autograd(c_in, c_out, k, groups, dil, pad, stride):
    with torch.enable_grad():
        layer = _layer(c_in, c_out, k, pad, stride, dil, groups, seed=k * 10 + dil)
        sd = _sd(layer)
        layer.cuda()
        x = torch.rand(2, c_in, 13, 11, generator=torch.Generator().manual_seed(1))
        shape = _oshape(layer, x)
        fwd = _draws(c_out, 2, shape, seed=2)
        kl_draws = _kl_draws(c_out, (c_in // groups) * k * k, seed=3)
        w = torch.randn(shape, generator=torch.Generator().manual_seed(5), dtype=torch.float64)

        sd64 = _sd64(sd)
        x64 = x.double().requires_grad_()
        y_ref = ref_forward(sd64, x64, NoiseTape(fwd), _geom(layer))
        kl_ref = mnf_cpu.conv_kl_div(sd64, NoiseTape(kl_draws))
        ((y_ref * w).sum() + kl_ref).backward()

        xg = x.cuda().requires_grad_()
        y = layer(xg, noise=NoiseTape(fwd))
        assert y.requires_grad
        close(y, y_ref, "training forward")
        kl = layer.kl_div(noise=NoiseTape(kl_draws))
        close(kl, kl_ref, "training kl_div", rtol=1e-4, atol_scale=1e-4)
        ((y * w.cuda().float()).sum() + kl).backward()
        scale = float(x64.grad.abs().max())
        assert float((xg.grad.cpu().double() - x64.grad).abs().max()) <= 3e-4 * scale, "input gradient"
        checked = 0
        for name, p in layer.named_parameters():
            ref = sd64[name].grad
            assert ref is not None and p.grad is not None, name
            scale = float(ref.abs().max()) + 1e-9
            err = float((p.grad.cpu().double() - ref).abs().max())
            assert err <= 3e-4 * scale + 1e-7, f"{name}: max err {err:.3e} vs scale {scale:.3e}"
            checked += 1
        assert checked == len(list(layer.parameters())) >= 8


@pytest.mark.parametrize("c_in,c_out,groups", [(8, 16, 4), (16, 16, 16), (12, 24, 12)])
def test_kl_div_of_grouped_layers(c_in, c_out, groups):
    """kl_div depends on the weights alone: with a tape it matches the oracle, and in Philox mode a grouped layer gives
    what the ungrouped layer MNFConv2d(c_in // groups, c_out, k) holding the same state gives.  The weight terms kl_W
    and kl_b are the same bits; log q and log r carry the flows' log-dets, which the fused kl kernel sums over its
    cluster's CTAs with float atomics in no fixed order, so they (and the total) agree to rounding."""
    from torch_mnf.layers import MNFConv2d

    layer = _layer(c_in, c_out, 3, groups=groups, seed=groups).cuda()
    sd64 = _sd(layer, torch.float64)
    draws = _kl_draws(c_out, (c_in // groups) * 9, seed=groups)
    close(layer.kl_div(noise=NoiseTape(draws)), mnf_cpu.conv_kl_div(sd64, NoiseTape(draws)), "kl_div tape",
          atol_scale=1e-4)
    dense = MNFConv2d(c_in // groups, c_out, 3).cuda()
    dense.load_state_dict(layer.state_dict())
    torch.manual_seed(42)  # the Philox seed of an untaped call follows torch's generator
    a = layer.kl_div()
    terms_a = layer.__dict__["_last_kl_terms"].clone()  # kl, kl_W, kl_b, log_q, log_r
    torch.manual_seed(42)
    b = dense.kl_div()
    terms_b = dense.__dict__["_last_kl_terms"].clone()
    assert torch.isfinite(a) and torch.isfinite(terms_a).all()
    assert torch.equal(terms_a[1:3], terms_b[1:3]), (terms_a, terms_b)
    torch.testing.assert_close(terms_a[[0, 3, 4]], terms_b[[0, 3, 4]], rtol=1e-6, atol=1e-4)
    torch.testing.assert_close(a, b, rtol=1e-6, atol=1e-4)
    with torch.enable_grad():
        ka = layer.kl_div(noise=NoiseTape(draws))
        assert ka.requires_grad
    close(ka, mnf_cpu.conv_kl_div(sd64, NoiseTape(draws)), "kl_div autograd", atol_scale=1e-4)


def _train_step_launches(groups):
    from torch_mnf import _lib

    layer = _layer(32, 32, 3, 1, 1, 1, groups, seed=0).cuda()
    x = torch.rand(4, 32, 10, 10, device="cuda")
    with torch.enable_grad():
        before = _lib.launch_count
        loss = layer(x).square().mean() + layer.kl_div() / 100
        loss.backward()
        return _lib.launch_count - before


def test_training_step_launch_count_does_not_grow_with_groups():
    assert _train_step_launches(2) == _train_step_launches(16) == _train_step_launches(32)


def test_tensor_core_conv_refuses_the_new_geometry():
    from torch_mnf.layers import _mnf_ops as ops

    x = torch.rand(2, 4, 12, 12, device="cuda")
    for kw in ({"dil": 2}, {"groups": 2}, {"groups": 4, "dil": 3}):
        layer = _layer(4, 4, 3, **kw).cuda()
        with pytest.raises(ValueError, match="dilation=1, groups=1"):
            ops.conv_forward_tc(layer, x, torch.ones(4, device="cuda"), ops.Noise(None, x.device))


def test_depthwise_separable_cnn_trains():
    """Two depthwise-separable MNF blocks (depthwise 3x3, then pointwise 1x1; the second depthwise conv dilated) and a
    linear read-out on synthetic 16x16 data: 50 Adam steps must lower nll + kl / N."""
    from torch_mnf.layers import MNFConv2d

    torch.manual_seed(0)
    n_cls, N = 4, 256
    templates = torch.rand(n_cls, 4, 16, 16, device="cuda")
    y = torch.arange(N, device="cuda") % n_cls
    x = (templates[y] + 0.3 * torch.randn(N, 4, 16, 16, device="cuda")).clamp(0, 1)

    class Net(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.dw1 = MNFConv2d(4, 8, 3, padding=1, groups=4)               # channel multiplier 2, 16 x 16
            self.pw1 = MNFConv2d(8, 16, 1)
            self.dw2 = MNFConv2d(16, 16, 3, padding=2, dilation=2, groups=16)  # 16 x 16
            self.pw2 = MNFConv2d(16, 16, 1)
            self.fc = torch.nn.Linear(16 * 8 * 8, n_cls)

        def forward(self, x):
            h = self.pw1(self.dw1(x).relu(), relu_pool=True)  # 8 x 8
            h = self.pw2(self.dw2(h).relu()).relu()
            return torch.log_softmax(self.fc(h.flatten(1)), -1)

        def kl_div(self):
            return sum(m.kl_div() for m in (self.dw1, self.pw1, self.dw2, self.pw2))

    net = Net().cuda()
    adam = torch.optim.Adam(net.parameters(), lr=3e-3)
    losses = []
    with torch.enable_grad():
        for _ in range(50):
            adam.zero_grad()
            loss = F.nll_loss(net(x), y) + net.kl_div() / N
            loss.backward()
            adam.step()
            losses.append(float(loss.detach()))
    assert all(v == v for v in losses)
    assert sum(losses[-5:]) < sum(losses[:5]), losses
    net.eval()
    with torch.no_grad():  # the inference kernels run the trained network
        assert torch.isfinite(net(x[:8])).all()
