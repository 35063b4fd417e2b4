"""MNFConv2d with zero padding and stride on the GPU, against an fp64 CPU restatement of the layer built here from
torch.nn.functional.conv2d(..., padding, stride) and fed the same injected noise:
forward (implicit-GEMM kernel, fused ReLU + pool, image replication, the arithmetic tap path), the moments entry point,
Philox sharding, bitwise equality of the default geometry with the unpadded entry points, gradients of the training
path, kl_div's independence of the geometry, and a short training run."""

import pytest
import torch
import torch.nn.functional as F

from oracle import mnf_cpu
from oracle.noise import NoiseTape

pytestmark = pytest.mark.gpu


def _layer(c_in, c_out, k, pad, stride, seed=0, n_flows_q=2, n_flows_r=2):
    from torch_mnf.layers import MNFConv2d

    torch.manual_seed(seed)
    layer = MNFConv2d(c_in, c_out, k, n_flows_q, n_flows_r, padding=pad, stride=stride)
    with torch.no_grad():
        layer.W_log_var.add_(5.0)  # a variance path of the same order as the mean path
        layer.b_log_var.add_(5.0)
    return layer


def _sd(layer, dtype=torch.float32):
    return {k: v.detach().cpu().clone().to(dtype) for k, v in layer.state_dict().items()}


def _draws(c_out, n_flows_q, out_shape, seed):
    g = torch.Generator().manual_seed(seed)
    d = [("normal", torch.randn(c_out, generator=g))]
    d += [("bernoulli", torch.bernoulli(torch.full((1, c_out), 0.5), generator=g)) for _ in range(n_flows_q)]
    d.append(("normal", torch.randn(out_shape, generator=g)))
    return d


def ref_forward(sd, x, tape, pad, stride):
    """MNFConv2d.forward (mnf_conv.py:67-78) with torch's zero padding and stride."""
    z, _ = mnf_cpu.conv_sample_z(sd, tape)
    W_mean = sd["W_mean"] * z.reshape(-1, 1, 1, 1)
    mean = F.conv2d(x, W_mean, padding=pad, stride=stride)
    var = F.conv2d(x**2, sd["W_log_var"].exp(), bias=sd["b_log_var"].exp(), padding=pad, stride=stride)
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


FORWARD_CASES = [  # (c_in, c_out, k, pad, stride, n, H, W)
    (3, 8, 1, 0, 2, 2, 9, 7),
    (3, 8, 1, 1, 1, 2, 5, 6),
    (3, 8, 1, 2, 2, 2, 5, 8),
    (4, 6, 3, 1, 1, 3, 11, 8),
    (4, 6, 3, 1, 2, 3, 11, 8),
    (4, 6, 3, 2, 1, 2, 7, 9),   # p >= k//2 + 1: whole rows and columns of padding
    (4, 6, 3, 2, 2, 2, 13, 6),
    (4, 6, 3, 0, 2, 2, 10, 7),
    (5, 7, 5, 0, 2, 2, 13, 11),
    (5, 7, 5, 1, 1, 2, 9, 12),
    (5, 7, 5, 2, 1, 2, 8, 8),   # "same"
    (5, 7, 5, 2, 2, 3, 15, 10),
    (2, 70, 3, 1, 2, 4, 17, 16),  # more than one column tile
]


@pytest.mark.parametrize("c_in,c_out,k,pad,stride,n,H,W", FORWARD_CASES)
def test_forward_matches_fp64_conv2d(c_in, c_out, k, pad, stride, n, H, W):
    layer = _layer(c_in, c_out, k, pad, stride, seed=c_in * 100 + k * 10 + pad)
    sd = _sd(layer, torch.float64)
    x = torch.rand(n, c_in, H, W, generator=torch.Generator().manual_seed(k + 7 * pad + 13 * stride))
    draws = _draws(c_out, 2, _oshape(layer, x), seed=5)
    ref = ref_forward(sd, x.double(), NoiseTape(draws), pad, stride)
    tape = NoiseTape(draws)
    got = layer.cuda()(x.cuda(), noise=tape)
    assert tape.pos == len(draws)
    assert got.shape == ref.shape == torch.Size(_oshape(layer, x))
    close(got, ref, f"k{k} p{pad} s{stride}")


def test_wide_filter_takes_the_arithmetic_tap_path():
    """c_in * k * k = 1800 taps: beyond the kernel's 1600-entry tap table, the remaining taps compute their offsets and
    coordinates arithmetically."""
    layer = _layer(200, 16, 3, 1, 1, seed=3)
    sd = _sd(layer, torch.float64)
    x = torch.rand(2, 200, 7, 6, generator=torch.Generator().manual_seed(1))
    for stride in (1, 2):
        layer.stride = stride
        draws = _draws(16, 2, _oshape(layer, x), seed=stride)
        ref = ref_forward(sd, x.double(), NoiseTape(draws), 1, stride)
        close(layer.cuda()(x.cuda(), noise=NoiseTape(draws)), ref, f"1800 taps, stride {stride}")


@pytest.mark.parametrize("k,pad,stride,H,W", [(3, 1, 1, 8, 12), (3, 1, 2, 15, 7), (5, 2, 2, 8, 8), (1, 1, 1, 6, 4)])
def test_fused_relu_pool(k, pad, stride, H, W):
    layer = _layer(3, 5, k, pad, stride, seed=k)
    sd = _sd(layer, torch.float64)
    x = torch.rand(3, 3, H, W, generator=torch.Generator().manual_seed(2))
    draws = _draws(5, 2, _oshape(layer, x), seed=4)
    ref = F.max_pool2d(torch.relu(ref_forward(sd, x.double(), NoiseTape(draws), pad, stride)), 2)
    close(layer.cuda()(x.cuda(), noise=NoiseTape(draws), relu_pool=True), ref, "relu_pool")


def test_fused_relu_pool_refuses_odd_output():
    layer = _layer(3, 5, 3, 1, 2).cuda()
    with pytest.raises(RuntimeError, match="even"):
        layer(torch.rand(2, 3, 9, 8, device="cuda"), relu_pool=True)  # OH = 5


def test_image_replication():
    """n_imgs > len(x): image r reads x[r % len(x)], every replica draws its own eps."""
    layer = _layer(4, 6, 3, 1, 2, seed=9)
    sd = _sd(layer, torch.float64)
    x = torch.rand(3, 4, 10, 9, generator=torch.Generator().manual_seed(3))
    R = 12
    draws = _draws(6, 2, _oshape(layer, x, R), seed=6)
    ref = ref_forward(sd, x.double().repeat(R // 3, 1, 1, 1), NoiseTape(draws), 1, 2)
    close(layer.cuda()(x.cuda(), noise=NoiseTape(draws), n_imgs=R), ref, "n_imgs")
    # the fused pool needs an even output: 12 x 11 gives OH = OW = 6
    x2 = torch.rand(3, 4, 12, 11, generator=torch.Generator().manual_seed(4))
    draws2 = _draws(6, 2, _oshape(layer, x2, R), seed=7)
    ref_pool = F.max_pool2d(torch.relu(ref_forward(sd, x2.double().repeat(R // 3, 1, 1, 1), NoiseTape(draws2), 1, 2)), 2)
    close(layer(x2.cuda(), noise=NoiseTape(draws2), n_imgs=R, relu_pool=True), ref_pool, "n_imgs relu_pool")


@pytest.mark.parametrize("k,pad,stride", [(3, 1, 1), (3, 1, 2), (5, 2, 2), (1, 0, 2)])
def test_moments_match_fp64(k, pad, stride):
    """conv_moments (mnf_conv2d_moments_ps): mean and sd without noise; small shapes that would take the direct kernel
    at padding 0 / stride 1 run the implicit GEMM here."""
    from torch_mnf.layers import _mnf_ops as ops

    layer = _layer(1, 20, k, pad, stride, seed=11).cuda()
    sd = _sd(layer, torch.float64)
    x = torch.rand(5, 1, 14, 13, generator=torch.Generator().manual_seed(8))
    z = torch.rand(20, generator=torch.Generator().manual_seed(9)) + 0.5
    mean, s = ops.conv_moments(layer, x.cuda(), z.cuda())
    x64 = x.double()
    ref_m = F.conv2d(x64, sd["W_mean"] * z.double().view(-1, 1, 1, 1), padding=pad, stride=stride)
    ref_v = F.conv2d(x64**2, sd["W_log_var"].exp(), bias=sd["b_log_var"].exp(), padding=pad, stride=stride)
    close(mean, ref_m, "moments mean")
    close(s, ref_v.sqrt(), "moments sd")


def test_philox_rows_split_by_row_offset_equal_one_call():
    from torch_mnf.layers._mnf_ops import Noise

    layer = _layer(4, 9, 3, 1, 2, seed=4).cuda()
    x = torch.rand(10, 4, 13, 12, device="cuda")
    dev = x.device
    for relu_pool in (False, True):
        x_ = x[..., :12, :] if relu_pool else x
        full = layer(x_, noise=Noise(None, dev, 0, seed=1234), relu_pool=relu_pool)
        assert torch.equal(full, layer(x_, noise=Noise(None, dev, 0, seed=1234), relu_pool=relu_pool))
        lo = layer(x_[:4], noise=Noise(None, dev, 0, seed=1234), relu_pool=relu_pool)
        hi = layer(x_[4:], noise=Noise(None, dev, 4, seed=1234), relu_pool=relu_pool)
        assert torch.equal(torch.cat([lo, hi]), full)
        assert not torch.equal(layer(x_, noise=Noise(None, dev, 0, seed=99), relu_pool=relu_pool), full)
    # replicated images: rows are replicas, keyed by the global replica index
    full = layer(x[:2], noise=Noise(None, dev, 0, seed=7), n_imgs=8)
    lo = layer(x[:2], noise=Noise(None, dev, 0, seed=7), n_imgs=4)
    hi = layer(x[:2], noise=Noise(None, dev, 4, seed=7), n_imgs=4)
    assert torch.equal(torch.cat([lo, hi]), full)


def _raw_forward(fn, layer, x, z, eps, out, R, relu_pool, seed, ps):
    from torch_mnf import _lib

    c_in, H, W = x.shape[1:]
    args = [x.data_ptr(), x.size(0), z.data_ptr(), layer.W_mean.data_ptr(), layer.W_log_var.data_ptr(),
            layer.b_log_var.data_ptr(), eps.data_ptr() if eps is not None else None, seed, 3, 0, out.data_ptr(), R,
            c_in, H, W, layer.n_out, layer.kernel_size, int(relu_pool)]
    rc = fn(*args, *((0, 1) if ps else ()), _lib.stream_ptr(x.device))
    _lib.check(rc, "conv forward")


@pytest.mark.parametrize("c_in,c_out,k,H", [(1, 20, 5, 28), (20, 50, 5, 12), (200, 8, 3, 6), (3, 70, 3, 9)])
def test_default_geometry_new_entry_points_equal_old_bitwise(c_in, c_out, k, H):
    from torch_mnf import _lib

    lib = _lib.lib()
    layer = _layer(c_in, c_out, k, 0, 1, seed=c_in).cuda()
    R = 6
    x = torch.rand(3, c_in, H, H, device="cuda")
    z = torch.rand(c_out, device="cuda") + 0.5
    O = H - k + 1
    pool = O % 2 == 0
    for eps in (None, torch.randn(R, c_out, O, O, device="cuda")):
        for relu_pool in ((False, True) if pool else (False,)):
            shape = (R, c_out, O // 2, O // 2) if relu_pool else (R, c_out, O, O)
            a, b = torch.empty(shape, device="cuda"), torch.empty(shape, device="cuda")
            _raw_forward(lib.mnf_conv2d_forward, layer, x, z, eps, a, R, relu_pool, 321, False)
            _raw_forward(lib.mnf_conv2d_forward_ps, layer, x, z, eps, b, R, relu_pool, 321, True)
            assert torch.equal(a, b)
    ma, sa, mb, sb = (torch.empty(3, c_out, O, O, device="cuda") for _ in range(4))
    common = (x.data_ptr(), z.data_ptr(), layer.W_mean.data_ptr(), layer.W_log_var.data_ptr(),
              layer.b_log_var.data_ptr())
    st = _lib.stream_ptr(x.device)
    _lib.check(lib.mnf_conv2d_moments(*common, ma.data_ptr(), sa.data_ptr(), 3, c_in, H, H, c_out, k, st), "moments")
    _lib.check(lib.mnf_conv2d_moments_ps(*common, mb.data_ptr(), sb.data_ptr(), 3, c_in, H, H, c_out, k, 0, 1, st),
               "moments_ps")
    assert torch.equal(ma, mb) and torch.equal(sa, sb)
    # the training path's im2col / col2im
    from torch_mnf.layers import _train

    cols_old = torch.empty(c_in * k * k, 3 * O * O, device="cuda")
    _train._call("mnf_im2col_t", x.data_ptr(), cols_old.data_ptr(), 3, c_in, H, H, k, device=x.device)
    assert torch.equal(cols_old, _train.im2col_t(x, k, 0, 1))
    g = torch.randn_like(cols_old)
    gx_old = torch.empty_like(x)
    _train._call("mnf_col2im_t", g.data_ptr(), gx_old.data_ptr(), 3, c_in, H, H, k, device=x.device)
    assert torch.equal(gx_old, _train.col2im_t(g, tuple(x.shape), k, 0, 1))


def test_default_geometry_module_with_tape_equals_unpadded_entry_point():
    from torch_mnf import _lib
    from torch_mnf.layers import _mnf_ops as ops

    layer = _layer(20, 50, 5, 0, 1, seed=2).cuda()
    x = torch.rand(4, 20, 12, 12)
    draws = _draws(50, 2, (4, 50, 8, 8), seed=3)
    got = layer(x.cuda(), noise=NoiseTape(draws))
    noise = ops.Noise(NoiseTape(draws), torch.device("cuda"))
    z, _ = layer.sample_z(noise)
    eps = draws[-1][1].cuda()
    want = torch.empty_like(got)
    _raw_forward(_lib.lib().mnf_conv2d_forward, layer, x.cuda(), z.contiguous(), eps, want, 4, False, 0, False)
    assert torch.equal(got, want)


def test_im2col_col2im_are_adjoint():
    """<im2col(x), g> == <x, col2im(g)> for padded, strided and overlapping windows."""
    from torch_mnf.layers import _train

    gen = torch.Generator(device="cuda").manual_seed(0)
    for (k, pad, stride, H, W) in ((3, 1, 1, 7, 9), (3, 1, 2, 9, 8), (5, 2, 2, 11, 10), (3, 3, 2, 5, 6), (1, 1, 3, 7, 7),
                                   (2, 0, 1, 5, 5)):
        x = torch.randn(2, 3, H, W, device="cuda", generator=gen)
        cols = _train.im2col_t(x, k, pad, stride)
        ref = F.unfold(x.double(), k, padding=pad, stride=stride)  # [R, C*k*k, L]
        assert torch.equal(cols.double(), ref.permute(1, 0, 2).reshape(cols.shape))
        g = torch.randn(cols.shape, device="cuda", generator=gen)
        gx = _train.col2im_t(g, tuple(x.shape), k, pad, stride)
        ref_gx = F.fold(g.double().reshape(cols.size(0), 2, -1).permute(1, 0, 2), (H, W), k, padding=pad, stride=stride)
        torch.testing.assert_close(gx.double(), ref_gx, rtol=1e-6, atol=1e-5)


def _sd64(sd):
    return {k: (v.double().requires_grad_() if v.is_floating_point() else v) for k, v in sd.items()}


@pytest.mark.parametrize("k,pad,stride", [(3, 1, 1), (3, 1, 2), (5, 2, 2), (3, 2, 3)])
def test_gradients_match_fp64_autograd(k, pad, stride):
    with torch.enable_grad():
        layer = _layer(3, 4, k, pad, stride, seed=k * 10 + stride)
        sd = _sd(layer)
        layer.cuda()
        x = torch.rand(2, 3, 11, 10, generator=torch.Generator().manual_seed(1))
        shape = _oshape(layer, x)
        fwd = _draws(4, 2, shape, seed=2)
        g = torch.Generator().manual_seed(3)
        # kl_div: z0 eps, flow_q masks, eps_w [c_in*k*k], eps_b (), flow_r masks (mnf_conv.py:90-133)
        kl_draws = ([("normal", torch.randn(4, generator=g))]
                    + [("bernoulli", torch.bernoulli(torch.full((1, 4), 0.5), generator=g)) for _ in range(2)]
                    + [("normal", torch.randn(3 * k * k, generator=g)), ("normal", torch.randn((), generator=g))]
                    + [("bernoulli", torch.bernoulli(torch.full((1, 4), 0.5), generator=g)) for _ in range(2)])
        w = torch.randn(shape, generator=torch.Generator().manual_seed(5), dtype=torch.float64)

        sd64 = _sd64(sd)
        x64 = x.double().requires_grad_()
        y_ref = ref_forward(sd64, x64, NoiseTape(fwd), pad, stride)
        ((y_ref * w).sum() + mnf_cpu.conv_kl_div(sd64, NoiseTape(kl_draws))).backward()

        xg = x.cuda().requires_grad_()
        y = layer(xg, noise=NoiseTape(fwd))
        assert y.requires_grad
        close(y, y_ref, "training forward")
        kl = layer.kl_div(noise=NoiseTape(kl_draws))
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


def test_kl_div_does_not_depend_on_the_geometry():
    from torch_mnf.layers import MNFConv2d

    plain = _layer(6, 10, 3, 0, 1, seed=5).cuda()
    geo = MNFConv2d(6, 10, 3, padding=2, stride=2).cuda()
    geo.load_state_dict(plain.state_dict())
    torch.manual_seed(42)  # the Philox seed of an untaped call follows torch's generator
    a = plain.kl_div()
    torch.manual_seed(42)
    b = geo.kl_div()
    assert torch.equal(a, b)
    kl_draws = _draws(10, 2, (6 * 9,), seed=1)
    g = torch.Generator().manual_seed(2)
    kl_draws += [("normal", torch.randn((), generator=g))]
    kl_draws += [("bernoulli", torch.bernoulli(torch.full((1, 10), 0.5), generator=g)) for _ in range(2)]
    assert torch.equal(plain.kl_div(noise=NoiseTape(kl_draws)), geo.kl_div(noise=NoiseTape(kl_draws)))
    with torch.enable_grad():
        ka, kb = plain.kl_div(noise=NoiseTape(kl_draws)), geo.kl_div(noise=NoiseTape(kl_draws))
    assert torch.equal(ka.detach(), kb.detach())


def test_padded_cnn_trains():
    """Two padded MNF conv layers (a "same" 3x3 conv, then a strided one) and a linear read-out on synthetic 16x16
    data: 50 Adam steps must lower nll + kl / N."""
    from torch_mnf.layers import MNFConv2d

    torch.manual_seed(0)
    n_cls, N = 4, 256
    templates = torch.rand(n_cls, 1, 16, 16, device="cuda")
    y = torch.arange(N, device="cuda") % n_cls
    x = (templates[y] + 0.3 * torch.randn(N, 1, 16, 16, device="cuda")).clamp(0, 1)

    class Net(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.c1 = MNFConv2d(1, 8, 3, padding=1)             # 16 x 16
            self.c2 = MNFConv2d(8, 16, 3, padding=1, stride=2)  # 8 x 8
            self.fc = torch.nn.Linear(16 * 4 * 4, n_cls)

        def forward(self, x):
            h = self.c1(x, relu_pool=False).relu()
            h = self.c2(h, relu_pool=True)                      # 4 x 4
            return torch.log_softmax(self.fc(h.flatten(1)), -1)

        def kl_div(self):
            return self.c1.kl_div() + self.c2.kl_div()

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
