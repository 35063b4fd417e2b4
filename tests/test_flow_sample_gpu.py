"""NormalizingFlowModel.sample_and_log_prob / mnf_flow_stack_sample: the Philox draw, parity of x and log q(x) with the
fp64 oracle on the kernel's own z, shard invariance, gradients and a reverse-KL fit."""

import math

import numpy as np
import pytest
import torch

from tests.helpers import golden_sd, golden_spec, load_flow_model, load_golden, random_flow_sd
from tests.test_flow_autograd_gpu import _oracle_stack
from tests.test_flows_gpu import close_vs_oracle

pytestmark = pytest.mark.gpu

CFG2 = [{"type": "ActNormFlow", "dim": 2, "scale": True, "shift": True}, {"type": "Glow", "dim": 2},
        {"type": "NSF_CL", "dim": 2, "K": 8, "B": 3, "n_h": 16}] * 3


def _philox_np(counter, stream, seed):
    """Philox4x32-10 (mnf_common.cuh) over an array of 64-bit counters, in exact integer arithmetic."""
    M0, M1, W0, W1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57), 0x9E3779B9, 0xBB67AE85
    mask = np.uint64(0xFFFFFFFF)
    counter = counter.astype(np.uint64)
    c0, c1 = counter & mask, counter >> np.uint64(32)
    c2, c3 = np.full_like(c0, stream), np.full_like(c0, 0x9E3779B9)
    k0, k1 = seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF
    for _ in range(10):
        p0, p1 = M0 * c0, M1 * c2
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ np.uint64(k0), p1 & mask, (p0 >> np.uint64(32)) ^ c3 ^ np.uint64(k1), p0 & mask
        k0, k1 = (k0 + W0) & 0xFFFFFFFF, (k1 + W1) & 0xFFFFFFFF
    return c0, c1, c2, c3


def philox_normal_np(elements, stream, seed):
    """philox_normal of global elements (fp64 Box-Muller on the kernel's 23-bit uniforms) and the pair's radius."""
    w = _philox_np(elements >> 2, stream, seed)
    lane = elements & 3
    a = np.where(lane >= 2, w[2], w[0]).astype(np.float64)
    b = np.where(lane >= 2, w[3], w[1]).astype(np.float64)
    u1 = 1.0 - np.floor(a / 512.0) / 2.0**23
    u2 = np.floor(b / 512.0) / 2.0**23
    r = np.sqrt(-2.0 * np.log(u1))
    return np.where(lane & 1, r * np.sin(2 * np.pi * u2), r * np.cos(2 * np.pi * u2)), r


def check_draw(z, seed, row_offset):
    """z [n, dim] against the restated generator.  The kernel's Box-Muller runs on MUFU: lg2 (absolute error ~2^-22,
    which moves r^2 = -2 ln u1 by ~3e-7, i.e. r by ~2e-7 / r), sqrt and sin / cos (absolute error ~2^-20.5, times r)."""
    n, dim = z.shape
    e = (np.arange(n, dtype=np.uint64)[:, None] + np.uint64(row_offset)) * np.uint64(dim) + np.arange(dim, dtype=np.uint64)
    ref, r = philox_normal_np(e, 0, seed)
    got = z.double().cpu().numpy()
    tol = 1e-6 + 2e-6 * r + 2e-7 / r
    bad = np.abs(got - ref) > tol
    assert not bad.any(), f"{int(bad.sum())} draws off, worst {float(np.abs(got - ref).max()):.3e}"


def _model(name):
    if name == "cfg2":
        specs, sd = CFG2, random_flow_sd(CFG2, seed=0, scale=0.6)
    else:
        g = load_golden(name)
        specs, sd = golden_spec(g), golden_sd(g)
    return specs, sd, load_flow_model(specs, sd, return_intermediates=False)


def _log_normal64(z):
    z = z.double().cpu()
    return -0.5 * z.square().sum(1) - 0.5 * z.size(1) * math.log(2 * math.pi)


FUSED = ["nsfcl3_stack", "rnvp9_moons", "cfg2"]
FALLBACK = ["maf_iaf_d2", "nsfar2_d3", "maf3_d8", "affine_misc_d4"]


@pytest.mark.parametrize("name", FUSED + FALLBACK)
@torch.no_grad()
def test_draw_and_parity_vs_oracle(name):
    """x vs the oracle's forward pass of the kernel's own z, log q(x) vs log N(z) - log_det of the oracle."""
    specs, sd, model = _model(name)
    prog = model._program()
    dim = specs[0]["dim"]
    n, seed, off = 4099, 0x1234_5678_9ABC, 77
    x, lp, z = prog.sample(n, dim, "cuda", seed, off, want_z=True)
    check_draw(z, seed, off)
    ld_equiv = _log_normal64(z) - lp.double().cpu()  # log_det the call implies
    close_vs_oracle((x, ld_equiv), sd, specs, z.cpu(), False, f"{name} sample")
    if name in FUSED:  # the table kernel took it: fused and generic draws are bitwise the same
        _, _, zg = prog.sample(n, dim, "cuda", seed, off, want_x=False, want_log_prob=False, want_z=True, kernel="generic")
        assert torch.equal(z, zg)
        xg, lpg, zg = prog.sample(n, dim, "cuda", seed, off, want_z=True, kernel="generic")
        assert torch.equal(z, zg)
        close_vs_oracle((xg, _log_normal64(zg) - lpg.double().cpu()), sd, specs, zg.cpu(), False, f"{name} generic")


@torch.no_grad()
def test_fused_call_is_one_launch_and_staged_equals_per_call_build():
    from torch_mnf import _lib

    specs, sd, model = _model("cfg2")
    prog = model._program()
    prog.sample(64, 2, "cuda", 1)  # stages the tables
    torch.cuda.synchronize()
    _lib.launch_stats(reset=True)
    x, lp, _ = prog.sample(1 << 16, 2, "cuda", 5)
    assert _lib.launch_stats(reset=True) == {"flow_pl_kernel": 1}
    xb, lpb, _ = prog.sample(1 << 16, 2, "cuda", 5, kernel=6)  # tables built into the workspace by this call
    assert _lib.launch_stats(reset=True) == {"flow_pl_build_kernel": 1, "flow_pl_kernel": 1}
    assert torch.equal(x, xb) and torch.equal(lp, lpb)
    _, sd4, m4 = _model("maf3_d8")
    m4._program().sample(1000, 8, "cuda", 5)
    stats = _lib.launch_stats(reset=True)
    assert sum(stats.values()) <= 3 and stats["flow_base_draw_kernel"] == 2, stats


@torch.no_grad()
def test_log_prob_of_samples_matches_log_prob():
    """log_prob(x) runs the inverse pass on the returned x: it agrees up to the inverse spline's fp32 error (the
    inverse solves a quadratic per bin; tests/test_flow_pl_spline_gpu.py bounds it against the oracle).  Measured on a B200:
    at most 1.4e-4 (config-2 stack, 2^16 draws), mean 4.4e-6."""
    for name in ("cfg2", "nsfcl3_stack", "rnvp9_moons", "affine_misc_d4"):
        _, _, model = _model(name)
        torch.manual_seed(3)
        x, lp = model.sample_and_log_prob(1 << 16)
        lp2 = model.log_prob(x)
        d = (lp - lp2).abs()
        print(f"{name}: max |log_prob(x) - sample lp| = {float(d.max()):.3e}, mean {float(d.mean()):.3e}")
        assert float(d.max()) <= 1e-3 and float(d.mean()) <= 2e-5


@pytest.mark.parametrize("name", ["cfg2", "maf3_d8"])
@torch.no_grad()
def test_shards_reproduce_the_single_call(name):
    _, _, model = _model(name)
    for n, cut in ((4097, 1001), (4097, 2048), (1 << 24, (1 << 23) + 1)):
        if n > 4097 and name != "cfg2":
            continue
        x, lp = model.sample_and_log_prob(n, seed=11)
        xa, lpa = model.sample_and_log_prob(cut, seed=11)
        xb, lpb = model.sample_and_log_prob(n - cut, seed=11, row_offset=cut)
        assert torch.equal(torch.cat([xa, xb]), x) and torch.equal(torch.cat([lpa, lpb]), lp), (n, cut)


@torch.no_grad()
def test_seeds_shapes_and_sample():
    _, _, model = _model("nsfcl3_stack")
    x, lp = model.sample_and_log_prob(3, 5, seed=9)
    assert x.shape == (3, 5, 2) and lp.shape == (3, 5)
    x2, lp2 = model.sample_and_log_prob((3, 5), seed=9)
    assert torch.equal(x, x2) and torch.equal(lp, lp2)
    assert torch.equal(model.sample(3, 5, seed=9), x)
    x3, _ = model.sample_and_log_prob(3, 5, seed=10)
    assert not torch.equal(x, x3)
    torch.manual_seed(4)
    a = model.sample_and_log_prob(64)[0]
    torch.manual_seed(4)
    assert torch.equal(model.sample_and_log_prob(64)[0], a)


def test_other_bases_pending_init_and_long_stacks():
    import torch_mnf.flows as nf
    from torch.distributions import MultivariateNormal

    specs, sd, model = _model("nsfcl3_stack")
    model.base = MultivariateNormal(torch.full((2,), 0.5), 2.0 * torch.eye(2))
    model.__dict__["_std_base"] = {}
    with pytest.raises(ValueError):
        model.sample_and_log_prob(8, seed=1)
    with torch.no_grad():
        x, lp = model.sample_and_log_prob(4096)
        torch.testing.assert_close(lp, model.log_prob(x), rtol=0, atol=2e-3)
    fresh = nf.NormalizingFlowModel(MultivariateNormal(torch.zeros(2), torch.eye(2)),
                                    [nf.ActNormFlow(2), nf.NSF_CL(2, K=8, B=3, n_h=8)]).cuda()
    with pytest.raises(RuntimeError, match="data-dependent"):
        fresh.sample_and_log_prob(8)
    long = nf.NormalizingFlowModel(MultivariateNormal(torch.zeros(2), torch.eye(2)),
                                   [nf.AffineConstantFlow(2) for _ in range(33)]).cuda()
    with pytest.raises(NotImplementedError):
        long.sample_and_log_prob(8)


@pytest.mark.parametrize("name", ["nsfcl3_stack", "maf_iaf_d2"])
@torch.enable_grad()
def test_gradients_match_oracle_autograd(name):
    """A loss on (x, log_prob) against torch autograd over the fp64 oracle on the same z."""
    specs, sd, model = _model(name)
    dim = specs[0]["dim"]
    B = 96
    x, lp = model.sample_and_log_prob(B, seed=21)
    with torch.no_grad():
        _, _, z = model._program().sample(B, dim, "cuda", 21, want_x=False, want_log_prob=False, want_z=True)
    gen = torch.Generator().manual_seed(7)
    w_x, w_lp = torch.randn(B, dim, generator=gen, dtype=torch.float64), torch.randn(B, generator=gen, dtype=torch.float64)
    ((x * w_x.cuda().float()).sum() + (lp * w_lp.cuda().float()).sum()).backward()

    sd64 = {k: (v.double().requires_grad_() if v.is_floating_point() and not k.endswith((".P", ".mask")) else v.double()
                if v.is_floating_point() else v) for k, v in sd.items()}
    z64 = z.double().cpu()
    outs, ld = _oracle_stack(sd64, specs, z64, False)
    lp64 = _log_normal64(z64) - ld
    ((outs[-1] * w_x).sum() + (lp64 * w_lp).sum()).backward()
    torch.testing.assert_close(x.detach().double().cpu(), outs[-1].detach(), rtol=1e-4, atol=1e-4)
    checked = 0
    for k, p in model.named_parameters():
        ref = sd64[k].grad
        if ref is None:
            continue
        assert p.grad is not None, f"no gradient reached {k}"
        scale = float(ref.abs().max()) + 1e-6
        err = float((p.grad.reshape(ref.shape).double().cpu() - ref).abs().max())
        assert err <= 3e-4 * scale, f"{name} {k}: max err {err:.3e} vs scale {scale:.3e}"
        checked += 1
    assert checked > 0


@pytest.mark.parametrize("kind", ["affine", "nsf"])
@torch.enable_grad()
def test_reverse_kl_fit_of_a_correlated_gaussian(kind):
    """Adam on the reverse KL (log q(x) - log p(x)).mean(), whose minimum is 0.  Measured on a B200 (mean of the last 20
    of 400 steps): 0.0008 for the AffineHalfFlow stack, 0.0029 for the NSF_CL stack, from 2.8 and 6.2."""
    import torch_mnf.flows as nf
    from torch.distributions import MultivariateNormal

    torch.manual_seed(0)
    if kind == "affine":
        flows = [nf.AffineHalfFlow(2, i % 2, h_sizes=(16, 16), scale=True, shift=True) for i in range(4)]
    else:
        flows = [nf.NSF_CL(2, K=8, B=6, n_h=16) for _ in range(2)]
    model = nf.NormalizingFlowModel(MultivariateNormal(torch.zeros(2), torch.eye(2)), flows).cuda()
    cov = torch.tensor([[1.0, 0.8], [0.8, 1.0]], device="cuda")
    target = MultivariateNormal(torch.tensor([1.0, -0.5], device="cuda"), 2.0 * cov)
    opt = torch.optim.Adam(model.parameters(), lr=5e-3)
    hist = []
    for step in range(400):
        x, lp = model.sample_and_log_prob(4096, seed=step)
        loss = (lp - target.log_prob(x)).mean()
        opt.zero_grad()
        loss.backward()
        opt.step()
        hist.append(float(loss.detach()))
    final = sum(hist[-20:]) / 20
    print(f"reverse KL {kind}: first {hist[0]:.4f}, final (mean of last 20) {final:.4f}")
    assert final < 0.02 and final < 0.2 * hist[0]


@torch.no_grad()
def test_cuda_graph_replays_draw_anew():
    _, _, model = _model("cfg2")
    model.sample_and_log_prob(1024)  # builds the program and the staged tables outside the capture
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        model.sample_and_log_prob(1024)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        x, lp = model.sample_and_log_prob(1024)
    g.replay()
    a, la = x.clone(), lp.clone()
    g.replay()
    assert not torch.equal(a, x) and not torch.equal(la, lp)
    ref = model.log_prob(x)
    assert float((ref - lp).abs().max()) < 2e-3
