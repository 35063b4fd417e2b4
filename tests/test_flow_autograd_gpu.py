"""Gradients of the flow hot path: mnf_flow_stack_backward (through the drop-in modules' autograd path) against
torch autograd over the fp64 CPU oracle on the golden stacks.  The reference has no backward of its own -- it trains
through torch autograd (tests/test_flows.py:14-31) -- so the oracle + autograd IS the reference gradient."""

import pytest
import torch

from tests.helpers import golden_sd, golden_spec, load_flow_model, load_golden, oracle_stack, t

pytestmark = pytest.mark.gpu

CASES = [  # (fixture, directions)
    ("rnvp9_moons", ("inv", "fwd")),
    ("nsfcl3_stack", ("inv", "fwd")),
    ("nsfcl_d4", ("inv", "fwd")),
    ("nsfar2_d3", ("inv", "fwd")),
    ("maf3_d8", ("inv", "fwd")),
    ("maf_iaf_d2", ("inv", "fwd")),
    ("affine_misc_d4", ("inv", "fwd")),
]


def _loss(outs, ld, weights):
    w_ld, w_out = weights
    loss = (ld * w_ld.to(ld)).sum()
    for o, w in zip(outs[1:], w_out):
        loss = loss + (o * w.to(o)).sum()
    return loss


@pytest.mark.parametrize("name,direction", [(n, d) for n, ds in CASES for d in ds])
@pytest.mark.parametrize("use_intermediates", [True, False])
def test_gradients_match_oracle_autograd(name, direction, use_intermediates):
    g = load_golden(name)
    specs, sd = golden_spec(g), golden_sd(g)
    inverse = direction == "inv"
    x = t(g, "inv/x" if inverse else "fwd/z")[:96]
    B, D = x.shape
    gen = torch.Generator().manual_seed(7)
    w_ld = torch.randn(B, generator=gen, dtype=torch.float64)
    w_out = [torch.randn(B, D, generator=gen, dtype=torch.float64) for _ in specs]
    if not use_intermediates:  # only the final output and the log-det enter the loss
        w_out = [torch.zeros_like(w) for w in w_out[:-1]] + [w_out[-1]]

    # reference gradient: fp64 oracle + torch autograd
    sd64 = {k: (v.double().requires_grad_() if v.is_floating_point() and not k.endswith((".P", ".mask")) else v.double()
                if v.is_floating_point() else v) for k, v in sd.items()}
    x64 = x.double().requires_grad_()
    outs, ld = oracle_stack(sd64, specs, x64, inverse)
    _loss(outs, ld, (w_ld, w_out)).backward()

    model = load_flow_model(specs, sd, return_intermediates=use_intermediates)
    xg = x.cuda().requires_grad_()
    outs_g, ld_g = model.inverse(xg) if inverse else model.forward(xg)
    if use_intermediates:
        loss = _loss(outs_g, ld_g, (w_ld.cuda(), [w.cuda() for w in w_out]))
    else:
        loss = (ld_g * w_ld.cuda().float()).sum() + (outs_g[-1] * w_out[-1].cuda().float()).sum()
    loss.backward()

    def close(ours, ref, what):
        ref = ref.float()
        scale = float(ref.abs().max()) + 1e-6
        err = float((ours.cpu() - ref).abs().max())
        assert err <= 3e-4 * scale, f"{name}/{direction} {what}: max err {err:.3e} vs scale {scale:.3e}"

    close(xg.grad, x64.grad, "d/dx")
    checked = 0
    for k, p in model.named_parameters():
        ref = sd64[k].grad
        if ref is None:
            continue
        assert p.grad is not None, f"no gradient reached {k}"
        close(p.grad.reshape(ref.shape), ref, k)
        checked += 1
    assert checked > 0


def test_single_flow_module_backward():
    """Flow.inverse / Flow.forward on a lone module also build the graph."""
    import torch_mnf.flows as nf

    torch.manual_seed(0)
    flow = nf.NSF_CL(dim=2, K=8, B=3, n_h=16).cuda()
    x = torch.randn(64, 2, device="cuda")
    z, ld = flow.inverse(x)
    (ld.sum() + z.square().sum()).backward()
    grads = [p.grad for p in flow.parameters()]
    assert all(g is not None and torch.isfinite(g).all() for g in grads)
    assert any(float(g.abs().max()) > 0 for g in grads)


def test_no_grad_keeps_inference_path():
    import torch_mnf.flows as nf
    from torch_mnf import _lib

    flow = nf.NormalizingFlow([nf.NSF_CL(dim=2, K=8, B=3, n_h=16) for _ in range(2)]).cuda()
    x = torch.randn(64, 2, device="cuda")
    with torch.no_grad():
        zs, ld = flow.inverse(x)
    assert not ld.requires_grad and not zs[-1].requires_grad
    zs, ld = flow.inverse(x)
    assert ld.requires_grad and zs[-1].requires_grad
    assert _lib.lib().mnf_launch_count() > 0
