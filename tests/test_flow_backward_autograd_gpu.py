"""mnf_flow_stack_backward (csrc/flow_backward.cu) against torch autograd over the fp64 CPU oracle beyond the golden
stacks: batches of one row up to more than two waves of blocks in each of the kernel's three ways of accumulating the
parameter gradients, spline inputs on the tail bounds and on the knots, saturated spline parameters, the kernel's shape
limits and every form of the loss autograd can hand it.

Each case checks the forward outputs and log-det, d/dx of every row and every parameter gradient that reaches the
model, and asserts the launch regime it claims to cover, so that a retuned launch policy shows which regime lost its
coverage.  Large batches weight the loss with non-negative weights: with signed weights the per-row terms of a
parameter gradient cancel, and at 150k rows the fp32 oracle itself then misses fp64 by more than the tolerance."""

import math

import pytest
import torch

from tests.helpers import load_flow_model, oracle_stack, random_flow_sd

pytestmark = pytest.mark.gpu

TOL = 3e-4  # per tensor, relative to max|reference| (as tests/test_flow_autograd_gpu.py)
SIGNED_MAX_ROWS = 4096  # larger batches take non-negative loss weights (module docstring)


# ---------------------------------------------------------------------------
# launch policy
# ---------------------------------------------------------------------------
def _launch(n_params, sm_count):
    """The launch policy of mnf_flow_stack_backward (csrc/flow_backward.cu:600-610): a blob of up to 12288 floats
    (48 KB) is summed per block in shared memory, up to 24576 floats (96 KB) in opt-in shared memory, a larger one with
    warp-reduced global atomics straight into the gradient blob; blocks of 128 rows, at most sm_count * per_sm of them,
    and a grid-stride loop over the rows beyond.  -> (band, rows per wave)."""
    if n_params <= 12288:
        band = "smem"
    elif n_params <= 24576:
        band = "smem_optin"
    else:
        band = "global"
    per_sm = 8 if band == "global" else min(max(204800 // (4 * n_params), 1), 8)
    return band, sm_count * per_sm * 128


def _regime(model, dim):
    """(band, rows per wave, blob size) of the backward launch of `model` (its packed blob is built by plan())."""
    prog = model._program()
    prog.plan("cuda", dim)
    n_params = prog._blob.numel()
    band, rows_per_wave = _launch(n_params, torch.cuda.get_device_properties(0).multi_processor_count)
    return band, rows_per_wave, n_params


def _assert_regime(model, dim, n_rows, band, min_blocks=2):
    got, rows_per_wave, n_params = _regime(model, dim)
    assert got == band, f"blob of {n_params} floats takes the {got} path, this case covers {band}"
    blocks = min(-(-n_rows // 128), rows_per_wave // 128)
    assert blocks >= min_blocks, f"{n_rows} rows launch {blocks} blocks, this case needs {min_blocks}"
    return rows_per_wave


# ---------------------------------------------------------------------------
# stacks
# ---------------------------------------------------------------------------
def _an(d):
    return {"type": "ActNormFlow", "dim": d, "scale": True, "shift": True}


def _cl(d, K, B, n_h):
    return {"type": "NSF_CL", "dim": d, "K": K, "B": B, "n_h": n_h}


def _ar(d, K, B, n_h):
    return {"type": "NSF_AR", "dim": d, "K": K, "B": B, "n_h": n_h}


def _ah(d, parity, h, scale=True, shift=True):
    return {"type": "AffineHalfFlow", "dim": d, "parity": parity, "h_sizes": list(h), "scale": scale, "shift": shift}


def _made(kind, d, parity, h):
    return {"type": kind, "dim": d, "parity": parity, "h_sizes": list(h)}


def _glow(d):
    return {"type": "Glow", "dim": d}


BAND_STACKS = {  # one dim-2 stack per gradient-accumulation band (blob sizes 7760, 20592, 29972 floats)
    "smem": [_an(2), _cl(2, 8, 3, 16)] * 4,
    "smem_optin": [_cl(2, 8, 3, 32), _ah(2, False, (32,) * 3), _cl(2, 8, 3, 32), _ah(2, True, (32,) * 3)],
    "global": [_an(2), _cl(2, 8, 3, 80)],
}


# ---------------------------------------------------------------------------
# one case: fp64 oracle + autograd against the CUDA backward
# ---------------------------------------------------------------------------
def _weights(n, d, n_flows, signed, seed=7):
    gen = torch.Generator().manual_seed(seed)
    w_ld = torch.randn(n, generator=gen, dtype=torch.float64)
    w_out = [torch.randn(n, d, generator=gen, dtype=torch.float64) for _ in range(n_flows)]
    if not signed:
        w_ld, w_out = w_ld.abs(), [w.abs() for w in w_out]
    return w_ld, w_out


def _loss_weights(w_ld, w_out, loss):
    """The weights that enter the loss: "all" = log-det and every flow's output, "final" = log-det and the final
    output, "ld" = the log-det alone, "out" = the final output alone."""
    if loss in ("final", "out"):
        w_out = [torch.zeros_like(w) for w in w_out[:-1]] + [w_out[-1]]
    if loss == "ld":
        w_out = [torch.zeros_like(w) for w in w_out]
    if loss == "out":
        w_ld = torch.zeros_like(w_ld)
    return w_ld, w_out


def _reference(specs, sd, x, inverse, w_ld, w_out, frozen=(), dtype=torch.float64):
    sd64 = {}
    for k, v in sd.items():
        if not v.is_floating_point():
            sd64[k] = v
            continue
        trainable = not k.endswith((".P", ".mask")) and int(k.split(".")[1]) not in frozen
        sd64[k] = v.detach().to(dtype).requires_grad_(trainable)
    x64 = x.detach().to(dtype).requires_grad_()
    outs, ld = oracle_stack(sd64, specs, x64, inverse)
    loss = (ld * w_ld.to(dtype)).sum()
    for o, w in zip(outs[1:], w_out):
        loss = loss + (o * w.to(dtype)).sum()
    loss.backward()
    return {"outs": [o.detach() for o in outs[1:]], "ld": ld.detach(), "gx": x64.grad,
            "grads": {k: v.grad for k, v in sd64.items() if isinstance(v, torch.Tensor) and v.grad is not None}}


def _cuda(specs, sd, x, inverse, w_ld, w_out, loss, frozen=(), x_grad=True, model=None):
    if model is None:
        model = load_flow_model(specs, sd, return_intermediates=loss == "all")
        for i in frozen:
            model.flows[i].requires_grad_(False)
    xg = x.cuda()
    if x_grad:
        xg.requires_grad_()
    outs_g, ld_g = model.inverse(xg) if inverse else model.forward(xg)
    total = torch.zeros((), device="cuda")
    if loss != "out":
        total = total + (ld_g * w_ld.cuda().float()).sum()
    if loss == "all":
        for o, w in zip(outs_g[1:], w_out):
            total = total + (o * w.cuda().float()).sum()
    elif loss in ("final", "out"):
        total = total + (outs_g[-1] * w_out[-1].cuda().float()).sum()
    total.backward()
    return model, outs_g, ld_g, xg


def _near_knot_rows(specs, sd, x, inverse, rel=1e-5):
    """Rows whose input to an NSF_CL spline lies within rel * B of an interior knot of its bin search (fp64 oracle).
    The spline is C1 only: the log-det's derivatives jump at a knot, and fp32 and fp64 may pick different sides, so
    such rows leave the log-det out of the loss (a large batch has a few)."""
    from oracle import flows_cpu

    sd64 = {k: v.double() if v.is_floating_point() else v for k, v in sd.items()}
    near = torch.zeros(x.shape[0], dtype=torch.bool)
    with torch.no_grad():
        outs, _ = oracle_stack(sd64, specs, x.double(), inverse)
    order = list(range(len(specs)))[::-1] if inverse else list(range(len(specs)))
    for step, i in enumerate(order):
        spec = specs[i]
        if spec["type"] != "NSF_CL":
            continue
        K, B, h = spec["K"], spec["B"], spec["dim"] // 2
        p = flows_cpu.sub(sd64, f"flows.{i}.")
        v = outs[step].clone()
        # forward: f1(lower) bins upper by width knots, then f2(upper') bins lower; inverse: f2(upper) bins lower by
        # height knots, then f1(lower') bins upper (spline_flow.py:249-285)
        halves = (("f1.", 0, 1), ("f2.", 1, 0)) if not inverse else (("f2.", 1, 0), ("f1.", 0, 1))
        for net, cond, tgt in halves:
            raw = flows_cpu.mlp(flows_cpu.sub(p, net), v[:, cond * h:(cond + 1) * h]).reshape(-1, h, 3 * K - 1)
            W, H, D = flows_cpu._spline_params(raw, K, B)
            knots = flows_cpu._knots(H if inverse else W, -B, B, flows_cpu.MIN_W)[0][..., 1:-1]
            t = v[:, tgt * h:(tgt + 1) * h]
            near |= ((knots - t[..., None]).abs() < rel * B).any(-1).any(-1)
            out, _ = flows_cpu.unconstrained_rqs(t, W, H, D, inverse, B)
            v[:, tgt * h:(tgt + 1) * h] = out
    return near


def _close(ours, ref, what, ref32):
    """|ours - ref| <= TOL * max|ref| per tensor plus, element by element, eight times the fp32 oracle's own error
    |ref32 - ref|: the kernel and the oracle round differently, and on the few ill-conditioned rows of a 348k-row batch
    (steep spline bins) the kernel's error exceeded four times the oracle's."""
    ref = ref.double()
    err = (ours.detach().cpu().double().reshape(ref.shape) - ref).abs()
    bound = TOL * (float(ref.abs().max()) + 1e-6) if ref.numel() else 0.0
    err = err - 8.0 * (ref32.double().reshape(ref.shape) - ref).abs()
    worst = float(err.max()) if ref.numel() else 0.0
    assert worst <= bound, f"{what}: max err {worst:.3e} over the bound {bound:.3e}"


def _check(specs, sd, x, inverse, loss="all", frozen=(), x_grad=True, signed=None, w_ld_mask=None, model=None):
    """Runs one case on the GPU and the oracle and compares everything; returns (model, CUDA d/dx, weights).
    w_ld_mask zeroes the log-det weight of chosen rows.  The bounds admit the fp32 oracle's own error (_close): at
    large batches some rows meet steep spline bins where fp32 itself is ill-conditioned."""
    n, d = x.shape
    signed = n <= SIGNED_MAX_ROWS if signed is None else signed
    w_ld, w_out = _loss_weights(*_weights(n, d, len(specs), signed), loss)
    if w_ld_mask is not None:
        w_ld = w_ld * w_ld_mask
    w_ld = torch.where(_near_knot_rows(specs, sd, x, inverse), 0.0, w_ld)
    ref = _reference(specs, sd, x, inverse, w_ld, w_out, frozen)
    r32 = _reference(specs, sd, x, inverse, w_ld, w_out, frozen, torch.float32)
    model, outs_g, ld_g, xg = _cuda(specs, sd, x, inverse, w_ld, w_out, loss, frozen, x_grad, model)

    _close(ld_g, ref["ld"], "log-det", r32["ld"])
    outs_ref = ref["outs"] if loss == "all" else ref["outs"][-1:]
    outs_32 = r32["outs"] if loss == "all" else r32["outs"][-1:]
    for k, (o, r, r_32) in enumerate(zip(outs_g[1:], outs_ref, outs_32)):
        _close(o, r, f"output {k}", r_32)
    if x_grad:
        _close(xg.grad, ref["gx"], "d/dx", r32["gx"])
    else:
        assert xg.grad is None
    checked = 0
    for k, p in model.named_parameters():
        if int(k.split(".")[1]) in frozen:
            assert p.grad is None, f"frozen {k} received a gradient"
            continue
        r = ref["grads"].get(k)
        if r is None:
            continue
        assert p.grad is not None, f"no gradient reached {k}"
        _close(p.grad, r, k, r32["grads"][k])
        checked += 1
    assert checked > 0
    return model, (xg.grad if x_grad else None), (w_ld, w_out)


def _inputs(n, d, seed=1, scale=1.0):
    return scale * torch.randn(n, d, generator=torch.Generator().manual_seed(seed))


# ---------------------------------------------------------------------------
# 1. batch regimes
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("band", list(BAND_STACKS))
@pytest.mark.parametrize("n_rows", [1, 31, 33, 129])
@pytest.mark.parametrize("direction", ["inv", "fwd"])
@pytest.mark.parametrize("loss", ["all", "final"])
def test_partial_blocks(band, n_rows, direction, loss):
    """Warps that mix valid rows with padding lanes (which must add nothing), and at 129 rows a second block holding
    one valid row."""
    specs = BAND_STACKS[band]
    sd = random_flow_sd(specs, seed=3, scale=0.4)
    model = load_flow_model(specs, sd, return_intermediates=loss == "all")
    _assert_regime(model, 2, n_rows, band, min_blocks=2 if n_rows > 128 else 1)
    _check(specs, sd, _inputs(n_rows, 2), direction == "inv", loss, model=model)


@pytest.mark.parametrize("band", list(BAND_STACKS))
@pytest.mark.parametrize("waves,direction,loss", [(1, "inv", "all"), (2.3, "fwd", "final"), (2.3, "inv", "all")])
def test_waves(band, waves, direction, loss):
    """A full wave plus a ragged tail, and more than two waves plus a ragged tail: the grid-stride loop, the per-block
    flush (or the global atomics) of every block.  d/dx needs no atomics, so a window of rows taken from the big call
    is bitwise equal to a one-block call on just those rows."""
    specs = BAND_STACKS[band]
    sd = random_flow_sd(specs, seed=4, scale=0.4)
    model = load_flow_model(specs, sd, return_intermediates=loss == "all")
    rows_per_wave = _regime(model, 2)[1]
    n_rows = int(waves * rows_per_wave) // 128 * 128 + 77  # a block of 77 valid rows last
    _assert_regime(model, 2, n_rows, band)
    assert n_rows > math.floor(waves) * rows_per_wave
    x = _inputs(n_rows, 2, seed=5)
    inverse = direction == "inv"
    model, gx, (w_ld, w_out) = _check(specs, sd, x, inverse, loss, model=model)

    for lo in (rows_per_wave - 64, n_rows - 128):  # across the first wave boundary; the ragged end
        sl = slice(lo, lo + 128)
        win = load_flow_model(specs, sd, return_intermediates=loss == "all")
        _, _, _, xw = _cuda(specs, sd, x[sl], inverse, w_ld[sl], [w[sl] for w in w_out], loss, model=win)
        assert torch.equal(xw.grad, gx[sl]), f"d/dx of rows {lo}.. depends on the batch around them"


# ---------------------------------------------------------------------------
# 2. spline edges
# ---------------------------------------------------------------------------
DERIV_RAW = (25.0, 19.9, -25.0, -40.0)  # above the softplus threshold 20, just below it, saturated low


def _set_spline_raw(sd, spec, prefix, deriv_off, saturate):
    """Raw knot derivatives cycling through DERIV_RAW (starting at deriv_off) and, with saturate, the first raw width
    at 30 (the other bins at the minimum width where 2B is large): on the last conditioner bias, the matching weight
    rows shrunk so that the raw values stay at these levels, and on NSF_AR's constant init_param.  Heights stay
    unsaturated: the inverse spline through a bin of minimum height is ill-conditioned in fp32 itself."""
    K = spec["K"]
    nb = 3 * K - 1

    def fill(raw):
        for i in range(K - 1):
            raw[2 * K + i] = DERIV_RAW[(i + deriv_off) % len(DERIV_RAW)]
        if saturate:
            raw[0] = 30.0

    if spec["type"] == "NSF_AR":
        fill(sd[prefix + "init_param"])
        nets = [f"{prefix}layers.{i}." for i in range(spec["dim"] - 1)]
    else:
        nets = [prefix + "f1.", prefix + "f2."]
    for net in nets:
        last = max(int(k[len(net):].split(".")[0]) for k in sd if k.startswith(net))
        b, w = sd[f"{net}{last}.bias"], sd[f"{net}{last}.weight"]
        for j in range(b.numel() // nb):
            fill(b[j * nb:(j + 1) * nb])
            w[j * nb + 2 * K:(j + 1) * nb] *= 0.01
            if saturate:
                w[j * nb] *= 0.01


def _edge_inputs(n, d, B, seed):
    """Rows alternate between inside [-B, B] and the identity tails (per column, so every warp has lanes of both);
    every 8th row carries -B, B and the neighbouring floats inside and outside the bound."""
    gen = torch.Generator().manual_seed(seed)
    u = torch.rand(n, d, generator=gen)
    sign = torch.where(torch.rand(n, d, generator=gen) < 0.5, -1.0, 1.0)
    tail = (torch.arange(n)[:, None] + torch.arange(d)[None, :]) % 2 == 1
    x = torch.where(tail, sign * B * (1.0 + 0.5 * u + 1e-3), B * (2 * u - 1))
    b = torch.tensor(B, dtype=torch.float32)
    special = torch.stack([-b, b, torch.nextafter(-b, -2 * b), torch.nextafter(-b, b),
                           torch.nextafter(b, -b), torch.nextafter(b, 2 * b)])
    for m, r in enumerate(range(0, n, 8)):
        x[r, m % d] = special[m % len(special)]
    return x


SPLINE_CASES = [  # (K, B, first raw derivative of DERIV_RAW, saturated width/height)
    (2, 0.5, 0, False),
    (2, 8.0, 3, False),
    (32, 0.5, 1, True),
    (32, 8.0, 2, False),
    (8, 3.0, 0, True),
]


@pytest.mark.parametrize("kind", ["NSF_CL", "NSF_AR"])
@pytest.mark.parametrize("K,B,deriv_off,saturate", SPLINE_CASES)
@pytest.mark.parametrize("direction", ["inv", "fwd"])
def test_spline_edges(kind, K, B, deriv_off, saturate, direction):
    """Divergent tails inside every warp, inputs on +-B and one float either side, raw knot derivatives on both sides
    of the softplus threshold, saturated bins, K = 2 and 32.  NSF_AR's column 0 (constant spline parameters) also
    sits on each interior knot of the bin search and one float either side: there the log-det's derivatives jump
    (the spline is C1 only), and fp32 and fp64 may pick different sides, so those rows leave the log-det out of the
    loss; outputs and their gradients are continuous across a knot."""
    inverse = direction == "inv"
    dim = 2 if kind == "NSF_CL" else 3
    spec = (_cl if kind == "NSF_CL" else _ar)(dim, K, B, 16)
    specs = [spec]
    sd = random_flow_sd(specs, seed=11 + K, scale=0.4)
    _set_spline_raw(sd, spec, "flows.0.", deriv_off, saturate)
    n = 4096
    x = _edge_inputs(n, dim, B, seed=K)
    w_ld_mask = None
    if kind == "NSF_AR":
        from oracle import flows_cpu

        # NSF_AR.inverse runs the spline forward (bins by width knots), NSF_AR.forward the spline inverse (height knots)
        W, H, _ = flows_cpu._spline_params(sd["flows.0.init_param"].float(), K, B)
        knots = flows_cpu._knots(W if inverse else H, -B, B, flows_cpu.MIN_W)[0][1:-1]
        on = torch.stack([torch.nextafter(knots, knots - 1), knots, torch.nextafter(knots, knots + 1)], 1).reshape(-1)
        rows = torch.arange(on.numel()) * 8 + 4
        x[rows, 0] = on
        w_ld_mask = torch.ones(n, dtype=torch.float64)
        w_ld_mask[rows] = 0.0
    model = load_flow_model(specs, sd)
    _assert_regime(model, dim, n, "smem")
    _check(specs, sd, x, inverse, "all", w_ld_mask=w_ld_mask, model=model)


# ---------------------------------------------------------------------------
# 3. shape limits
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("kind,direction", [("MAF", "inv"), ("MAF", "fwd"), ("IAF", "fwd"), ("IAF", "inv")])
def test_made_dim64(kind, direction):
    """Dim 64 with both parities: the one-pass adjoint at hidden width 128 (MAF.inverse, IAF.forward) and the D-pass
    sequential adjoint (MAF.forward, IAF.inverse) at width 64, whose fp64 reference takes D MADE passes on the CPU."""
    inverse = direction == "inv"
    sequential = (kind == "MAF") != inverse
    h, n = ((64, 64), 1024) if sequential else ((128,) * 3, 2048)
    specs = [_made(kind, 64, False, h), _made(kind, 64, True, h)]
    sd = random_flow_sd(specs, seed=21, scale=0.3)
    model = load_flow_model(specs, sd)
    _assert_regime(model, 64, n, "global")
    _check(specs, sd, _inputs(n, 64, seed=22), inverse, "all", model=model)


@pytest.mark.parametrize("direction", ["inv", "fwd"])
def test_glow_affine_half_dim64(direction):
    """Dim 64 through ActNorm, Glow and AffineHalfFlow with hidden width 128 and ragged widths (5, 17, 31)."""
    specs = [_an(64), _glow(64), _ah(64, False, (128,)), _ah(64, True, (5, 17, 31))]
    sd = random_flow_sd(specs, seed=23, scale=0.3)
    model = load_flow_model(specs, sd)
    _assert_regime(model, 64, 1024, "global")
    _check(specs, sd, _inputs(1024, 64, seed=24), direction == "inv", "all", model=model)


@pytest.mark.parametrize("direction", ["inv", "fwd"])
def test_affine_half_depths_and_halves(direction):
    """AffineHalfFlow with one Linear layer (h_sizes=()), with six (MNF_MAX_LIN), shift only (NICE) and scale only."""
    specs = [_ah(8, False, ()), _ah(8, True, (16,) * 5), _ah(8, False, (5, 17, 31), scale=False),
             _ah(8, True, (24,), shift=False)]
    sd = random_flow_sd(specs, seed=25, scale=0.4)
    model = load_flow_model(specs, sd)
    _assert_regime(model, 8, 3000, "smem")
    _check(specs, sd, _inputs(3000, 8, seed=26), direction == "inv", "all", model=model)


@pytest.mark.parametrize("direction", ["inv", "fwd"])
def test_nsf_cl_widest_conditioner(direction):
    """NSF_CL dim 64, K 11: the conditioner has exactly kMaxNetOut = 32 * 32 = 1024 outputs."""
    specs = [_cl(64, 11, 3, 8)]
    sd = random_flow_sd(specs, seed=27, scale=0.4)
    model = load_flow_model(specs, sd)
    _assert_regime(model, 64, 512, "smem_optin")
    _check(specs, sd, _inputs(512, 64, seed=28, scale=2.0), direction == "inv", "all", model=model)


def test_nsf_cl_too_wide_conditioner_is_rejected():
    """K 12 gives 32 * 35 = 1120 conditioner outputs: the forward runs, backward() raises before any launch."""
    from torch_mnf import _lib

    specs = [_cl(64, 12, 3, 8)]
    model = load_flow_model(specs, random_flow_sd(specs, seed=29, scale=0.4))
    x = _inputs(256, 64, seed=30).cuda().requires_grad_()
    zs, ld = model.inverse(x)
    torch.cuda.synchronize()
    before = _lib.lib().mnf_launch_count()
    with pytest.raises(RuntimeError, match="wider than 1024"):
        (ld.sum() + zs[-1].sum()).backward()
    assert _lib.lib().mnf_launch_count() == before
    torch.cuda.synchronize()


@pytest.mark.parametrize("direction", ["inv", "fwd"])
def test_nsf_ar_dim1(direction):
    """NSF_AR with one dimension: no conditioner net, only the constant spline parameters."""
    specs = [_an(1), _ar(1, 8, 3, 8)]
    sd = random_flow_sd(specs, seed=31, scale=0.4)
    model = load_flow_model(specs, sd)
    _assert_regime(model, 1, 1000, "smem")
    _check(specs, sd, _inputs(1000, 1, seed=32, scale=2.0), direction == "inv", "all", model=model)


@pytest.mark.parametrize("direction", ["inv", "fwd"])
def test_32_flows(direction):
    """MNF_MAX_OPS flows in one program, every intermediate in the loss."""
    specs = [_an(2), _glow(2), _cl(2, 4, 3, 8), _ah(2, True, (8,))] * 8
    assert len(specs) == 32
    sd = random_flow_sd(specs, seed=33, scale=0.3)
    model = load_flow_model(specs, sd)
    _assert_regime(model, 2, 5000, "smem")
    _check(specs, sd, _inputs(5000, 2, seed=34), direction == "inv", "all", model=model)


def test_33_flows_rejected():
    specs = [_an(2), _cl(2, 4, 3, 8), _ah(2, True, (8,))] * 11
    assert len(specs) == 33
    model = load_flow_model(specs, random_flow_sd(specs, seed=35, scale=0.3))
    x = _inputs(64, 2).cuda().requires_grad_()
    with pytest.raises(NotImplementedError):
        model._program().run_autograd(x, inverse=True)


# ---------------------------------------------------------------------------
# 4. loss and requires_grad forms
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("form", ["ld", "out", "no_x_grad", "frozen"])
@pytest.mark.parametrize("direction", ["inv", "fwd"])
def test_loss_forms(form, direction):
    """A loss of the log-det alone (autograd hands the backward an all-zero output gradient), of the final output
    alone (an all-zero log-det gradient), an input without requires_grad (no d/dx is written) and one frozen flow."""
    specs = BAND_STACKS["smem"]
    sd = random_flow_sd(specs, seed=36, scale=0.4)
    loss = form if form in ("ld", "out") else "all"
    frozen = (3,) if form == "frozen" else ()
    model = load_flow_model(specs, sd, return_intermediates=loss == "all")
    for i in frozen:
        model.flows[i].requires_grad_(False)
    _assert_regime(model, 2, 5000, "smem")
    _check(specs, sd, _inputs(5000, 2, seed=37), direction == "inv", loss, frozen=frozen,
           x_grad=form != "no_x_grad", model=model)
