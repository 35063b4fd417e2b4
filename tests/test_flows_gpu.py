"""GPU parity: CUDA flow kernels (through the C ABI, via the drop-in modules) vs the golden
vectors recorded from the reference and vs the CPU oracle on larger seeded inputs.

Tolerance (BASELINE.json north_star): rtol 1e-5 for fp32 flow outputs and log-dets; an
absolute floor of 1e-5 x (typical magnitude) covers values near zero (log-dets of ~0 at
the spline tails)."""

import pytest
import torch

from oracle import flows_cpu
from tests.helpers import golden_sd, golden_spec, load_flow_model, load_golden, random_flow_sd, t

pytestmark = pytest.mark.gpu

RTOL = 1e-5


def close(a, b, what, rtol=RTOL, atol_scale=1e-5):
    """Direct comparison with recorded reference outputs: rtol 1e-5 plus an absolute floor of
    atol_scale x (mean magnitude).  Log-dets use 4e-5: the reference's own fp32 log-det on the
    spline fixtures is only good to 2.1e-5 (|oracle32 - oracle64|, tests/measure/flow_error_stats.py)."""
    a = a.detach().float().cpu()
    scale = max(1.0, float(b.abs().mean()))
    torch.testing.assert_close(a, b, rtol=rtol, atol=atol_scale * scale, msg=lambda m: f"{what}: {m}")


def _q999(e):
    e = e.flatten()
    return float(e.kthvalue(max(1, int(0.999 * e.numel()))).values)


def close_vs_oracle(a, sd, specs, x, inverse, what):
    """Parity against the oracle at the precision the reference itself has.

    The reference evaluates in fp32; on these stacks its own outputs differ from an exact (fp64)
    evaluation of the same formulas by 1e-5 .. 1e-4 (measured: tests/measure/flow_error_stats.py), so a
    bare rtol of 1e-5 against fp32 outputs is below the reference's noise floor.  The test
    therefore asks three things of the CUDA result `got`, with r32 / r64 the oracle in fp32 / fp64:
      (1) elementwise |got - r32| <= 1e-5*|r64| + 1e-5*scale + 4*|r32 - r64|  for >= 99.9% of elements
          (rtol 1e-5 wherever the reference itself is that accurate),
      (2) max  |got - r64| <= 2 * max  |r32 - r64| + 1e-5*scale   (as exact as the reference, worst case)
      (3) p99.9|got - r64| <= 2 * p99.9|r32 - r64| + 1e-5*scale   (and in distribution)."""
    ref32, ld32 = flows_cpu.stack(sd, specs, x, inverse=inverse)
    sd64 = {k: (v.double() if v.is_floating_point() else v) for k, v in sd.items()}
    ref64, ld64 = flows_cpu.stack(sd64, specs, x.double(), inverse=inverse)
    for got, r32, r64, name in ((a[0], ref32[-1], ref64[-1], "out"), (a[1], ld32, ld64, "log_det")):
        got = got.detach().cpu().double()
        scale = max(1.0, float(r64.abs().mean()))
        floor = 1e-5 * scale
        ref_err = (r32.double() - r64).abs()
        err32, err64 = (got - r32.double()).abs(), (got - r64).abs()
        n_bad = int((err32 > RTOL * r64.abs() + floor + 4.0 * ref_err).sum())
        assert n_bad <= max(1, got.numel() // 1000), (
            f"{what} {name}: {n_bad} of {got.numel()} elements outside rtol 1e-5 of the oracle")
        assert float(err64.max()) <= 2.0 * float(ref_err.max()) + floor, (
            f"{what} {name}: max error vs exact {float(err64.max()):.3e}, reference's own {float(ref_err.max()):.3e}")
        if got.numel() >= 2000:
            assert _q999(err64) <= 2.0 * _q999(ref_err) + floor, (
                f"{what} {name}: p99.9 error vs exact {_q999(err64):.3e}, reference's own {_q999(ref_err):.3e}")


FLOW_CASES = ["rnvp9_moons", "nsfcl3_stack", "nsfcl_d4", "nsfar2_d3", "maf9_d64", "maf3_d8", "maf_iaf_d2",
              "affine_misc_d4"]


@pytest.mark.parametrize("name", FLOW_CASES)
@pytest.mark.parametrize("kernel", [None, "generic"])
def test_stack_vs_golden(name, kernel):
    g = load_golden(name)
    sd, specs = golden_sd(g), golden_spec(g)
    model = load_flow_model(specs, sd)
    prog = model._program()
    x = t(g, "inv/x").cuda()
    y, ld, inter, lp = prog.run(x, inverse=True, want_inter=True, want_base_lp=True, kernel=kernel)
    close(y, t(g, "inv/z"), "z", atol_scale=2e-5)
    close(ld, t(g, "inv/ld"), "log_det", atol_scale=4e-5)
    close_vs_oracle((y, ld), sd, specs, t(g, "inv/x"), True, name)
    n = len(specs) + 1
    mid = n // 2
    close(inter[mid - 1], t(g, "inv/z_mid"), "z_mid")
    close(lp, t(g, "inv/base_log_prob"), "base_log_prob", atol_scale=4e-5)
    if "fwd/z" in g:
        z = t(g, "fwd/z").cuda()
        y, ld, inter, _ = prog.run(z, inverse=False, want_inter=True, kernel=kernel)
        close(y, t(g, "fwd/x"), "x")
        close(ld, t(g, "fwd/ld"), "log_det fwd", atol_scale=4e-5)
        close(inter[mid - 1], t(g, "fwd/x_mid"), "x_mid")


@pytest.mark.parametrize("name", ["rnvp9_moons", "nsfcl3_stack"])
@pytest.mark.parametrize("variant", [None, 0, 1, 2, 3, 4, 5, 6])
def test_dim2_kernel_variants(name, variant):
    """The library default (staged tables) and every MNF_RUN_VARIANT(v) request (tables built in the call; 6 names that
    kernel, the others name kernels that were removed and run it too): all the table kernel."""
    from tests.test_flow_pl_gpu import _launched

    g = load_golden(name)
    sd, specs = golden_sd(g), golden_spec(g)
    model = load_flow_model(specs, sd)
    prog = model._program()
    assert prog.plan(torch.device("cuda"), 2) == 1, "BASELINE dim-2 stacks must take the table kernel"
    x = t(g, "inv/x").cuda()
    if variant is not None:
        assert _launched(lambda: prog.run(x, inverse=True, kernel=variant)) == {"flow_pl_build_kernel": 1, "flow_pl_kernel": 1}
    y, ld, _, _ = prog.run(x, inverse=True, kernel=variant)
    close(y, t(g, "inv/z"), "z", atol_scale=2e-5)
    close(ld, t(g, "inv/ld"), "log_det", atol_scale=4e-5)
    close_vs_oracle((y, ld), sd, specs, t(g, "inv/x"), True, f"{name} variant {variant}")
    # odd row count
    y, ld, _, _ = prog.run(x[:101].contiguous(), inverse=True, kernel=variant)
    close(y, t(g, "inv/z")[:101], "z odd", atol_scale=2e-5)
    close(ld, t(g, "inv/ld")[:101], "log_det odd", atol_scale=4e-5)


def test_module_api_matches_reference_contract():
    """forward(z) -> (x, log_det), container -> (list incl. input, log_det[B]) (core.py:17-35)."""
    g = load_golden("nsfcl3_stack")
    sd, specs = golden_sd(g), golden_spec(g)
    model = load_flow_model(specs, sd)
    x = t(g, "inv/x").cuda()
    zs, ld = model.inverse(x)
    assert isinstance(zs, list) and len(zs) == len(specs) + 1 and zs[0] is x
    assert ld.shape == (x.size(0),) and ld.dtype == torch.float32 and ld.is_cuda
    close(zs[-1], t(g, "inv/z"), "z", atol_scale=2e-5)
    close(model.base_log_prob(x), t(g, "inv/base_log_prob"), "base_log_prob", atol_scale=4e-5)
    close(model.log_prob(x), t(g, "inv/ld") + t(g, "inv/base_log_prob"), "log_prob", atol_scale=4e-5)
    # single-flow API and log_det shapes of the reference: [1] for affine-constant, [] for Glow
    z1, ld1 = model.flows[0].inverse(x)
    assert ld1.shape == (1,)
    z2, ld2 = model.flows[1].inverse(z1)
    assert ld2.shape == ()
    z3, ld3 = model.flows[2].inverse(z2)
    assert ld3.shape == (x.size(0),)
    # round trip (encode -> decode), the size-independent property of the domain
    xs, ld_f = model.forward(zs[-1])
    torch.testing.assert_close(xs[-1], x, rtol=1e-4, atol=2e-5)
    torch.testing.assert_close(ld_f, -ld, rtol=1e-4, atol=5e-5)
    with pytest.raises(RuntimeError):
        model.inverse(x.cpu())  # no CPU fallback


def test_actnorm_data_dependent_init():
    import torch_mnf.flows as nf

    g = load_golden("actnorm_init")
    torch.manual_seed(0)
    f = nf.ActNormFlow(3).cuda()
    z, ld = f.inverse(t(g, "x").cuda())
    assert f.data_dep_init_done
    close(f.s, t(g, "s"), "s")
    close(f.t, t(g, "t"), "t")
    close(z, t(g, "z"), "z")
    close(ld, t(g, "ld"), "ld")


def test_made_constant_bank_kernel():
    """MAF x9 dim 64 (BASELINE config 3) takes the constant-bank MADE kernel: ragged batch, intermediates,
    log-prob-only mode, against the generic interpreter and the CPU oracle."""
    g = load_golden("maf9_d64")
    specs, sd = golden_spec(g), golden_sd(g)
    model = load_flow_model(specs, sd)
    prog = model._program()
    assert prog.plan("cuda", 64) == 2
    x = torch.randn(2 * 256 + 37, 64, generator=torch.Generator().manual_seed(5))
    xg = x.cuda()
    y_f, ld_f, inter_f, lp_f = prog.run(xg, True, want_inter=True, want_base_lp=True)
    y_g, ld_g, inter_g, lp_g = prog.run(xg, True, want_inter=True, want_base_lp=True, kernel="generic")
    for a, b, what in ((y_f, y_g, "z"), (ld_f, ld_g, "ld"), (inter_f, inter_g, "inter"), (lp_f, lp_g, "base_lp")):
        torch.testing.assert_close(a, b, rtol=1e-5, atol=2e-5, msg=lambda m: f"{what}: {m}")
    y_n, ld_n, _, _ = prog.run(xg, True)  # no intermediates: in-place chain on y
    torch.testing.assert_close(y_n, y_g, rtol=1e-5, atol=2e-5)
    torch.testing.assert_close(ld_n, ld_g, rtol=1e-5, atol=2e-5)
    torch.testing.assert_close(model.log_prob(xg), ld_g + lp_g, rtol=1e-5, atol=5e-5)
    close_vs_oracle((y_f, ld_f), sd, specs, x, True, "made_fast")


def test_made_sequential_kernel():
    """MAF.forward (sampling: 64 sequential passes per flow) through the incremental sequential kernel, against the
    generic interpreter, and as the exact inverse of the density direction."""
    g = load_golden("maf9_d64")
    specs, sd = golden_spec(g), golden_sd(g)
    model = load_flow_model(specs, sd)
    prog = model._program()
    z = torch.randn(64 * 5 + 11, 64, generator=torch.Generator().manual_seed(9)).cuda()
    x_f, ld_f, inter_f, _ = prog.run(z, False, want_inter=True)
    x_g, ld_g, inter_g, _ = prog.run(z, False, want_inter=True, kernel="generic")
    torch.testing.assert_close(x_f, x_g, rtol=2e-5, atol=2e-5)
    torch.testing.assert_close(inter_f, inter_g, rtol=2e-5, atol=2e-5)
    torch.testing.assert_close(ld_f, ld_g, rtol=2e-5, atol=5e-5)
    z_back, ld_back, _, _ = prog.run(x_f, True)
    torch.testing.assert_close(z_back, z, rtol=1e-4, atol=1e-4)
    torch.testing.assert_close(ld_back, -ld_f, rtol=1e-4, atol=1e-3)


def test_graphed_log_prob_small_batch():
    """BASELINE config 1 (RNVP x9, batch 4096) replayed from a CUDA graph gives the eager result."""
    from torch_mnf.graphs import graphed_inference

    g = load_golden("rnvp9_moons")
    model = load_flow_model(golden_spec(g), golden_sd(g))
    x = t(g, "inv/x").cuda()
    x = x.repeat((4096 + x.size(0) - 1) // x.size(0), 1)[:4096].contiguous()
    call = graphed_inference(lambda v: model.log_prob(v), (x,))
    torch.testing.assert_close(call(x), model.log_prob(x), rtol=0, atol=0)
    x2 = x.flip(0).contiguous()
    torch.testing.assert_close(call(x2), model.log_prob(x2), rtol=0, atol=0)


def test_model_sample_draws_on_device():
    """NormalizingFlowModel.sample (core.py:51-55): base draw + forward; same distribution as pushing torch's own
    standard-normal draws through forward()."""
    g = load_golden("nsfcl3_stack")
    model = load_flow_model(golden_spec(g), golden_sd(g))
    torch.manual_seed(0)
    x = model.sample((4096,))
    assert x.shape == (4096, 2) and x.is_cuda and torch.isfinite(x).all()
    torch.manual_seed(0)
    z = torch.randn(4096, 2, device="cuda")
    torch.testing.assert_close(x, model.forward(z)[0][-1])
    assert model.sample(3, 5).shape == (3, 5, 2)


def test_actnorm_init_inside_a_stack():
    """Each ActNorm initialises from ITS input -- the output of the flows that run before it in the inverse
    direction (affine_constant_flow.py:42-50 called from core.py:30-33) -- not from the stack's input."""
    from oracle import flows_cpu

    specs = [{"type": "ActNormFlow", "dim": 4, "scale": True, "shift": True}, {"type": "Glow", "dim": 4},
             {"type": "ActNormFlow", "dim": 4, "scale": True, "shift": True},
             {"type": "AffineHalfFlow", "dim": 4, "parity": False, "scale": True, "shift": True, "h_sizes": [8, 8]}]
    sd = random_flow_sd(specs, seed=5, scale=0.6)
    model = load_flow_model(specs, sd)
    for f in model.flows:
        if hasattr(f, "data_dep_init_done"):
            f.data_dep_init_done = False
    x = 2.0 * torch.randn(512, 4, generator=torch.Generator().manual_seed(3)) + 1.0
    zs, ld = model.inverse(x.cuda())

    v, ld_ref = x, torch.zeros(x.size(0))
    for i in reversed(range(len(specs))):
        p = flows_cpu.sub(sd, f"flows.{i}.")
        if specs[i]["type"] == "ActNormFlow":
            p["s"], p["t"] = flows_cpu.actnorm_init(p, specs[i], v)
            close(getattr(model.flows[i], "s"), p["s"], f"flows.{i}.s")
            close(getattr(model.flows[i], "t"), p["t"], f"flows.{i}.t")
        v, l = flows_cpu.apply_flow(p, specs[i], v, True)
        ld_ref = ld_ref + l
    close(zs[-1], v, "z")
    close(ld, ld_ref, "ld")
    assert all(f.data_dep_init_done for f in model.flows if hasattr(f, "data_dep_init_done"))


ORACLE_CASES = {
    "cfg2_shape": [{"type": "ActNormFlow", "dim": 2, "scale": True, "shift": True}, {"type": "Glow", "dim": 2},
                   {"type": "NSF_CL", "dim": 2, "K": 8, "B": 3, "n_h": 16}] * 3,
    "cfg1_shape": [{"type": "AffineHalfFlow", "dim": 2, "parity": bool(i % 2), "scale": True, "shift": True,
                    "h_sizes": [24, 24, 24]} for i in range(9)],
    "nsf_default": [{"type": "NSF_CL", "dim": 2, "K": 5, "B": 3, "n_h": 8}] * 2,
    "nsf_wide_d6": [{"type": "Glow", "dim": 6}, {"type": "NSF_CL", "dim": 6, "K": 12, "B": 4, "n_h": 20},
                    {"type": "NSF_AR", "dim": 6, "K": 6, "B": 2, "n_h": 12}],
}


@pytest.mark.parametrize("name", sorted(ORACLE_CASES))
def test_stack_vs_oracle_seeded(name):
    """Bigger seeded batches (incl. tail points and exact +-B) against the CPU oracle."""
    specs = ORACLE_CASES[name]
    sd = random_flow_sd(specs, seed=3, scale=0.6 if "cfg1" not in name else 0.3)
    model = load_flow_model(specs, sd)
    dim = specs[0]["dim"]
    g = torch.Generator().manual_seed(11)
    x = 1.5 * torch.randn(20001, dim, generator=g)
    B = max([s.get("B", 3) for s in specs])
    x[0, :] = float(B)
    x[1, :] = -float(B)
    x[2, :] = 0.0
    for inverse in (True, False):
        y, ld, _, _ = model._program().run(x.cuda(), inverse=inverse)
        close_vs_oracle((y, ld), sd, specs, x, inverse, f"{name} inverse={inverse}")


def test_empty_and_single_row():
    g = load_golden("nsfcl3_stack")
    model = load_flow_model(golden_spec(g), golden_sd(g))
    zs, ld = model.inverse(torch.empty(0, 2, device="cuda"))
    assert zs[-1].shape == (0, 2) and ld.shape == (0,)
    x = t(g, "inv/x")[:1].cuda()
    zs, ld = model.inverse(x)
    close(zs[-1], t(g, "inv/z")[:1], "single row", atol_scale=2e-5)


@pytest.mark.parametrize("n_rows", [2, 3, 127, 129, 18944, 18945, 18947])
def test_small_and_ragged_batches_match_interpreter(n_rows):
    """Batches up to 148 x 128 points take the one-point-per-thread form of the dim-2 kernel, larger ones the paired form
    (odd sizes leave a half-filled last pair); both must agree with the exact-fp32 interpreter on every output."""
    for name in ("cfg2_shape", "cfg1_shape"):
        specs = ORACLE_CASES[name]
        model = load_flow_model(specs, random_flow_sd(specs, seed=4, scale=0.4))
        x = 1.2 * torch.randn(n_rows, 2, generator=torch.Generator().manual_seed(n_rows)).cuda()
        prog = model._program()
        for inverse in (True, False):
            y, ld, inter, lp = prog.run(x, inverse, want_inter=True, want_base_lp=True)
            yg, ldg, interg, lpg = prog.run(x, inverse, want_inter=True, want_base_lp=True, kernel="generic")
            # indexing test: the tolerance is the fast-math noise floor (see close_vs_oracle), a wrong row would be O(1)
            torch.testing.assert_close(y, yg, rtol=1e-4, atol=1e-4)
            torch.testing.assert_close(inter, interg, rtol=1e-4, atol=1e-4)
            torch.testing.assert_close(ld, ldg, rtol=1e-4, atol=3e-4)
            torch.testing.assert_close(lp, lpg, rtol=1e-4, atol=3e-4)
        torch.testing.assert_close(model.log_prob(x), ldg_lp(prog, x), rtol=1e-4, atol=5e-4)


def ldg_lp(prog, x):
    _, ld, _, lp = prog.run(x, True, want_base_lp=True, kernel="generic")
    return ld + lp


def test_all_points_outside_spline_domain_is_identity():
    """The reference crashes here (spline_flow.py:85, SURVEY.md 5); the drop-in maps to identity."""
    import torch_mnf.flows as nf

    torch.manual_seed(0)
    f = nf.NSF_CL(2, K=8, B=3, n_h=16).cuda()
    x = torch.tensor([[4.0, -5.0], [100.0, 3.5]], device="cuda")
    z, ld = f.inverse(x)
    assert torch.equal(z, x) and torch.equal(ld, torch.zeros(2, device="cuda"))


def test_full_size_properties_cfg2():
    """BASELINE config 2 at full size (2^24 points): round trip + log-det antisymmetry."""
    specs = ORACLE_CASES["cfg2_shape"]
    sd = random_flow_sd(specs, seed=0, scale=0.6)
    model = load_flow_model(specs, sd, return_intermediates=False)
    g = torch.Generator(device="cuda").manual_seed(0)
    x = 1.5 * torch.randn(1 << 24, 2, device="cuda", generator=g)
    zs, ld = model.inverse(x)
    xs, ld_f = model.forward(zs[-1])
    err = (xs[-1] - x).abs().max().item()
    assert err < 5e-4, err
    assert (ld + ld_f).abs().max().item() < 1e-3
    assert torch.isfinite(ld).all()
    # checksum against the oracle on a strided sample
    idx = torch.arange(0, 1 << 24, 4099, device="cuda")
    close_vs_oracle((zs[-1][idx], ld[idx]), sd, specs, x[idx].cpu(), True, "sampled")


def test_conditioner_free_stack_streaming_kernel():
    """[ActNorm, Glow] x 3 in 2-D is a single affine map: the composed streaming kernel (HBM-bound path) must agree
    with the oracle, and so must the op-by-op table kernel without tables that takes the calls the streaming kernel
    cannot (intermediates requested, an odd row count)."""
    from tests.test_flow_pl_gpu import _launched

    specs = [{"type": "ActNormFlow", "dim": 2, "scale": True, "shift": True}, {"type": "Glow", "dim": 2}] * 3
    sd = random_flow_sd(specs, seed=5, scale=0.4)
    model = load_flow_model(specs, sd, return_intermediates=False)
    prog = model._program()
    assert prog.plan(torch.device("cuda"), 2) == 1  # also packs the parameters (Glow assembly) before launches are counted
    g = torch.Generator().manual_seed(2)
    x = 2.0 * torch.randn(40000, 2, generator=g)
    xo = x[:39999]
    for inverse in (True, False):
        ref, ref_ld = flows_cpu.stack(sd, specs, x, inverse=inverse)
        stream = lambda: prog.run(x.cuda(), inverse)                       # composed streaming path
        op_by_op = lambda: prog.run(x.cuda(), inverse, want_inter=True)    # table kernel, every flow's output
        odd = lambda: prog.run(xo.cuda(), inverse)                         # table kernel, odd row count
        assert _launched(stream) == {"affine_compose_kernel": 1, "affine_stream_kernel": 1}
        assert _launched(op_by_op) == {"flow_pl_kernel": 1}
        assert _launched(odd) == {"flow_pl_kernel": 1}
        y, ld, _, _ = stream()
        y2, ld2, inter, _ = op_by_op()
        y3, ld3, _, _ = odd()
        for a, b, n in ((y, ld, 40000), (y2, ld2, 40000), (y3, ld3, 39999)):
            torch.testing.assert_close(a.cpu(), ref[-1][:n], rtol=1e-5, atol=2e-5)
            torch.testing.assert_close(b.cpu(), ref_ld[:n], rtol=1e-5, atol=1e-5)
        torch.testing.assert_close(inter.cpu(), torch.stack(ref[1:]), rtol=1e-5, atol=2e-5)
    lp = model.log_prob(x.cuda())
    torch.testing.assert_close(lp.cpu(), flows_cpu.log_prob(sd, specs, x), rtol=1e-5, atol=5e-5)


@pytest.mark.parametrize("name,n_rows", [("cfg1_shape", 4096), ("cfg2_shape", 777), ("cfg2_shape", 70001), ("nsf_wide_d6", 501)])
def test_bound_log_prob_equals_module_call(name, n_rows):
    """NormalizingFlowModel.log_prob_fn (mnf_flow_handle_*: the program bound once) returns exactly what log_prob
    returns, for the table kernel on staged tables at small and large batches, and for the interpreter."""
    specs = ORACLE_CASES[name]
    model = load_flow_model(specs, random_flow_sd(specs, seed=2, scale=0.4), return_intermediates=False)
    dim = specs[0]["dim"]
    x = 1.2 * torch.randn(n_rows, dim, generator=torch.Generator().manual_seed(n_rows)).cuda()
    f = model.log_prob_fn(max_rows=n_rows)
    want = model.log_prob(x)
    assert torch.equal(f(x), want)
    out = torch.empty(n_rows, device="cuda")
    assert f(x, out) is out and torch.equal(out, want)
    assert torch.equal(f(x[: n_rows // 2].contiguous()), model.log_prob(x[: n_rows // 2].contiguous()))
    if dim == 2:  # no row limit for dim-2 programs: twice the rows the object was made for
        xx = torch.cat([x, x])
        assert torch.equal(f(xx), model.log_prob(xx))


def test_two_programs_on_two_streams_do_not_share_state():
    """SURVEY 8b: entry points are re-entrant, the library keeps no device state.  Two different models of the benchmark
    shape, launched interleaved on two streams (the table kernel on each model's staged tables, at a large and a small batch), must give
    bit-identical results to running them one after the other."""
    specs = ORACLE_CASES["cfg2_shape"]
    models = [load_flow_model(specs, random_flow_sd(specs, seed=s, scale=0.5), return_intermediates=False) for s in (1, 2)]
    for n_rows in (70001, 3000):
        xs = [1.3 * torch.randn(n_rows, 2, generator=torch.Generator().manual_seed(10 + i)).cuda() for i in range(2)]
        serial = [m.log_prob(x).clone() for m, x in zip(models, xs)]
        torch.cuda.synchronize()
        streams = [torch.cuda.Stream(), torch.cuda.Stream()]
        outs = [[], []]
        for rep in range(6):  # interleaved: model 0 on stream 0, model 1 on stream 1, alternating
            for i in (0, 1):
                with torch.cuda.stream(streams[i]):
                    outs[i].append(models[i].log_prob(xs[i]))
        torch.cuda.synchronize()
        for i in (0, 1):
            for o in outs[i]:
                assert torch.equal(o, serial[i]), f"model {i}, {n_rows} rows: concurrent result differs from the serial one"


@pytest.mark.parametrize("n_rows", [1, 15, 16, 17, 4096, 20001])
def test_table_kernel_small_ragged_batches_match_oracle(n_rows):
    """The table kernel (the default path) on AffineHalfFlow stacks at small and ragged batch sizes: both directions,
    every output, against the oracle and the interpreter; h = 24 and h = 8."""
    for h in (24, 8):
        specs = [{"type": "ActNormFlow", "dim": 2, "scale": True, "shift": True}] + [
            {"type": "AffineHalfFlow", "dim": 2, "parity": bool(i % 2), "scale": i != 1, "shift": i != 2, "h_sizes": [h, h, h]}
            for i in range(5)] + [{"type": "Glow", "dim": 2}]
        sd = random_flow_sd(specs, seed=6, scale=0.3)
        prog = load_flow_model(specs, sd)._program()
        x = 1.2 * torch.randn(n_rows, 2, generator=torch.Generator().manual_seed(n_rows + h))
        for inverse in (True, False):
            y, ld, inter, lp = prog.run(x.cuda(), inverse, want_inter=True, want_base_lp=True)
            yg, ldg, interg, lpg = prog.run(x.cuda(), inverse, want_inter=True, want_base_lp=True, kernel="generic")
            torch.testing.assert_close(y, yg, rtol=1e-5, atol=1e-5)
            torch.testing.assert_close(inter, interg, rtol=1e-5, atol=1e-5)
            torch.testing.assert_close(ld, ldg, rtol=1e-5, atol=2e-5)
            torch.testing.assert_close(lp, lpg, rtol=1e-5, atol=2e-5)
            if n_rows >= 16:
                close_vs_oracle((y, ld), sd, specs, x, inverse, f"table kernel h={h} inverse={inverse}")


@pytest.mark.parametrize("dim,hidden", [(8, 16), (16, 32), (32, 32), (32, 16), (64, 32), (64, 16), (8, 32), (16, 16)])
def test_made_fast_kernel_shape_grid(dim, hidden):
    """The exact-fp32 MADE kernels (density and sequential direction) are instantiated for a grid of (dim, hidden)
    shapes, not only BASELINE config 3's (64, 24): each against the interpreter and the oracle."""
    specs = [{"type": "MAF", "dim": dim, "parity": bool(i % 2), "h_sizes": [hidden] * 3} for i in range(3)]
    sd = random_flow_sd(specs, seed=dim + hidden, scale=0.3)
    prog = load_flow_model(specs, sd)._program()
    assert prog.plan("cuda", dim) == 2, "shape must take the MADE kernel"
    x = torch.randn(300 + dim, dim, generator=torch.Generator().manual_seed(dim))
    y_f, ld_f, inter_f, lp_f = prog.run(x.cuda(), True, want_inter=True, want_base_lp=True)
    y_g, ld_g, inter_g, lp_g = prog.run(x.cuda(), True, want_inter=True, want_base_lp=True, kernel="generic")
    for a, b, what in ((y_f, y_g, "z"), (ld_f, ld_g, "ld"), (inter_f, inter_g, "inter"), (lp_f, lp_g, "base_lp")):
        torch.testing.assert_close(a, b, rtol=1e-5, atol=2e-5, msg=lambda m: f"{what}: {m}")
    close_vs_oracle((y_f, ld_f), sd, specs, x, True, f"made_fast<{dim},{hidden}>")
    x_f, ldx_f, _, _ = prog.run(y_f, False)  # sequential direction inverts the density direction
    x_g, ldx_g, _, _ = prog.run(y_f, False, kernel="generic")
    torch.testing.assert_close(x_f, x_g, rtol=2e-5, atol=2e-5)
    torch.testing.assert_close(ldx_f, ldx_g, rtol=2e-5, atol=5e-5)
    torch.testing.assert_close(x_f, x.cuda(), rtol=1e-4, atol=1e-4)


@pytest.mark.parametrize("n_h,K", [(8, 8), (16, 5), (32, 8), (8, 5), (24, 8)])
@pytest.mark.parametrize("n_rows", [3001, 70001])
def test_dim2_kernel_shape_grid(n_h, K, n_rows):
    """The table kernel runs a grid of (hidden width, bins), not only the BASELINE shapes, at small and large batches:
    against the oracle, with an AffineHalfFlow of the same width in the stack."""
    specs = [{"type": "ActNormFlow", "dim": 2, "scale": True, "shift": True},
             {"type": "NSF_CL", "dim": 2, "K": K, "B": 3, "n_h": n_h},
             {"type": "AffineHalfFlow", "dim": 2, "parity": True, "scale": True, "shift": True, "h_sizes": [n_h] * 3},
             {"type": "Glow", "dim": 2}, {"type": "NSF_CL", "dim": 2, "K": K, "B": 3, "n_h": n_h}]
    sd = random_flow_sd(specs, seed=n_h + K, scale=0.4)
    prog = load_flow_model(specs, sd)._program()
    assert prog.plan("cuda", 2) == 1, "shape must take the table kernel"
    x = 1.4 * torch.randn(n_rows, 2, generator=torch.Generator().manual_seed(n_h * K))
    for inverse in (True, False):
        y, ld, _, _ = prog.run(x.cuda(), inverse)
        close_vs_oracle((y, ld), sd, specs, x, inverse, f"dim2 n_h={n_h} K={K} inverse={inverse}")
