"""GPU parity of the piecewise-linear table kernel (csrc/flow_pl.cu, dim-2 kernel variant 6 and the library default for
AffineHalfFlow / NSF_CL stacks): golden vectors of the reference, the CPU oracle on seeded batches, and the exact-fp32
interpreter on the cases that exercise the kernel's own machinery (tables staged per parameter version or built per call,
tables larger than shared memory, tables that overflow and fall back to the layer-by-layer evaluation, inputs far outside
the breakpoints, conditioner shapes no other fast kernel covers)."""

import pytest
import torch

from tests.helpers import golden_sd, golden_spec, load_flow_model, load_golden, random_flow_sd, t
from tests.test_flows_gpu import ORACLE_CASES, close, close_vs_oracle

pytestmark = pytest.mark.gpu

PL = 6  # MNF_RUN_VARIANT(6)


def _launched(fn):
    from torch_mnf import _lib

    _lib.launch_stats(reset=True)
    fn()
    torch.cuda.synchronize()
    return _lib.launch_stats()


@pytest.mark.parametrize("name", ["rnvp9_moons", "nsfcl3_stack"])
def test_pl_vs_golden(name):
    g = load_golden(name)
    sd, specs = golden_sd(g), golden_spec(g)
    model = load_flow_model(specs, sd)
    prog = model._program()
    x = t(g, "inv/x").cuda()
    sites = _launched(lambda: prog.run(x, inverse=True, kernel=PL))
    assert "flow_pl_kernel" in sites and "flow_pl_build_kernel" in sites, sites
    y, ld, inter, lp = prog.run(x, inverse=True, want_inter=True, want_base_lp=True, kernel=PL)
    close(y, t(g, "inv/z"), "z", atol_scale=2e-5)
    close(ld, t(g, "inv/ld"), "log_det", atol_scale=4e-5)
    close(lp, t(g, "inv/base_log_prob"), "base_log_prob", atol_scale=4e-5)
    close(inter[(len(specs) + 1) // 2 - 1], t(g, "inv/z_mid"), "z_mid")
    close_vs_oracle((y, ld), sd, specs, t(g, "inv/x"), True, f"{name} pl")
    z = t(g, "fwd/z").cuda()
    y, ld, _, _ = prog.run(z, inverse=False, kernel=PL)
    close(y, t(g, "fwd/x"), "x")
    close(ld, t(g, "fwd/ld"), "log_det fwd", atol_scale=4e-5)
    close_vs_oracle((y, ld), sd, specs, t(g, "fwd/z"), False, f"{name} pl fwd")


def test_default_path_is_the_table_kernel():
    """Module calls of the BASELINE dim-2 stacks: the tables are staged once per parameter version, a call of any size is
    ONE launch; an explicit variant request (no staging) builds them inside the call."""
    for name, rows, want in (("cfg1_shape", 4096, {"flow_pl_kernel": 1}), ("cfg2_shape", 1 << 16, {"flow_pl_kernel": 1})):
        specs = ORACLE_CASES[name]
        model = load_flow_model(specs, random_flow_sd(specs, seed=1, scale=0.4), return_intermediates=False)
        x = torch.randn(rows, 2, device="cuda")
        model.log_prob(x)  # first call stages
        assert _launched(lambda: model.log_prob(x)) == want
        assert _launched(lambda: model._program().run(x, True, log_prob_only=True, kernel=PL)) == {"flow_pl_build_kernel": 1, "flow_pl_kernel": 1}


@pytest.mark.parametrize("name,scale", [("cfg2_shape", 0.6), ("cfg1_shape", 0.3), ("nsf_default", 0.6)])
def test_pl_vs_oracle_seeded(name, scale):
    specs = ORACLE_CASES[name]
    sd = random_flow_sd(specs, seed=7, scale=scale)
    model = load_flow_model(specs, sd)
    g = torch.Generator().manual_seed(13)
    x = 1.5 * torch.randn(30001, 2, generator=g)
    x[0, :], x[1, :], x[2, :] = 3.0, -3.0, 0.0
    for inverse in (True, False):
        y, ld, _, _ = model._program().run(x.cuda(), inverse=inverse, kernel=PL)
        close_vs_oracle((y, ld), sd, specs, x, inverse, f"{name} pl inverse={inverse}")


SHAPES = {
    # conditioner shapes outside the (hidden, bins) grid of the earlier dim-2 kernels: any depth 2..6, any widths <= 64
    "affine_32_16": [{"type": "AffineHalfFlow", "dim": 2, "parity": bool(i % 2), "scale": True, "shift": True, "h_sizes": [32, 16]} for i in range(4)],
    "affine_one_hidden": [{"type": "AffineHalfFlow", "dim": 2, "parity": bool(i % 2), "scale": True, "shift": True, "h_sizes": [40]} for i in range(3)],
    "affine_scale_only": [{"type": "AffineHalfFlow", "dim": 2, "parity": False, "scale": True, "shift": False, "h_sizes": [24, 24, 24]},
                          {"type": "AffineHalfFlow", "dim": 2, "parity": True, "scale": False, "shift": True, "h_sizes": [24, 24, 24]}],
    "nsf_h20": [{"type": "Glow", "dim": 2}, {"type": "NSF_CL", "dim": 2, "K": 8, "B": 2.5, "n_h": 20}] * 2,
    "mixed": [{"type": "ActNormFlow", "dim": 2, "scale": True, "shift": True},
              {"type": "AffineHalfFlow", "dim": 2, "parity": True, "scale": True, "shift": True, "h_sizes": [16, 16, 16]},
              {"type": "NSF_CL", "dim": 2, "K": 8, "B": 3, "n_h": 16}, {"type": "Glow", "dim": 2},
              {"type": "AffineHalfFlow", "dim": 2, "parity": False, "scale": True, "shift": True, "h_sizes": [16, 16, 16]}],
    # every instantiated bin count
    "nsf_k4_k16": [{"type": "NSF_CL", "dim": 2, "K": 4, "B": 3, "n_h": 12}, {"type": "Glow", "dim": 2}, {"type": "NSF_CL", "dim": 2, "K": 4, "B": 3, "n_h": 12}],
    "nsf_k6": [{"type": "NSF_CL", "dim": 2, "K": 6, "B": 2, "n_h": 16}] * 2,
    "nsf_k10": [{"type": "NSF_CL", "dim": 2, "K": 10, "B": 4, "n_h": 16}] * 2,
    "nsf_k12": [{"type": "NSF_CL", "dim": 2, "K": 12, "B": 3, "n_h": 24}] * 2,
    "nsf_k16": [{"type": "ActNormFlow", "dim": 2, "scale": True, "shift": True}, {"type": "NSF_CL", "dim": 2, "K": 16, "B": 3, "n_h": 16}] * 2,
    # tables that do not fit: 6 tables of ~200 pieces x 208 B > 227 KB of shared memory -> read from the image in global memory
    "nsf_h64_x3": [{"type": "NSF_CL", "dim": 2, "K": 8, "B": 3, "n_h": 64}] * 3,
    # an (s, t) pair of 1-64-64-64-64-64-1 nets has ~600 breakpoints > 511: flagged by the builder, evaluated layer by layer
    "affine_overflow": [{"type": "AffineHalfFlow", "dim": 2, "parity": bool(i % 2), "scale": True, "shift": True, "h_sizes": [64] * 5} for i in range(2)]
                       + [{"type": "NSF_CL", "dim": 2, "K": 8, "B": 3, "n_h": 16}],
}


@pytest.mark.parametrize("name", sorted(SHAPES))
@pytest.mark.parametrize("rows", [777, 70001])
def test_pl_shapes_match_interpreter(name, rows):
    specs = SHAPES[name]
    model = load_flow_model(specs, random_flow_sd(specs, seed=5, scale=0.6 if "affine" not in name else 0.3))
    prog = model._program()
    x = 1.3 * torch.randn(rows, 2, generator=torch.Generator().manual_seed(rows)).cuda()
    for inverse in (True, False):
        sites = _launched(lambda: prog.run(x, inverse, kernel=PL))
        assert "flow_pl_kernel" in sites, sites
        y, ld, inter, lp = prog.run(x, inverse, want_inter=True, want_base_lp=True, kernel=PL)
        yg, ldg, interg, lpg = prog.run(x, inverse, want_inter=True, want_base_lp=True, kernel="generic")
        torch.testing.assert_close(y, yg, rtol=1e-4, atol=1e-4)
        torch.testing.assert_close(inter, interg, rtol=1e-4, atol=1e-4)
        torch.testing.assert_close(ld, ldg, rtol=1e-4, atol=3e-4)
        torch.testing.assert_close(lp, lpg, rtol=1e-4, atol=3e-4)


def test_pl_staged_equals_built_per_call():
    """The same points through the staged tables (module call) and through tables built inside the call (explicit variant)."""
    specs = ORACLE_CASES["cfg2_shape"]
    model = load_flow_model(specs, random_flow_sd(specs, seed=2, scale=0.6), return_intermediates=False)
    x = 1.5 * torch.randn(1 << 17, 2, device="cuda")
    big = model._program().run(x, True, log_prob_only=True, kernel=PL)[3]
    assert torch.equal(model.log_prob(x), big)
    small = torch.cat([model.log_prob(x[i:i + 30000].contiguous()) for i in range(0, x.size(0), 30000)])
    assert torch.equal(big, small)
    bound = model.log_prob_fn(1 << 17)
    assert torch.equal(bound(x), big)


def test_pl_tracks_parameter_updates():
    """The staged tables are rebuilt when a parameter changes (cache keyed on every tensor's version)."""
    specs = ORACLE_CASES["cfg1_shape"]
    model = load_flow_model(specs, random_flow_sd(specs, seed=2, scale=0.3), return_intermediates=False)
    x = torch.randn(2048, 2, device="cuda")
    a = model.log_prob(x)
    with torch.no_grad():
        model.flows[4].s_net[2].weight.mul_(1.5)
    b = model.log_prob(x)
    _, _, _, ref = model._program().run(x, True, log_prob_only=True, kernel="generic")
    assert not torch.equal(a, b)
    torch.testing.assert_close(b, ref, rtol=1e-4, atol=3e-4)


def test_pl_far_inputs_and_non_finite():
    """Coordinates far beyond every breakpoint use the outermost pieces (exact: the net is linear there); NaN / inf inputs
    give what the layer-by-layer evaluation gives."""
    specs = ORACLE_CASES["cfg1_shape"]
    sd = random_flow_sd(specs, seed=9, scale=0.05)  # small weights: exp(s) stays finite at |c| ~ 1e4
    model = load_flow_model(specs, sd)
    x = torch.randn(4096, 2, generator=torch.Generator().manual_seed(3))
    x[:1024] *= 1e4
    x[5, 0], x[6, 1], x[7, 0] = float("nan"), float("inf"), float("-inf")
    prog = model._program()
    for inverse in (True, False):
        y, ld, _, _ = prog.run(x.cuda(), inverse, kernel=PL)
        yg, ldg, _, _ = prog.run(x.cuda(), inverse, kernel="generic")
        fin = torch.isfinite(yg).all(dim=1) & torch.isfinite(ldg)
        assert torch.equal(torch.isfinite(y).all(dim=1) & torch.isfinite(ld), fin)
        torch.testing.assert_close(y[fin], yg[fin], rtol=2e-5, atol=1e-5)
        torch.testing.assert_close(ld[fin], ldg[fin], rtol=2e-5, atol=1e-4)
    specs = ORACLE_CASES["cfg2_shape"]
    sd = random_flow_sd(specs, seed=9, scale=0.6)
    model = load_flow_model(specs, sd)
    x = 1e6 * torch.randn(4096, 2, generator=torch.Generator().manual_seed(4))  # spline tails: identity, log-det 0
    y, ld, _, _ = model._program().run(x.cuda(), True, kernel=PL)
    close_vs_oracle((y, ld), sd, specs, x, True, "cfg2 far inputs")


def _check_tables_against_numpy(model, sd, specs):
    """The tables flow_pl_build_kernel writes (the staged image) against tests/pl_reference.py: same breakpoints, same
    per-piece slopes and values.  Image layout: flow_pl.cu (header of 4 ints per table, then per table 512 padded
    breakpoints and 512 rows)."""
    import numpy as np

    from tests import pl_reference as plr
    from torch_mnf import _lib

    prog = model._program()
    prog._build(torch.device("cuda:0"))
    img = prog._staged_image(_lib.lib(), 1, 2, None)
    torch.cuda.synchronize()
    assert img is not None
    raw = img.cpu().numpy()
    hdr = raw[:256].view(np.int32).reshape(64, 4)
    off, gi = 256, 0
    for i, spec in enumerate(specs):
        if spec["type"] not in ("NSF_CL", "AffineHalfFlow"):
            continue
        nsf = spec["type"] == "NSF_CL"
        stride = 52 if nsf else 12
        for nets in plr.nets_of_flow(sd, i, spec):
            bp = plr.breakpoints(nets)
            tab = plr.tables(nets, bp)
            n = int(hdr[gi, 0])
            assert hdr[gi, 1] == 0 and n == len(bp), (gi, n, len(bp))
            got_bp = raw[off:off + 512]
            np.testing.assert_allclose(got_bp[:n], bp.astype(np.float32), rtol=1e-6, atol=1e-30)
            assert np.isinf(got_bp[n:]).all()
            rows = raw[off + 512:off + 512 + (n + 1) * stride].reshape(n + 1, stride)
            for piece in range(n + 1):
                if 0 < piece < n and got_bp[piece - 1] == got_bp[piece]:
                    continue  # coincident breakpoints: a piece of zero width is never selected (and has no interior point)
                org = float(got_bp[0] if piece == 0 else got_bp[piece - 1]) if n else 0.0
                assert rows[piece, 48 if nsf else 4] == np.float32(org)
                for q, (A, B) in enumerate(tab[piece]):
                    V = A * org + B
                    if nsf:
                        K = spec["K"]
                        ia = np.array([4 * (o >> 1) + (o & 1) if o < 2 * K else 4 * K + 2 * (o - 2 * K) for o in range(3 * K - 1)])
                        iv = np.array([ia[o] + 2 if o < 2 * K else ia[o] + 1 for o in range(3 * K - 1)])
                    else:
                        ia, iv = np.array([q]), np.array([2 + q])
                    scale = np.abs(A).max() + np.abs(V).max() + 1e-30
                    np.testing.assert_allclose(rows[piece, ia], A, rtol=0, atol=3e-7 * scale)
                    np.testing.assert_allclose(rows[piece, iv], V, rtol=0, atol=3e-7 * scale)
            off += 512 + 512 * stride
            gi += 1
    assert gi > 0


@pytest.mark.parametrize("name", ["rnvp9_moons", "nsfcl3_stack"])
def test_cuda_builder_matches_numpy_restatement(name):
    g = load_golden(name)
    sd, specs = golden_sd(g), golden_spec(g)
    _check_tables_against_numpy(load_flow_model(specs, sd), sd, specs)


DEGENERATE = ["dead_units", "constant_net", "duplicate_units", "steep", "very_steep", "no_first_layer_kink", "kink_beyond_fp32", "all"]


@pytest.mark.parametrize("case", DEGENERATE)
def test_pl_degenerate_conditioners(case):
    """Dead first-layer units (zero weight: no kink), an all-zero hidden layer (constant conditioner), duplicated units
    (coincident kinks), large first-layer weights (kinks packed around zero, steep pieces) and a first layer without any
    kink: the tables against the oracle in fp32 AND fp64 (the criterion of tests/test_flows_gpu.py::close_vs_oracle: as
    close to the exact result as the reference's own arithmetic).  "very_steep" (first-layer weights x 1e4, activations of
    ~1e3) is a regime where the fp32 layer-by-layer evaluation itself is only good to ~1e-2: there the tables must be no
    further from the exact (fp64) result than the reference's own fp32 arithmetic is."""
    specs = [{"type": "AffineHalfFlow", "dim": 2, "parity": False, "scale": True, "shift": True, "h_sizes": [16, 16, 16]},
             {"type": "NSF_CL", "dim": 2, "K": 8, "B": 3, "n_h": 16},
             {"type": "AffineHalfFlow", "dim": 2, "parity": True, "scale": True, "shift": True, "h_sizes": [16, 16, 16]}]
    sd = random_flow_sd(specs, seed=21, scale=0.5)
    if case in ("dead_units", "all"):
        sd["flows.0.s_net.0.weight"][:5] = 0.0
    if case in ("constant_net", "all"):
        sd["flows.0.t_net.2.weight"].zero_()
        sd["flows.0.t_net.2.bias"].zero_()
    if case in ("duplicate_units", "all"):
        sd["flows.1.f1.0.weight"][3] = sd["flows.1.f1.0.weight"][2]
        sd["flows.1.f1.0.bias"][3] = sd["flows.1.f1.0.bias"][2]
    if case in ("steep", "all"):
        sd["flows.1.f2.0.weight"].mul_(1e2)
    if case == "very_steep":
        sd["flows.1.f2.0.weight"].mul_(1e4)
    if case in ("kink_beyond_fp32", "all"):
        sd["flows.0.s_net.0.weight"][7] = 1e-39   # -b/w ~ 1e38 .. 1e39: outside what fp32 can hold
        sd["flows.0.s_net.0.weight"][8] = -3e-39
    if case in ("no_first_layer_kink", "all"):
        sd["flows.2.s_net.4.weight"].mul_(0.01)
        sd["flows.2.t_net.0.weight"].zero_()
    model = load_flow_model(specs, sd)
    _check_tables_against_numpy(model, sd, specs)  # the builder itself, entry by entry
    prog = model._program()
    x = torch.randn(20000, 2, generator=torch.Generator().manual_seed(2))
    x[:100, 0] = 0.0
    x[100:200] *= 1e-5
    steep = case in ("steep", "very_steep", "all")
    for inverse in (True, False):
        sites = _launched(lambda: prog.run(x.cuda(), inverse, kernel=PL))
        assert "flow_pl_kernel" in sites, sites
        y, ld, _, _ = prog.run(x.cuda(), inverse, kernel=PL)
        if not steep:
            close_vs_oracle((y, ld), sd, specs, x, inverse, f"degenerate {case} inverse={inverse}")
            continue
        # raw spline parameters of +-50 .. +-5000: bins at the 1e-3 floor next to bins of width ~6 amplify every rounding of
        # the (fast-math) spline by ~1e3, in the reference's own fp32 as well -- here the tables are what is under test
        # (checked entry by entry above), end to end only the order of magnitude: no further from the exact result than
        # 4x the reference's own fp32 error
        from oracle import flows_cpu

        ref32, ld32 = flows_cpu.stack(sd, specs, x, inverse=inverse)
        sd64 = {k: (v.double() if v.is_floating_point() else v) for k, v in sd.items()}
        ref64, ld64 = flows_cpu.stack(sd64, specs, x.double(), inverse=inverse)
        for got, r32, r64 in ((y, ref32[-1], ref64[-1]), (ld, ld32, ld64)):
            err = (got.cpu().double() - r64).abs().flatten()
            ref_err = (r32.double() - r64).abs().flatten()
            floor = 1e-5 * max(1.0, float(r64.abs().mean()))
            assert float(err.max()) <= 4.0 * float(ref_err.max()) + floor, (float(err.max()), float(ref_err.max()))
            k = int(0.99 * err.numel())
            assert float(err.kthvalue(k).values) <= 4.0 * float(ref_err.kthvalue(k).values) + floor
            assert float(err.mean()) <= 4.0 * float(ref_err.mean()) + floor
