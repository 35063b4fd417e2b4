"""The fast form of the piecewise-linear tables (csrc/flow_pl.cu): the staged image against the numpy restatement of
tests/pl_fast_reference.py, and stacks whose tables take the fast form, the plain form or both against the oracle."""

import numpy as np
import pytest
import torch

from tests import pl_fast_reference as plf
from tests import pl_reference as plr
from tests.helpers import golden_sd, golden_spec, load_flow_model, load_golden, random_flow_sd, t
from tests.test_flows_gpu import ORACLE_CASES, close_vs_oracle

pytestmark = pytest.mark.gpu

PL = 6  # MNF_RUN_VARIANT(6)
LN2 = float(np.log(2.0))


def _nsf_layout(K):
    """flow_pl.cu: row stride, origin slot, (slope, value) slots of every output of an NSF_CL row."""
    org = 4 * K + (2 * (K - 1) + 3) // 4 * 4
    ia = np.array([4 * (o >> 1) + (o & 1) if o < 2 * K else 4 * K + 2 * (o - 2 * K) for o in range(3 * K - 1)])
    iv = np.array([ia[o] + 2 if o < 2 * K else ia[o] + 1 for o in range(3 * K - 1)])
    return 4 * ((org // 4 + 1) | 1), org, ia, iv


def _tables(model, sd, specs):
    """(spec, nets, image, header row, float offset of the region, row stride) of every table of the staged image."""
    from torch_mnf import _lib

    prog = model._program()
    prog._build(torch.device("cuda:0"))
    img = prog._staged_image(_lib.lib(), 1, 2, None)
    torch.cuda.synchronize()
    raw = img.cpu().numpy()
    hdr = raw[:256].view(np.int32).reshape(64, 4)
    off, gi = 256, 0
    for i, spec in enumerate(specs):
        if spec["type"] not in ("NSF_CL", "AffineHalfFlow"):
            continue
        stride = _nsf_layout(spec["K"])[0] if spec["type"] == "NSF_CL" else 12
        for nets in plr.nets_of_flow(sd, i, spec):
            yield spec, nets, raw, hdr[gi], off, stride
            off += 512 + 512 * stride
            gi += 1


def _piece_samples(F, j):
    """Points of fast piece j (both ends included where finite)."""
    nf = len(F)
    if 0 < j < nf:
        return float(F[j - 1]) + (float(F[j]) - float(F[j - 1])) * np.array([0.0, 0.25, 0.5, 0.75, 1.0])
    e = float(F[0] if j == 0 else F[-1])
    return e + (-1.0 if j == 0 else 1.0) * max(1.0, abs(e)) * np.array([0.0, 0.5, 3.0, 10.0])


def check_fast_forms(model, sd, specs):
    """Every table's fast form (if it has one) against the restatement.  Returns (fast tables, plain tables, tables with splits)."""
    n_fast = n_plain = n_split = 0
    rng = np.random.default_rng(0)
    for spec, nets, raw, h, off, stride in _tables(model, sd, specs):
        if h[1]:
            continue  # overflowed: evaluated layer by layer
        n = int(h[0])
        f = plf.parse(raw, off, h, stride)
        if f is None:
            n_plain += 1
            continue
        n_fast += 1
        grid, recs, rows = f
        F = plf.breakpoints(recs)
        nf = len(F)
        assert rows.shape == (nf + 1, stride), (rows.shape, nf)
        n_split += nf > n
        # every fast piece lies inside one original piece: the original breakpoints are among the fast ones
        bp32 = raw[off:off + n]
        u, cu = np.unique(bp32, return_counts=True)
        uf, cf = np.unique(F, return_counts=True)
        k = np.minimum(np.searchsorted(uf, u), len(uf) - 1) if len(uf) else np.zeros(0, int)
        assert len(u) == 0 or ((uf[k] == u).all() and (cf[k] >= cu).all())
        # bucket lookup == count of fast breakpoints below c
        scale = max(1.0, float(np.abs(F).max())) if nf else 1.0
        c = np.concatenate([F, np.nextafter(F, np.float32(np.inf)), np.nextafter(F, np.float32(-np.inf)),
                            (rng.standard_normal(20000) * scale).astype(np.float32),
                            np.array([1e30, -1e30, np.inf, -np.inf, 0.0], np.float32)]).astype(np.float32)
        np.testing.assert_array_equal(plf.lookup(c, grid, recs), np.searchsorted(F, c, "left"))
        assert plf.lookup(np.array([np.nan], np.float32), grid, recs)[0] == 0
        if spec["type"] != "NSF_CL":
            continue
        K = spec["K"]
        _, org_slot, ia, iv = _nsf_layout(K)
        bp = plr.breakpoints(nets)
        tab = plr.tables(nets, bp)
        for j in range(nf + 1):
            if 0 < j < nf and F[j - 1] == F[j]:
                continue  # zero width: never selected
            pts = _piece_samples(F, j)
            mid = pts[2]
            (A, B), = tab[int(np.searchsorted(bp, mid))]
            out = A[None, :] * pts[:, None] + B[None, :]  # natural units, exact
            d = pts - float(rows[j, org_slot])
            z = rows[j, ia][None, :].astype(np.float64) * d[:, None] + rows[j, iv][None, :].astype(np.float64)  # log2 units
            for ax in (slice(0, K), slice(K, 2 * K)):
                zm = z[:, ax].max(axis=1)
                assert (zm >= -1e-4).all() and (zm <= plf.FAST_T + 1e-3).all(), (j, zm)  # the envelope invariant
                pf = np.exp2(z[:, ax] - zm[:, None])
                pf /= pf.sum(axis=1, keepdims=True)
                o = out[:, ax]
                po = np.exp(o - o.max(axis=1, keepdims=True))
                po /= po.sum(axis=1, keepdims=True)
                np.testing.assert_allclose(pf, po, rtol=2e-5, atol=1e-6)
            dsc = 1.0 + np.abs(out[:, 2 * K:]).max()
            np.testing.assert_allclose(z[:, 2 * K:] * LN2, out[:, 2 * K:], rtol=0, atol=2e-6 * dsc)
    return n_fast, n_plain, n_split


def _both_directions_vs_oracle(model, sd, specs, x, what, x_fwd=None):
    prog = model._program()
    for inverse, xi in ((True, x), (False, x if x_fwd is None else x_fwd)):
        y, ld, _, _ = prog.run(xi.cuda(), inverse, kernel=PL)
        close_vs_oracle((y, ld), sd, specs, xi, inverse, f"{what} inverse={inverse}")


@pytest.mark.parametrize("name", ["cfg2_shape", "nsfcl3_stack", "rnvp9_moons"])
def test_fast_forms(name):
    if name in ORACLE_CASES:
        specs = ORACLE_CASES[name]
        sd = random_flow_sd(specs, seed=7, scale=0.6)
        x = x_fwd = 1.5 * torch.randn(30001, 2, generator=torch.Generator().manual_seed(13))
    else:  # the golden points (the trained RNVP stack's inverse leaves fp32 range on wide Gaussian inputs)
        g = load_golden(name)
        sd, specs = golden_sd(g), golden_spec(g)
        x, x_fwd = t(g, "inv/x"), t(g, "fwd/z")
    model = load_flow_model(specs, sd)
    n_fast, n_plain, _ = check_fast_forms(model, sd, specs)
    # the spline tables all get a fast form; of the RNVP tables (~140 kinks spread over +-500) only those whose kinks a
    # grid of <= 1024 buckets separates
    assert n_fast > 0 and (n_plain == 0 or name == "rnvp9_moons"), (n_fast, n_plain)
    _both_directions_vs_oracle(model, sd, specs, x, f"{name} fast", x_fwd)


def test_fast_and_plain_tables_in_one_stack():
    """Four coincident first-layer kinks (no bucket grid holds them) and a 1-64x5 scale net next to fast tables."""
    specs = [{"type": "NSF_CL", "dim": 2, "K": 8, "B": 3, "n_h": 16},
             {"type": "AffineHalfFlow", "dim": 2, "parity": True, "scale": True, "shift": False, "h_sizes": [64] * 5},
             {"type": "Glow", "dim": 2},
             {"type": "NSF_CL", "dim": 2, "K": 8, "B": 3, "n_h": 16}]
    sd = random_flow_sd(specs, seed=3, scale=0.4)
    for u in (1, 2, 3):
        sd["flows.0.f1.0.weight"][u] = sd["flows.0.f1.0.weight"][0]
        sd["flows.0.f1.0.bias"][u] = sd["flows.0.f1.0.bias"][0]
    model = load_flow_model(specs, sd)
    n_fast, n_plain, _ = check_fast_forms(model, sd, specs)
    assert n_fast >= 3 and n_plain >= 1, (n_fast, n_plain)
    x = 1.3 * torch.randn(30001, 2, generator=torch.Generator().manual_seed(5))
    _both_directions_vs_oracle(model, sd, specs, x, "mixed fast / plain")


def test_steep_outputs_split_pieces():
    """Width / height outputs scaled by 300 (weights and biases, so every gap between an axis's upper envelope and the
    line a piece stores relative to grows 300x): some pieces exceed FAST_T and are cut so that no exponent does; end to
    end the result is as close to the exact one as the reference's own fp32 arithmetic (up to 4x, as for the steep cases
    of tests/test_flow_pl_gpu.py)."""
    from oracle import flows_cpu

    specs = [{"type": "NSF_CL", "dim": 2, "K": 8, "B": 3, "n_h": 16}, {"type": "Glow", "dim": 2},
             {"type": "NSF_CL", "dim": 2, "K": 8, "B": 3, "n_h": 16}]
    sd = random_flow_sd(specs, seed=11, scale=0.6)
    last = max(int(k.split(".")[-2]) for k in sd if k.startswith("flows.0.f2.") and k.endswith("weight"))
    sd[f"flows.0.f2.{last}.weight"][:16] *= 300.0
    sd[f"flows.0.f2.{last}.bias"][:16] *= 300.0
    nets = plr.nets_of_flow(sd, 0, specs[0])[1]
    assert plf.max_envelope_gap(nets, 8) > plf.FAST_T  # the case does need cuts
    model = load_flow_model(specs, sd)
    n_fast, _, n_split = check_fast_forms(model, sd, specs)
    assert n_fast > 0 and n_split > 0, (n_fast, n_split)
    x = 1.3 * torch.randn(20000, 2, generator=torch.Generator().manual_seed(6))
    sd64 = {k: (v.double() if v.is_floating_point() else v) for k, v in sd.items()}
    for inverse in (True, False):
        y, ld, _, _ = model._program().run(x.cuda(), inverse, kernel=PL)
        ref32, ld32 = flows_cpu.stack(sd, specs, x, inverse=inverse)
        ref64, ld64 = flows_cpu.stack(sd64, specs, x.double(), inverse=inverse)
        for got, r32, r64 in ((y, ref32[-1], ref64[-1]), (ld, ld32, ld64)):
            err = (got.cpu().double() - r64).abs().flatten()
            ref_err = (r32.double() - r64).abs().flatten()
            floor = 1e-5 * max(1.0, float(r64.abs().mean()))
            assert float(err.max()) <= 4.0 * float(ref_err.max()) + floor, (float(err.max()), float(ref_err.max()))
            assert float(err.mean()) <= 4.0 * float(ref_err.mean()) + floor


def test_huge_conditioner_inputs():
    """|c| up to 1e30 with the transformed coordinate inside [-B, B]: the outer pieces of a fast table, where every
    exponent but the extreme line's is hugely negative.  (Knot-derivative outputs made constant: softplus of +-1e30 is
    beyond what the reference's fp32 spline survives.)"""
    specs = [{"type": "NSF_CL", "dim": 2, "K": 8, "B": 3, "n_h": 16}]
    sd = random_flow_sd(specs, seed=4, scale=0.6)
    for net in ("f1", "f2"):
        last = max(int(k.split(".")[-2]) for k in sd if k.startswith(f"flows.0.{net}.") and k.endswith("weight"))
        sd[f"flows.0.{net}.{last}.weight"][16:] = 0.0
    model = load_flow_model(specs, sd)
    assert check_fast_forms(model, sd, specs)[0] == 2
    g = torch.Generator().manual_seed(8)
    n = 20000
    c = torch.sign(torch.randn(n, generator=g)) * 10.0 ** (30.0 * torch.rand(n, generator=g))
    v = 5.0 * torch.rand(n, generator=g) - 2.5
    x = torch.stack([c, v], 1)
    x[n // 2:] = x[n // 2:].flip(1)
    _both_directions_vs_oracle(model, sd, specs, x, "huge c")
