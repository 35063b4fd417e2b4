"""Parity table (VERDICT r1 item 1c): for every flow fixture recorded from the reference, both directions and every
kernel that can run it, the fraction of output elements inside

  literal : |got - ref| <= 1e-5 * |ref|                         (BASELINE.json north_star, no absolute floor)
  adopted : |got - ref| <= 1e-5 * |ref| + floor * scale         (floor 2e-5 for outputs, 4e-5 for log-dets,
                                                                 scale = max(1, mean |ref|); BASELINE.md section 5)

where `ref` is the value the reference itself produced (tests/golden/*.npz), plus the same two fractions for the
fp32 ORACLE against an fp64 evaluation of the same formulas -- i.e. how well the reference's own fp32 arithmetic meets
the literal criterion.  The table is written to gpurun_out/r02_parity_table.json (copied to profiles/ and committed);
the test asserts the adopted criterion on every element and that the CUDA kernels are no further from the exact (fp64)
result than 2x the reference's own fp32 error."""

import json
import os

import pytest
import torch

from oracle import flows_cpu
from tests.helpers import ROOT, golden_sd, golden_spec, load_flow_model, load_golden, random_flow_sd, t

pytestmark = pytest.mark.gpu

FLOW_CASES = ["rnvp9_moons", "nsfcl3_stack", "nsfcl_d4", "nsfar2_d3", "maf9_d64", "maf3_d8", "maf_iaf_d2",
              "affine_misc_d4"]
FLOOR = {"out": 2e-5, "log_det": 4e-5}


def _fractions(got, ref, floor):
    got, ref = got.double(), ref.double()
    err = (got - ref).abs()
    scale = max(1.0, float(ref.abs().mean()))
    return {
        "n": int(ref.numel()),
        "frac_literal_rtol_1e-5": float((err <= 1e-5 * ref.abs()).double().mean()),
        "frac_adopted": float((err <= 1e-5 * ref.abs() + floor * scale).double().mean()),
        "max_abs_err": float(err.max()),
        "max_rel_err": float((err / ref.abs().clamp_min(1e-30)).max()),
    }


def _kernels_for(prog, dim):
    ks = [("default", None), ("generic", "generic")]
    if dim == 2 and prog.plan(torch.device("cuda"), 2) == 1:
        ks += [(f"dim2_variant{v}", v) for v in (6,)]  # table kernel, tables built in the call
    return ks


def test_write_parity_table():
    table = {"criterion": {"literal": "|got-ref| <= 1e-5*|ref|",
                           "adopted": "|got-ref| <= 1e-5*|ref| + floor*max(1, mean|ref|), floor 2e-5 (outputs) / 4e-5 (log-dets)",
                           "ref": "outputs recorded from the reference itself (tests/golden), torch 2.11 CPU fp32"},
             "fixtures": {}}
    worst_adopted = 1.0
    for name in FLOW_CASES:
        g = load_golden(name)
        sd, specs = golden_sd(g), golden_spec(g)
        model = load_flow_model(specs, sd)
        prog = model._program()
        dim = specs[0]["dim"]
        sd64 = {k: (v.double() if v.is_floating_point() else v) for k, v in sd.items()}
        entry = {}
        for direction, xin, kout, kld in (("inverse", "inv/x", "inv/z", "inv/ld"), ("forward", "fwd/z", "fwd/x", "fwd/ld")):
            if xin not in g:
                continue
            x = t(g, xin)
            inverse = direction == "inverse"
            r64, l64 = flows_cpu.stack(sd64, specs, x.double(), inverse=inverse)
            ref_out, ref_ld = t(g, kout), t(g, kld)
            row = {"reference_fp32_vs_fp64": {
                "out": _fractions(ref_out, r64[-1], FLOOR["out"]), "log_det": _fractions(ref_ld, l64, FLOOR["log_det"])}}
            for label, kernel in _kernels_for(prog, dim):
                y, ld, _, _ = prog.run(x.cuda(), inverse=inverse, kernel=kernel)
                y, ld = y.cpu(), ld.cpu()
                fr = {"out": _fractions(y, ref_out, FLOOR["out"]), "log_det": _fractions(ld, ref_ld, FLOOR["log_det"]),
                      "out_vs_fp64": _fractions(y, r64[-1], FLOOR["out"]), "log_det_vs_fp64": _fractions(ld, l64, FLOOR["log_det"])}
                row[label] = fr
                worst_adopted = min(worst_adopted, fr["out"]["frac_adopted"], fr["log_det"]["frac_adopted"])
                # as exact as the reference: error vs fp64 within 2x the reference's own fp32 error (+ the floor)
                for key, ref_key, fl in (("out_vs_fp64", "out", FLOOR["out"]), ("log_det_vs_fp64", "log_det", FLOOR["log_det"])):
                    scale = max(1.0, float((r64[-1] if ref_key == "out" else l64).abs().mean()))
                    own = row["reference_fp32_vs_fp64"][ref_key]["max_abs_err"]
                    assert fr[key]["max_abs_err"] <= 2.0 * own + fl * scale, (name, direction, label, key, fr[key], own)
            entry[direction] = row
        table["fixtures"][name] = entry
    # the bench configuration (cfg2 stack, seeded weights, 20 001 points incl. tails): no recorded reference output
    # exists at this size, so `ref` is the fp32 oracle (bit-identical to the reference on every golden, test_oracle_golden)
    specs = [{"type": "ActNormFlow", "dim": 2, "scale": True, "shift": True}, {"type": "Glow", "dim": 2},
             {"type": "NSF_CL", "dim": 2, "K": 8, "B": 3, "n_h": 16}] * 3
    sd = random_flow_sd(specs, seed=3, scale=0.6)
    x = 1.5 * torch.randn(20001, 2, generator=torch.Generator().manual_seed(11))
    model = load_flow_model(specs, sd)
    prog = model._program()
    sd64 = {k: (v.double() if v.is_floating_point() else v) for k, v in sd.items()}
    entry = {}
    for direction in ("inverse", "forward"):
        inverse = direction == "inverse"
        r32, l32 = flows_cpu.stack(sd, specs, x, inverse=inverse)
        r64, l64 = flows_cpu.stack(sd64, specs, x.double(), inverse=inverse)
        row = {"reference_fp32_vs_fp64": {"out": _fractions(r32[-1], r64[-1], FLOOR["out"]),
                                          "log_det": _fractions(l32, l64, FLOOR["log_det"])}}
        for label, kernel in _kernels_for(prog, 2):
            y, ld, _, _ = prog.run(x.cuda(), inverse=inverse, kernel=kernel)
            row[label] = {"out": _fractions(y.cpu(), r32[-1], FLOOR["out"]), "log_det": _fractions(ld.cpu(), l32, FLOOR["log_det"]),
                          "out_vs_fp64": _fractions(y.cpu(), r64[-1], FLOOR["out"]),
                          "log_det_vs_fp64": _fractions(ld.cpu(), l64, FLOOR["log_det"])}
        entry[direction] = row
    table["fixtures"]["cfg2_seeded_20001 (ref = fp32 oracle)"] = entry
    table["worst_frac_adopted_on_goldens"] = worst_adopted
    for d in (os.path.join(ROOT, "gpurun_out"),):
        try:
            os.makedirs(d, exist_ok=True)
            with open(os.path.join(d, "r02_parity_table.json"), "w") as f:
                json.dump(table, f, indent=1)
        except OSError:
            pass
    assert worst_adopted == 1.0, f"adopted criterion violated on a golden fixture: worst fraction {worst_adopted}"
