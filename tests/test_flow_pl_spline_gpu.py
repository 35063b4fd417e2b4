"""Spline conditioners of the table kernel (csrc/flow_pl.cu) where its arithmetic is at its edges: a stack whose
per-point log-det product spans many binades (the running product is renormalised on every conditioner) and the
widest spline bound a fast table takes (the FMA-pipe 2^x sees its whole argument range).  Both directions against
the oracle."""

import pytest
import torch

from oracle import flows_cpu
from tests.helpers import load_flow_model, random_flow_sd
from tests.test_flow_pl_fast_gpu import _both_directions_vs_oracle, check_fast_forms

pytestmark = pytest.mark.gpu

FAST_B_MAX = 32.0


def _scale_last_layer(sd, i, rows, factor):
    for net in ("f1", "f2"):
        last = max(int(k.split(".")[-2]) for k in sd if k.startswith(f"flows.{i}.{net}.") and k.endswith("weight"))
        sd[f"flows.{i}.{net}.{last}.weight"][rows] *= factor
        sd[f"flows.{i}.{net}.{last}.bias"][rows] *= factor


def test_log_det_spanning_many_binades():
    """Six fast-form splines with steepened knot derivatives: the log-dets of the points span more than 17 binades."""
    specs = [{"type": "NSF_CL", "dim": 2, "K": 8, "B": 3, "n_h": 16}, {"type": "Glow", "dim": 2}] * 3
    sd = random_flow_sd(specs, seed=21, scale=0.6)
    for i in (0, 2, 4):
        _scale_last_layer(sd, i, slice(16, None), 2.0)  # knot-derivative outputs
    model = load_flow_model(specs, sd)
    n_fast, n_plain, _ = check_fast_forms(model, sd, specs)
    assert n_fast == 6 and n_plain == 0, (n_fast, n_plain)
    x = 1.2 * torch.randn(30001, 2, generator=torch.Generator().manual_seed(17))
    _, ld = flows_cpu.stack(sd, specs, x, inverse=True)
    assert float(ld.max() - ld.min()) > 12.0, float(ld.max() - ld.min())  # > 17 binades
    _both_directions_vs_oracle(model, sd, specs, x, "many binades")


def test_widest_fast_spline_bound():
    """B = FAST_B_MAX: the widest bound a fast table takes; the second softmax's arguments reach +-B log2e = +-46."""
    specs = [{"type": "NSF_CL", "dim": 2, "K": 8, "B": FAST_B_MAX, "n_h": 16}, {"type": "Glow", "dim": 2},
             {"type": "NSF_CL", "dim": 2, "K": 8, "B": FAST_B_MAX, "n_h": 16}]
    sd = random_flow_sd(specs, seed=23, scale=0.6)
    model = load_flow_model(specs, sd)
    n_fast, n_plain, _ = check_fast_forms(model, sd, specs)
    assert n_fast == 4 and n_plain == 0, (n_fast, n_plain)
    x = 12.0 * torch.randn(30001, 2, generator=torch.Generator().manual_seed(19))
    _both_directions_vs_oracle(model, sd, specs, x, "B = FAST_B_MAX")
