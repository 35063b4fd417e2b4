"""Shared helpers for the parity tests (golden loading, spec handling)."""

import json
import os

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")


def load_golden(name):
    return np.load(os.path.join(GOLDEN, name + ".npz"))


def golden_sd(npz, prefix="sd/"):
    return {k[len(prefix):]: torch.from_numpy(npz[k]).clone() for k in npz.keys() if k.startswith(prefix)}


def golden_spec(npz):
    return json.loads(str(npz["spec"]))


def golden_tape(npz, prefix):
    from oracle.noise import NoiseTape  # lazy: bench.py's product arm imports this module for the model builders only

    return NoiseTape.from_npz(npz, prefix)


def t(npz, key):
    return torch.from_numpy(npz[key]).clone()


def max_rel(a, b, atol=0.0):
    a, b = a.double(), b.double()
    return float(((a - b).abs() / (b.abs() + atol + 1e-30)).max())


# ---------------------------------------------------------------------------
# building product modules from a golden spec
# ---------------------------------------------------------------------------
def build_flow(spec):
    import torch_mnf.flows as nf

    t = spec["type"]
    if t == "AffineConstantFlow":
        return nf.AffineConstantFlow(spec["dim"], scale=spec["scale"], shift=spec["shift"])
    if t == "ActNormFlow":
        f = nf.ActNormFlow(spec["dim"], scale=spec["scale"], shift=spec["shift"])
        f.data_dep_init_done = True  # golden weights are post-init
        return f
    if t == "AffineHalfFlow":
        return nf.AffineHalfFlow(spec["dim"], spec["parity"], h_sizes=tuple(spec["h_sizes"]),
                                 scale=spec["scale"], shift=spec["shift"])
    if t == "Glow":
        return nf.Glow(spec["dim"])
    if t in ("MAF", "IAF"):
        return getattr(nf, t)(spec["dim"], spec["parity"], h_sizes=tuple(spec["h_sizes"]))
    if t in ("NSF_CL", "NSF_AR"):
        return getattr(nf, t)(spec["dim"], K=spec["K"], B=spec["B"], n_h=spec["n_h"])
    if t == "RNVP":
        return nf.RNVP(spec["dim"], h_sizes=tuple(spec["h_sizes"]))
    raise ValueError(t)


def load_flow_model(specs, sd, device="cuda", return_intermediates=True):
    """Product NormalizingFlowModel with the golden/reference state_dict loaded (strict)."""
    import torch_mnf.flows as nf
    from torch.distributions import MultivariateNormal

    dim = specs[0]["dim"]
    flows = [build_flow(s) for s in specs]
    base = MultivariateNormal(torch.zeros(dim), torch.eye(dim))
    model = nf.NormalizingFlowModel(base, flows, return_intermediates=return_intermediates)
    extras = {k: v for k, v in sd.items() if k.endswith(".P")}
    model.load_state_dict({k: v for k, v in sd.items() if k not in extras}, strict=True)
    for k, v in extras.items():  # Glow.P is not part of the state_dict (glow.py:14)
        model.flows[int(k.split(".")[1])].P.copy_(v)
    return model.to(device)


def random_flow_sd(specs, seed=0, scale=0.5):
    """A reference-shaped state_dict with seeded random values (for oracle-vs-CUDA cases that
    have no golden file).  Built from the product modules' own shapes."""
    model = load_flow_model_unloaded(specs)
    g = torch.Generator().manual_seed(seed)
    sd = {}
    for k, v in model.state_dict().items():
        if v.dtype == torch.bool:
            sd[k] = v.clone()
        elif k.endswith(".S"):
            sd[k] = (0.5 + torch.rand(v.shape, generator=g)) * (torch.randint(0, 2, v.shape, generator=g) * 2 - 1)
        else:
            sd[k] = scale * torch.randn(v.shape, generator=g) / max(1.0, float(v.shape[-1]) ** 0.5 if v.dim() > 1 else 1.0)
    for i, f in enumerate(model.flows):
        if type(f).__name__ == "Glow":
            sd[f"flows.{i}.P"] = torch.eye(f.dim)[torch.randperm(f.dim, generator=g)]
    return sd


def load_flow_model_unloaded(specs):
    import torch_mnf.flows as nf
    from torch.distributions import MultivariateNormal

    dim = specs[0]["dim"]
    return nf.NormalizingFlowModel(MultivariateNormal(torch.zeros(dim), torch.eye(dim)), [build_flow(s) for s in specs])


# ---------------------------------------------------------------------------
# oracle flow stacks that torch autograd can differentiate
# ---------------------------------------------------------------------------
def nsf_ar_forward_functional(p, spec, v):
    """oracle.flows_cpu.nsf_ar(inverse=False) without the in-place column writes: the reference's NSF_AR.forward
    (spline_flow.py:199-216) assigns x[:, i] in place after x[:, :i] fed the conditioner, which torch autograd rejects, so
    the reference itself cannot differentiate this direction; the CUDA backward can, and is checked against this."""
    from oracle import flows_cpu

    d, K, B = spec["dim"], spec["K"], spec["B"]
    cols, ld = [], torch.zeros(v.shape[0], dtype=v.dtype)
    for i in range(d):
        raw = (p["init_param"].expand(v.shape[0], 3 * K - 1) if i == 0
               else flows_cpu.mlp(flows_cpu.sub(p, f"layers.{i - 1}."), torch.stack(cols, 1)))
        W, H, D = flows_cpu._spline_params(raw, K, B)
        col, l = flows_cpu.unconstrained_rqs(v[:, i], W, H, D, True, B)
        cols.append(col)
        ld = ld + l
    return torch.stack(cols, 1), ld


def oracle_stack(sd, specs, v, inverse):
    """oracle.flows_cpu.stack, with NSF_AR.forward replaced by its autograd-friendly form."""
    from oracle import flows_cpu

    if inverse or not any(s["type"] == "NSF_AR" for s in specs):
        return flows_cpu.stack(sd, specs, v, inverse)
    ld, outs = torch.zeros(v.size(0), dtype=v.dtype), [v]
    for i, spec in enumerate(specs):
        p = flows_cpu.sub(sd, f"flows.{i}.")
        v, l = (nsf_ar_forward_functional(p, spec, v) if spec["type"] == "NSF_AR"
                else flows_cpu.apply_flow(p, spec, v, False))
        ld = ld + l
        outs.append(v)
    return outs, ld
