"""Timing + error statistics of the piecewise-linear table kernel (variant 6, flow_pl.cu: tables built in the call) on
BASELINE config 2, and of the config-1 bound call.
Run on a GPU box:  python tests/measure/flow_pl_timing.py [log2_rows]"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path[:0] = [os.path.join(ROOT, "torch-mnf_b200"), ROOT]
import torch

from tests.helpers import golden_sd, golden_spec, load_flow_model, load_golden, random_flow_sd

torch.set_grad_enabled(False)
specs = [{"type": "ActNormFlow", "dim": 2, "scale": True, "shift": True}, {"type": "Glow", "dim": 2},
         {"type": "NSF_CL", "dim": 2, "K": 8, "B": 3, "n_h": 16}] * 3
sd = random_flow_sd(specs, seed=0, scale=0.6)
model = load_flow_model(specs, sd, device="cuda:0", return_intermediates=False)
prog = model._program()
n = 1 << (int(sys.argv[1]) if len(sys.argv) > 1 else 24)
x = 1.5 * torch.randn(n, 2, device="cuda", generator=torch.Generator(device="cuda").manual_seed(0))
out = {"rows": n}
lp_out = torch.empty(n, device="cuda")
lps = {}
for kernel in (6,):
    for _ in range(3):
        prog.run(x, True, log_prob_only=True, kernel=kernel, log_prob_out=lp_out)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5):
        prog.run(x, True, log_prob_only=True, kernel=kernel, log_prob_out=lp_out)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 5
    out[f"k{kernel}_ms"] = ms
    out[f"k{kernel}_gpts"] = n / ms / 1e6
    lps[kernel] = lp_out[: 1 << 16].clone()
_, _, _, lpg = prog.run(x[: 1 << 16].contiguous(), True, log_prob_only=True, kernel="generic")
for k in (6,):
    d = (lps[k] - lpg).abs()
    out[f"k{k}_vs_generic_max"] = float(d.max())
    out[f"k{k}_vs_generic_mean"] = float(d.mean())
print(json.dumps(out))

# config 1: RNVP x9 bound call, 4096 points
g = load_golden("rnvp9_moons")
m1 = load_flow_model(golden_spec(g), golden_sd(g), device="cuda:0", return_intermediates=False)
res = {}
for rows in (256, 4096, 65536):
    x1 = torch.randn(rows, 2, device="cuda")
    f = m1.log_prob_fn(rows)
    o = torch.empty(rows, device="cuda")
    for _ in range(20):
        f(x1, o)
    torch.cuda.synchronize()
    import time
    t0 = time.perf_counter()
    for _ in range(200):
        f(x1, o)
    torch.cuda.synchronize()
    res[f"bound_call_us_{rows}"] = (time.perf_counter() - t0) / 200 * 1e6
    _, _, _, lpg = m1._program().run(x1, True, log_prob_only=True, kernel="generic")
    res[f"max_abs_diff_vs_generic_{rows}"] = float((o - lpg).abs().max())
print(json.dumps(res))
