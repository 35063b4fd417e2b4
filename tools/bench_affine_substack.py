"""HBM-bound sub-stack of config 2: [ActNormFlow, Glow] x 3 (no conditioner MLPs), 2^24 points."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "torch-mnf_b200"), ROOT]
import torch

torch.set_grad_enabled(False)  # inference kernels; training goes through mnf_flow_stack_backward
from tests.helpers import load_flow_model, random_flow_sd
specs = [{"type": "ActNormFlow", "dim": 2, "scale": True, "shift": True}, {"type": "Glow", "dim": 2}] * 3
model = load_flow_model(specs, random_flow_sd(specs, seed=0), return_intermediates=False)
n = 1 << 24
x = torch.randn(n, 2, device="cuda")
prog = model._program()
print("plan (1 = dim-2 kernels):", prog.plan(x.device, 2))
y = torch.empty_like(x); ld = torch.empty(n, device="cuda"); lp = torch.empty(n, device="cuda")
def t(fn, it=10):
    fn(); torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(it)]
    for a, b in ev:
        a.record(); fn(); b.record()
    torch.cuda.synchronize()
    return min(a.elapsed_time(b) for a, b in ev)
ms = t(lambda: prog.run(x, True, out=y, log_det=ld))
print(f"inverse (z + log_det, 20 B/pt): {ms:.3f} ms  {20*n/ms/1e6:.0f} GB/s  {n/ms/1e6:.2f} Gpts/s")
ms = t(lambda: prog.run(x, True, log_prob_only=True, log_prob_out=lp))
print(f"log_prob only (12 B/pt): {ms:.3f} ms  {12*n/ms/1e6:.0f} GB/s  {n/ms/1e6:.2f} Gpts/s")
