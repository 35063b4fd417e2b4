"""Runs the cfg2 flow stack a few times with a chosen kernel variant (for ncu captures)."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "torch-mnf_b200"), ROOT]
import torch

torch.set_grad_enabled(False)  # inference kernels; training goes through mnf_flow_stack_backward
from tests.helpers import load_flow_model, random_flow_sd
from tests.test_flows_gpu import ORACLE_CASES

name = os.environ.get("CASE", "cfg2_shape")
variant = os.environ.get("VARIANT", "6")
variant = variant if variant == "generic" else int(variant)
n = int(os.environ.get("N", 1 << 24))
specs = ORACLE_CASES[name]
model = load_flow_model(specs, random_flow_sd(specs, seed=0, scale=0.6), return_intermediates=False)
x = 1.5 * torch.randn(n, 2, device="cuda", generator=torch.Generator(device="cuda").manual_seed(0))
lp = torch.empty(n, device="cuda")
for _ in range(int(os.environ.get("ITERS", 4))):
    model._program().run(x, True, log_prob_only=True, log_prob_out=lp, kernel=variant)
torch.cuda.synchronize()
print("done", float(lp.mean()))
