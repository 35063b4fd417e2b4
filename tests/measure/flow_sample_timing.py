"""Timing of flow sampling on BASELINE config 2's stack (ActNorm + Glow + NSF_CL(K=8, n_h=16), x3; the stack
tests/measure/flow_pl_timing.py builds) at 2^24 points:
  (a) sample_and_log_prob: Philox draw, forward pass and log q(x) in one launch of the table kernel
  (b) sample(): torch.randn + forward
  (c) sample() + log_prob(x): the composition a caller needs today for the density of its draws
  (d) forward pass of the table kernel on a resident z (x and log_det out, as mnf_flow_stack_run writes them)
CUDA events around 5 calls per round, variants alternated round by round, median of the rounds.  Card name, power
limit and max SM clock are read in the same run.
Run on a GPU box:  python tests/measure/flow_sample_timing.py [log2_rows] [rounds]"""
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path[:0] = [os.path.join(ROOT, "torch-mnf_b200"), ROOT]
import torch

from tests.helpers import load_flow_model, random_flow_sd

torch.set_grad_enabled(False)
specs = [{"type": "ActNormFlow", "dim": 2, "scale": True, "shift": True}, {"type": "Glow", "dim": 2},
         {"type": "NSF_CL", "dim": 2, "K": 8, "B": 3, "n_h": 16}] * 3
sd = random_flow_sd(specs, seed=0, scale=0.6)
model = load_flow_model(specs, sd, device="cuda:0", return_intermediates=False)
prog = model._program()
n = 1 << (int(sys.argv[1]) if len(sys.argv) > 1 else 24)
rounds = int(sys.argv[2]) if len(sys.argv) > 2 else 7
z = torch.randn(n, 2, device="cuda", generator=torch.Generator(device="cuda").manual_seed(0))
y, ld = torch.empty_like(z), torch.empty(n, device="cuda")

variants = {
    "a_sample_and_log_prob": lambda: model.sample_and_log_prob(n, seed=1),
    "b_sample": lambda: model.sample(n),
    "c_sample_then_log_prob": lambda: model.log_prob(model.sample(n)),
    "d_forward_resident_z": lambda: prog.run(z, False, out=y, log_det=ld),
}
times = {k: [] for k in variants}
for fn in variants.values():
    for _ in range(3):
        fn()
torch.cuda.synchronize()
for _ in range(rounds):
    for k, fn in variants.items():
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(5):
            fn()
        e1.record()
        torch.cuda.synchronize()
        times[k].append(e0.elapsed_time(e1) / 5)

out = {"rows": n, "rounds": rounds}
try:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True, timeout=30).stdout.strip()
    out["gpu"] = q
except Exception as e:  # noqa: BLE001
    out["gpu"] = f"nvidia-smi unavailable: {e}"
out["gpu_torch"] = torch.cuda.get_device_name(0)
for k, v in times.items():
    out[f"{k}_ms_median"] = statistics.median(v)
    out[f"{k}_ms_min"] = min(v)
    out[f"{k}_ms_max"] = max(v)
a, c, d = (out[f"{k}_ms_median"] for k in ("a_sample_and_log_prob", "c_sample_then_log_prob", "d_forward_resident_z"))
out["a_over_d"] = a / d
out["c_over_a"] = c / a

# the same draws, scored by the inverse pass: how far log q(x) from the forward pass is from log_prob(x)
x, lp = model.sample_and_log_prob(1 << 20, seed=2)
dlp = (model.log_prob(x) - lp).abs()
out["log_prob_of_sample_max_abs_diff"] = float(dlp.max())
out["log_prob_of_sample_mean_abs_diff"] = float(dlp.mean())
print(json.dumps(out))
