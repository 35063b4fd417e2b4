"""Timing of Monte-Carlo predictive uncertainty (predict_uncertainty) next to the prediction it extends:
  MNFLeNet, config 4's shape: 1024 images x 500 samples, chunk 25 (tensor-core branch), the golden trained weights
    (a) predict                                   fp32 sums of exp(log-probs) per chunk in torch
    (b) predict_uncertainty                       mnf_mc_class_moments per chunk, fp64 sums + entropy sums
    (c) predict_uncertainty(per_sample_conv_z=True)   one conv z per sample
  MNFFeedForward([784, 1024, 1024, 10]), B = 1024, S = 100 (hidden layers on tcgen05), trained-looking batch norms
    (d) predict(softmax=True)
    (e) predict_uncertainty
  and the reduction alone on one config-4 chunk of log-probs [25 * 1024, 10]:
    (f) mnf_mc_moments(softmax = 1)   (g) mnf_mc_class_moments
CUDA events around 3 calls per round, the variants of a group alternated round by round, median of the rounds.  Card
name, power limit and SM clocks are read in the same run.  Run on a GPU box:
    python tests/measure/mc_uncertainty_timing.py [rounds]"""
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path[:0] = [os.path.join(ROOT, "torch-mnf_b200"), ROOT]
import torch

from tests.helpers import golden_sd, load_golden
from torch_mnf.layers import _mnf_ops as ops
from torch_mnf.models import MNFFeedForward, MNFLeNet

torch.set_grad_enabled(False)
rounds = int(sys.argv[1]) if len(sys.argv) > 1 else 7


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader",
                            "-i", "0"], capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        q = f"nvidia-smi unavailable: {e}"
    return q


def time_group(variants, reps=3):
    for fn in variants.values():
        for _ in range(2):
            fn()
    torch.cuda.synchronize()
    times = {k: [] for k in variants}
    for _ in range(rounds):
        for k, fn in variants.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                fn()
            e1.record()
            torch.cuda.synchronize()
            times[k].append(e0.elapsed_time(e1) / reps)
    rec = {}
    for k, v in times.items():
        rec[f"{k}_ms_median"] = statistics.median(v)
        rec[f"{k}_ms_min"] = min(v)
        rec[f"{k}_ms_max"] = max(v)
    return rec


out = {"rounds": rounds, "gpu_torch": torch.cuda.get_device_name(0), "gpu_before": gpu_info()}

# ---- MNFLeNet, config 4 ---------------------------------------------------------------------------------------------
net = MNFLeNet()
net.load_state_dict(golden_sd(load_golden("mnf_lenet")))
net.cuda()
x = torch.rand(1024, 1, 28, 28, generator=torch.Generator().manual_seed(0)).cuda()
S, chunk = 500, 25
rec = time_group({
    "a_predict": lambda: net.predict(x, S, chunk=chunk, seed=1),
    "b_predict_uncertainty": lambda: net.predict_uncertainty(x, S, chunk=chunk, seed=1),
    "c_predict_uncertainty_per_sample_z": lambda: net.predict_uncertainty(x, S, chunk=chunk, seed=1,
                                                                          per_sample_conv_z=True),
})
rec["b_over_a"] = rec["b_predict_uncertainty_ms_median"] / rec["a_predict_ms_median"]
rec["c_over_a"] = rec["c_predict_uncertainty_per_sample_z_ms_median"] / rec["a_predict_ms_median"]
u = net.predict_uncertainty(x, S, chunk=chunk, seed=1)
up = net.predict_uncertainty(x, S, chunk=chunk, seed=1, per_sample_conv_z=True)
rec["max_abs_mean_gap_b_vs_a"] = float((u.mean - net.predict(x, S, chunk=chunk, seed=1)).abs().max())
for name, v in (("shared_z", u), ("per_sample_z", up)):
    rec[f"{name}_mean_predictive_entropy"] = float(v.predictive_entropy.mean())
    rec[f"{name}_mean_expected_entropy"] = float(v.expected_entropy.mean())
    rec[f"{name}_mean_mutual_information"] = float(v.mutual_information.mean())
out["lenet_cfg4"] = {"B": 1024, "S": S, "chunk": chunk, **rec}

# the reduction alone on one chunk of config-4 log-probs
lp = torch.log_softmax(torch.randn(chunk * 1024, 10, device="cuda") * 3, dim=-1)
sums = torch.zeros(2, 1024, 10, device="cuda", dtype=torch.float64)
ent = torch.zeros(1024, device="cuda", dtype=torch.float64)
out["reduction_one_chunk"] = time_group({
    "f_mc_moments_softmax": lambda: ops.mc_moments(lp, 1024, chunk, sums, softmax=True),
    "g_mc_class_moments": lambda: ops.mc_moments(lp, 1024, chunk, sums, softmax=True, entropy_sums=ent),
}, reps=50)
del net, x, lp
torch.cuda.empty_cache()

# ---- MNFFeedForward -------------------------------------------------------------------------------------------------
sizes, B, S = [784, 1024, 1024, 10], 1024, 100
torch.manual_seed(0)
model = MNFFeedForward(sizes)
for i in range(2, len(model), 3):
    bn = model[i]
    bn.running_mean.normal_(0, 0.05)
    bn.running_var.uniform_(0.5, 2.0)
    bn.weight.normal_(1, 0.2)
    bn.bias.normal_(0, 0.2)
model = model.cuda().eval()
x = torch.randn(B, sizes[0], device="cuda", generator=torch.Generator(device="cuda").manual_seed(1))
rec = time_group({
    "d_predict_softmax": lambda: model.predict(x, S, seed=1, softmax=True),
    "e_predict_uncertainty": lambda: model.predict_uncertainty(x, S, seed=1),
})
rec["e_over_d"] = rec["e_predict_uncertainty_ms_median"] / rec["d_predict_softmax_ms_median"]
out["feed_forward"] = {"sizes": sizes, "B": B, "S": S,
                       "chunk": max(1, MNFFeedForward.CHUNK_FLOATS // (B * max(sizes))), **rec}
out["gpu"] = gpu_info()
print(json.dumps(out))
