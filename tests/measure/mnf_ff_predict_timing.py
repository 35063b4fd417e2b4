"""Timing of MNFFeedForward's Monte-Carlo prediction on two shapes:
  [784, 1024, 1024, 10], B = 1024, S = 100   (hidden layers on the tcgen05 path)
  [8, 50, 50, 1],        B = 4096, S = 500   (exact-fp32 SIMT path throughout)
variants, alternated round by round in one run:
  (a) predict(x, S, seed=): forward_mc chunk by chunk (ReLU + folded BatchNorm1d in the layer epilogues, x read through
      its B distinct rows) and mnf_mc_moments into fp64 sums -> mean, var
  (b) the eval-mode model(x.repeat(S, 1)) followed by torch mean / population variance over the samples
  (c) forward_mc(x, S, seed=) alone, no reduction (one chunk)
CUDA events around 3 calls per round, median of the rounds.  Card name, power limit and SM clocks are read in the same
run.  Run on a GPU box:  python tests/measure/mnf_ff_predict_timing.py [rounds]"""
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path[:0] = [os.path.join(ROOT, "torch-mnf_b200"), ROOT]
import torch

from torch_mnf.models import MNFFeedForward

torch.set_grad_enabled(False)
rounds = int(sys.argv[1]) if len(sys.argv) > 1 else 7


def trained_looking(sizes, seed):
    torch.manual_seed(seed)
    model = MNFFeedForward(sizes)
    for i in range(2, len(model), 3):
        bn = model[i]
        bn.running_mean.normal_(0, 0.05)
        bn.running_var.uniform_(0.5, 2.0)
        bn.weight.normal_(1, 0.2)
        bn.bias.normal_(0, 0.2)
    return model.cuda().eval()


def repeat_baseline(model, x, S):
    y = model(x.repeat(S, 1)).view(S, x.size(0), -1)
    return y.mean(0), y.var(0, unbiased=False)


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader",
                            "-i", "0"], capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        q = f"nvidia-smi unavailable: {e}"
    return q


out = {"rounds": rounds, "gpu_torch": torch.cuda.get_device_name(0), "shapes": []}
for sizes, B, S in (([784, 1024, 1024, 10], 1024, 100), ([8, 50, 50, 1], 4096, 500)):
    model = trained_looking(sizes, seed=0)
    x = torch.randn(B, sizes[0], device="cuda", generator=torch.Generator(device="cuda").manual_seed(1))
    variants = {
        "a_predict": lambda: model.predict(x, S, seed=1),
        "b_repeat_then_torch_moments": lambda: repeat_baseline(model, x, S),
        "c_forward_mc_only": lambda: model.forward_mc(x, S, seed=1),
    }
    times = {k: [] for k in variants}
    for fn in variants.values():
        for _ in range(2):
            fn()
    torch.cuda.synchronize()
    for _ in range(rounds):
        for k, fn in variants.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(3):
                fn()
            e1.record()
            torch.cuda.synchronize()
            times[k].append(e0.elapsed_time(e1) / 3)
    rec = {"sizes": sizes, "B": B, "S": S, "chunk": max(1, MNFFeedForward.CHUNK_FLOATS // (B * max(sizes))),
           "gpu_after": gpu_info()}
    for k, v in times.items():
        rec[f"{k}_ms_median"] = statistics.median(v)
        rec[f"{k}_ms_min"] = min(v)
        rec[f"{k}_ms_max"] = max(v)
    rec["b_over_a"] = rec["b_repeat_then_torch_moments_ms_median"] / rec["a_predict_ms_median"]
    # the two estimates of the predictive mean draw different noise; their gap is Monte-Carlo error, reported as a check
    m_a, v_a = model.predict(x, S, seed=1)
    m_b, v_b = repeat_baseline(model, x, S)
    rec["mean_abs_gap_a_vs_b"] = float((m_a - m_b).abs().mean())
    rec["mean_sd"] = float(v_a.sqrt().mean())
    out["shapes"].append(rec)
    del model, x
    torch.cuda.empty_cache()
out["gpu"] = gpu_info()
print(json.dumps(out))
