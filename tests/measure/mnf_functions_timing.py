"""Timing of posterior function samples (MNFLinear / MNFFeedForward.forward_functions) on three shapes:
  (a) MNFFeedForward([784, 1024, 1024, 10]), eval, B = 1024, S = 100: forward_functions next to forward_mc(x, 100), which
      covers the same B * S rows (forward_mc at the default precision, whose hidden layers run on the TF32 tensor cores,
      and at precision "fp32", the exact SIMT path the function GEMM also runs)
  (b) the same model, B = 8, S = 1024: the Thompson-sampling shape, where the weight draw dominates
  (c) MNFLinear(4096, 4096), B = 64, S = 64
CUDA events around 3 calls per round after two warm-up calls, rounds alternated between the variants, median of the
rounds.  A separate torch.profiler run of each forward_functions call splits its kernel time between the weight draw
(function_weights_kernel), the function GEMM (simt_gemm_kernel<MnfFunctionProb>) and the rest (z draws and q-flows).
Rates from shapes: normals/s = S * sum(n_out * (n_in + 1)) over the draw kernel's time, FMA/s = S * B * sum(n_in * n_out)
over the GEMM's.  Card name and power limit are read in the same run.
Run on a GPU box:  python tests/measure/mnf_functions_timing.py [rounds] [out.json]"""
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path[:0] = [os.path.join(ROOT, "torch-mnf_b200"), ROOT]
import torch
from torch.profiler import ProfilerActivity, profile

from torch_mnf.layers import MNFLinear
from torch_mnf.models import MNFFeedForward

torch.set_grad_enabled(False)
rounds = int(sys.argv[1]) if len(sys.argv) > 1 else 7
out_path = sys.argv[2] if len(sys.argv) > 2 else None


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm",
                               "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                              timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        return f"nvidia-smi unavailable: {e}"


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


def time_variants(variants):
    for fn in variants.values():
        for _ in range(2):
            fn()
    torch.cuda.synchronize()
    times = {k: [] for k in variants}
    for _ in range(rounds):
        for k, fn in variants.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(3):
                fn()
            e1.record()
            torch.cuda.synchronize()
            times[k].append(e0.elapsed_time(e1) / 3)
    return {k: {"ms_median": statistics.median(v), "ms_min": min(v), "ms_max": max(v)} for k, v in times.items()}


def kernel_split(fn):
    """Device time (ms) of one call of fn per kernel class, from a torch.profiler run of its own."""
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    split = {"draw": 0.0, "gemm": 0.0, "other": 0.0}
    for ev in prof.key_averages():
        us = getattr(ev, "device_time_total", None)
        if us is None:
            us = ev.cuda_time_total
        if us <= 0:
            continue
        if "function_weights_kernel" in ev.key:
            split["draw"] += us / 1e3
        elif "MnfFunctionProb" in ev.key:
            split["gemm"] += us / 1e3
        else:
            split["other"] += us / 1e3
    return split


def rates(split, layers, B, S):
    normals = S * sum(o * (i + 1) for i, o in layers)
    fmas = S * B * sum(i * o for i, o in layers)
    return {"normals": normals, "fmas": fmas,
            "draw_normals_per_s": normals / (split["draw"] / 1e3) if split["draw"] else None,
            "gemm_fma_per_s": fmas / (split["gemm"] / 1e3) if split["gemm"] else None}


out = {"rounds": rounds, "gpu_torch": torch.cuda.get_device_name(0), "gpu": gpu_info(), "cases": []}
ff_sizes = [784, 1024, 1024, 10]
ff_layers = list(zip(ff_sizes[:-1], ff_sizes[1:]))
for name, B, S in (("a", 1024, 100), ("b", 8, 1024)):
    model = trained_looking(ff_sizes, seed=0)
    x = torch.randn(B, ff_sizes[0], device="cuda", generator=torch.Generator(device="cuda").manual_seed(1))
    fp32 = trained_looking(ff_sizes, seed=0)
    for m in fp32:
        if isinstance(m, MNFLinear):
            m.precision = "fp32"
    variants = {
        "forward_functions": lambda: model.forward_functions(x, S, seed=1),
        "forward_mc_default": lambda: model.forward_mc(x, S, seed=1),
        "forward_mc_fp32": lambda: fp32.forward_mc(x, S, seed=1),
    }
    rec = {"case": name, "sizes": ff_sizes, "B": B, "S": S, "times": time_variants(variants)}
    rec["split_ms"] = kernel_split(variants["forward_functions"])
    rec.update(rates(rec["split_ms"], ff_layers, B, S))
    rec["gpu_after"] = gpu_info()
    out["cases"].append(rec)
    print(json.dumps(rec), flush=True)
    del model, fp32, x
    torch.cuda.empty_cache()

torch.manual_seed(0)
layer = MNFLinear(4096, 4096).cuda()
x = torch.randn(64, 4096, device="cuda", generator=torch.Generator(device="cuda").manual_seed(1))
variants = {"forward_functions": lambda: layer.forward_functions(x, 64, seed=1),
            "forward_mc_default": lambda: layer.forward_mc(x, 64)}
rec = {"case": "c", "sizes": [4096, 4096], "B": 64, "S": 64, "times": time_variants(variants)}
rec["split_ms"] = kernel_split(variants["forward_functions"])
rec.update(rates(rec["split_ms"], [(4096, 4096)], 64, 64))
rec["gpu_after"] = gpu_info()
out["cases"].append(rec)
print(json.dumps(rec), flush=True)
print(json.dumps(out))
if out_path:
    os.makedirs(os.path.dirname(out_path) or ".", exist_ok=True)
    with open(out_path, "w") as f:
        json.dump(out, f, indent=1)
