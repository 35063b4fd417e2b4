"""Timing of MNFConv2d with padding and stride, against the same arithmetic in fp32 torch eager on the same GPU:
  forward, inference (Philox noise), B = 256 images of 64 x 32 x 32:
    (a) MNFConv2d(64, 64, 3, padding=1)            implicit GEMM with bounds-tested tap loads (mnf_conv2d_forward_ps)
    (b) the same layer, stride 2                   16 x 16 output
    (c) MNFConv2d(64, 64, 3) on 34 x 34 inputs      the unpadded kernel at the same 32 x 32 output (cost of the bounds tests)
    (d) torch eager: F.conv2d(x, W_mean * z, padding=1) and F.conv2d(x^2, exp(W_log_var), exp(b_log_var), padding=1),
        then mean + sqrt(var) * randn, cuDNN in fp32 (TF32 off, the arithmetic of (a))
    (e) (d) with cuDNN's TF32 convolutions allowed (torch's default for convolutions)
  training, batch 128 of 64 x 32 x 32:
    (f) one step of MNFConv2d(64, 64, 3, padding=1): forward, kl_div, backward of mean(out^2) + kl / N, Adam
    (g) torch eager forward + backward of the conv arithmetic of (d) alone (no z flows, no kl_div), fp32
The forward's moments are compared with (d)'s in fp64 at the timed size.  CUDA events around 5 calls per round, the
variants of a group alternated round by round, median of the rounds.  Card name, power limit and SM clocks are read in
the same run.  Run on a GPU box:
    python tests/measure/mnf_conv_geometry_timing.py [rounds]"""
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path[:0] = [os.path.join(ROOT, "torch-mnf_b200"), ROOT]
import torch
import torch.nn.functional as F

from torch_mnf.layers import MNFConv2d
from torch_mnf.layers import _mnf_ops as ops

rounds = int(sys.argv[1]) if len(sys.argv) > 1 else 9


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader",
                            "-i", "0"], capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        q = f"nvidia-smi unavailable: {e}"
    return q


def time_group(variants, reps=5):
    for fn in variants.values():
        for _ in range(3):
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


def eager_forward(layer, x, z, pad, stride):
    mean = F.conv2d(x, layer.W_mean * z.view(-1, 1, 1, 1), padding=pad, stride=stride)
    var = F.conv2d(x * x, layer.W_log_var.exp(), layer.b_log_var.exp(), padding=pad, stride=stride)
    return mean + var.sqrt() * torch.randn_like(var)


out = {"rounds": rounds, "gpu_torch": torch.cuda.get_device_name(0), "gpu_before": gpu_info()}
dev = torch.device("cuda", 0)
B, C, HW = 256, 64, 32
fan_in_flops = 2 * 2 * C * 9  # two moments, one FMA (2 flops) per tap and channel

# ---- forward ----------------------------------------------------------------------------------------------------------
torch.manual_seed(0)
with torch.no_grad():
    same = MNFConv2d(C, C, 3, padding=1).to(dev)
    strided = MNFConv2d(C, C, 3, padding=1, stride=2).to(dev)
    strided.load_state_dict(same.state_dict())
    plain = MNFConv2d(C, C, 3).to(dev)
    plain.load_state_dict(same.state_dict())
    x = torch.rand(B, C, HW, HW, device=dev)
    x34 = torch.rand(B, C, HW + 2, HW + 2, device=dev)
    z, _ = same.sample_z(ops.Noise(None, dev, seed=3))
    z = z.reshape(-1).contiguous()

    def fwd(layer, xx):
        return lambda: layer(xx, noise=ops.Noise(None, dev, seed=1))

    torch.backends.cudnn.allow_tf32 = False
    rec = time_group({"a_same_3x3": fwd(same, x), "b_stride2": fwd(strided, x), "c_unpadded_34x34": fwd(plain, x34),
                      "d_eager_fp32": lambda: eager_forward(same, x, z, 1, 1)})
    torch.backends.cudnn.allow_tf32 = True
    rec.update(time_group({"e_eager_tf32_allowed": lambda: eager_forward(same, x, z, 1, 1)}))
    torch.backends.cudnn.allow_tf32 = False
    flops = B * C * HW * HW * fan_in_flops
    rec["a_tflops"] = flops / rec["a_same_3x3_ms_median"] / 1e9
    rec["a_over_d"] = rec["a_same_3x3_ms_median"] / rec["d_eager_fp32_ms_median"]
    rec["a_over_c"] = rec["a_same_3x3_ms_median"] / rec["c_unpadded_34x34_ms_median"]
    # moments against fp64 at the timed size (first 32 images)
    mean, sd = ops.conv_moments(same, x[:32], z)
    x64 = x[:32].double()
    ref_m = F.conv2d(x64, same.W_mean.double() * z.double().view(-1, 1, 1, 1), padding=1)
    ref_s = F.conv2d(x64 * x64, same.W_log_var.double().exp(), same.b_log_var.double().exp(), padding=1).sqrt()
    rec["moments_max_rel_err_mean"] = float(((mean.double() - ref_m).abs() / ref_m.abs().mean()).max())
    rec["moments_max_rel_err_sd"] = float(((sd.double() - ref_s).abs() / ref_s.abs().mean()).max())
out["forward"] = {"B": B, "C": C, "HW": HW, "flops_per_call": flops, **rec}
del x34
torch.cuda.empty_cache()

# ---- training ---------------------------------------------------------------------------------------------------------
Bt = 128
torch.manual_seed(1)
layer = MNFConv2d(C, C, 3, padding=1).to(dev)
adam = torch.optim.Adam(layer.parameters(), lr=1e-4)
xt = torch.rand(Bt, C, HW, HW, device=dev)


def mnf_step():
    adam.zero_grad()
    y = layer(xt)
    loss = y.square().mean() + layer.kl_div() / Bt
    loss.backward()
    adam.step()


Wm = layer.W_mean.detach().clone().requires_grad_()
Wlv = layer.W_log_var.detach().clone().requires_grad_()
blv = layer.b_log_var.detach().clone().requires_grad_()
zt = z.detach().clone().requires_grad_()


def eager_step():
    mean = F.conv2d(xt, Wm * zt.view(-1, 1, 1, 1), padding=1)
    var = F.conv2d(xt * xt, Wlv.exp(), blv.exp(), padding=1)
    (mean + var.sqrt() * torch.randn_like(var)).square().mean().backward()


rec = time_group({"f_mnf_training_step": mnf_step, "g_eager_conv_fwd_bwd": eager_step}, reps=3)
out["training"] = {"B": Bt, "C": C, "HW": HW, **rec}
out["gpu"] = gpu_info()
print(json.dumps(out))
