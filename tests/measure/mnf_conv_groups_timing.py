"""Timing of MNFConv2d with channel groups and dilation, each against the same arithmetic in fp32 torch eager on the same
GPU (two F.conv2d with the layer's geometry, cuDNN with TF32 off, then sqrt and randn_like).  Inference, Philox noise:
  (a) depthwise 3x3, MNFConv2d(128, 128, 3, padding=1, groups=128) on 256 x 128 x 32 x 32 (134 MB in, 134 MB out,
      larger than L2; the data-sheet HBM floor for one read and one write is ~35 us)      -> grouped direct kernel
  (b) pointwise 1x1, MNFConv2d(128, 128, 1) on the same input                           -> default implicit GEMM
  (c) MNFConv2d(64, 64, 3, padding=1, groups=8) on 256 x 64 x 32 x 32, 8 channels a group -> grouped direct kernel
  (d) MNFConv2d(64, 64, 3, padding=1, groups=16) on the same input, 4 channels a group   -> grouped direct kernel
  (e) dilated 3x3, MNFConv2d(64, 64, 3, padding=2, dilation=2) on the same input          -> bounds-tested implicit GEMM
  (h) MNFConv2d(64, 64, 3, padding=1, groups=4) on the same input, 16 channels a group   -> grouped implicit GEMM
(c) and (h) sit on the two sides of the library's choice between the direct kernel and the grouped GEMM.
Where the depthwise forward (a) spends its time, same input, alternated:
  (a)          the forward with Philox noise
  (a_eps)      the forward reading an injected eps tensor instead of generating Philox normals (one more 134 MB read)
  (a_moments)  conv_moments: both moments, no noise, two outputs written (one more 134 MB write)
  (copy)       torch's device copy of the input into an output of the same size: the measured floor for one read and
               one write of these bytes
Training, batch 128 of 128 x 32 x 32:
  (f) one step of a depthwise-separable block (the layers of (a) and (b)): forward, kl_div of both layers, backward of
      mean(out^2) + kl / N, Adam
  (g) torch eager forward + backward of the block's conv arithmetic alone (no z flows, no kl_div, no Adam), fp32
Each forward's moments are compared with fp64 F.conv2d at the timed shape on 16 images.  CUDA events around 5 calls
per round (3 for training), the MNF variant and its eager counterpart alternated round by round, median of the rounds.
Card name, power limit and SM clocks are read in the same run.  Run on a GPU box:
    python tests/measure/mnf_conv_groups_timing.py [rounds]"""
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


def geom(layer):
    return dict(padding=layer.padding, stride=layer.stride, dilation=layer.dilation, groups=layer.groups)


def eager_forward(layer, x, z):
    mean = F.conv2d(x, layer.W_mean * z.view(-1, 1, 1, 1), **geom(layer))
    var = F.conv2d(x * x, layer.W_log_var.exp(), layer.b_log_var.exp(), **geom(layer))
    return mean + var.sqrt() * torch.randn_like(var)


def moments_error(layer, x, z):
    mean, sd = ops.conv_moments(layer, x, z)
    x64 = x.double()
    ref_m = F.conv2d(x64, layer.W_mean.double() * z.double().view(-1, 1, 1, 1), **geom(layer))
    ref_s = F.conv2d(x64 * x64, layer.W_log_var.double().exp(), layer.b_log_var.double().exp(), **geom(layer)).sqrt()
    return (float(((mean.double() - ref_m).abs() / ref_m.abs().mean()).max()),
            float(((sd.double() - ref_s).abs() / ref_s.abs().mean()).max()))


out = {"rounds": rounds, "gpu_torch": torch.cuda.get_device_name(0), "gpu_before": gpu_info()}
dev = torch.device("cuda", 0)
torch.backends.cudnn.allow_tf32 = False
B, HW = 256, 32

forward = {}
with torch.no_grad():
    torch.manual_seed(0)
    x128 = torch.rand(B, 128, HW, HW, device=dev)
    x64 = torch.rand(B, 64, HW, HW, device=dev)
    cases = {  # name: (layer, input, kernel)
        "a_depthwise_3x3": (MNFConv2d(128, 128, 3, padding=1, groups=128), x128, "grouped direct"),
        "b_pointwise_1x1": (MNFConv2d(128, 128, 1), x128, "default implicit GEMM"),
        "c_groups8_64": (MNFConv2d(64, 64, 3, padding=1, groups=8), x64, "grouped direct"),
        "d_groups16_64": (MNFConv2d(64, 64, 3, padding=1, groups=16), x64, "grouped direct"),
        "e_dilated_3x3_d2": (MNFConv2d(64, 64, 3, padding=2, dilation=2), x64, "bounds-tested implicit GEMM"),
        "h_groups4_64": (MNFConv2d(64, 64, 3, padding=1, groups=4), x64, "grouped implicit GEMM"),
    }
    for name, (layer, x, kernel) in cases.items():
        layer.to(dev)
        z, _ = layer.sample_z(ops.Noise(None, dev, seed=3))
        z = z.reshape(-1).contiguous()
        rec = time_group({"mnf": lambda: layer(x, noise=ops.Noise(None, dev, seed=1)),
                          "eager_fp32": lambda: eager_forward(layer, x, z)})
        c_in, taps = x.size(1) // layer.groups, layer.kernel_size**2
        flops = B * layer.n_out * HW * HW * 2 * 2 * c_in * taps  # two moments, one FMA per tap and input channel
        io_bytes = 4 * (x.numel() + B * layer.n_out * HW * HW)
        err_m, err_s = moments_error(layer, x[:16], z)
        forward[name] = {"layer": layer.extra_repr(), "kernel": kernel, "flops_per_call": flops,
                         "in_out_bytes": io_bytes, **rec,
                         "mnf_over_eager": rec["mnf_ms_median"] / rec["eager_fp32_ms_median"],
                         "mnf_tflops": flops / rec["mnf_ms_median"] / 1e9,
                         "mnf_in_out_tb_per_s": io_bytes / rec["mnf_ms_median"] / 1e9,
                         "moments_max_rel_err_mean": err_m, "moments_max_rel_err_sd": err_s}
        layer.cpu()
    layer = cases["a_depthwise_3x3"][0].to(dev)
    x = x128
    z, _ = layer.sample_z(ops.Noise(None, dev, seed=3))
    z = z.reshape(-1).contiguous()
    eps = torch.randn(B, 128, HW, HW, device=dev)
    dst = torch.empty_like(x)
    rec = time_group({"a": lambda: layer(x, noise=ops.Noise(None, dev, seed=1)),
                      "a_eps": lambda: ops.conv_forward(layer, x, z, ops.Noise(None, dev, seed=1),
                                                        drawn=(eps, 0, 0)),
                      "a_moments": lambda: ops.conv_moments(layer, x, z),
                      "copy": lambda: dst.copy_(x)})
    rec["copy_tb_per_s"] = 2 * 4 * x.numel() / rec["copy_ms_median"] / 1e9
    forward["depthwise_breakdown"] = rec
    del eps, dst
    layer.cpu()
out["forward"] = forward
del x128, x64
torch.cuda.empty_cache()

# ---- training: one depthwise-separable block ------------------------------------------------------------------------
Bt, C = 128, 128
torch.manual_seed(1)
dw = MNFConv2d(C, C, 3, padding=1, groups=C).to(dev)
pw = MNFConv2d(C, C, 1).to(dev)
adam = torch.optim.Adam(list(dw.parameters()) + list(pw.parameters()), lr=1e-4)
xt = torch.rand(Bt, C, HW, HW, device=dev)


def mnf_step():
    adam.zero_grad()
    y = pw(dw(xt).relu())
    loss = y.square().mean() + (dw.kl_div() + pw.kl_div()) / Bt
    loss.backward()
    adam.step()


params = [t.detach().clone().requires_grad_() for t in (dw.W_mean, dw.W_log_var, dw.b_log_var, pw.W_mean,
                                                         pw.W_log_var, pw.b_log_var)]
zs = [torch.rand(C, device=dev).requires_grad_() for _ in range(2)]


def eager_conv(x, Wm, Wlv, blv, z, groups, padding):
    mean = F.conv2d(x, Wm * z.view(-1, 1, 1, 1), padding=padding, groups=groups)
    var = F.conv2d(x * x, Wlv.exp(), blv.exp(), padding=padding, groups=groups)
    return mean + var.sqrt() * torch.randn_like(var)


def eager_step():
    h = eager_conv(xt, *params[:3], zs[0], C, 1).relu()
    eager_conv(h, *params[3:], zs[1], 1, 0).square().mean().backward()


from torch_mnf import _lib  # noqa: E402

with torch.enable_grad():
    l0 = _lib.launch_count
    mnf_step()
    launches = _lib.launch_count - l0
    rec = time_group({"f_mnf_training_step": mnf_step, "g_eager_conv_fwd_bwd": eager_step}, reps=3)
out["training"] = {"B": Bt, "C": C, "HW": HW, "library_launches_per_step": launches, **rec}
out["gpu"] = gpu_info()
print(json.dumps(out))
