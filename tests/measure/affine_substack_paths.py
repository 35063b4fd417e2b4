"""[ActNormFlow, Glow] x 3 in 2-D (a stack without conditioner nets) on the calls the streaming affine kernel does not take:
intermediates requested (2^20 and 2^24 rows) and an odd row count (2^20 + 1 rows, no intermediates), both directions.
Prints one JSON line: per case the kernels launched, the time per call (CUDA events, median of 20 after 3 warm-up calls)
and the largest difference to the interpreter and to the fp64 oracle on the first 2^16 rows.  With an output path it
also saves those rows' results, to compare two builds.  Results: profiles/r07_affine_substack_paths.md.
Run on a GPU box:  python tests/measure/affine_substack_paths.py [out.pt]"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path[:0] = [os.path.join(ROOT, "torch-mnf_b200"), ROOT]
import torch

from oracle import flows_cpu
from tests.helpers import load_flow_model, random_flow_sd
from torch_mnf import _lib

torch.set_grad_enabled(False)
specs = [{"type": "ActNormFlow", "dim": 2, "scale": True, "shift": True}, {"type": "Glow", "dim": 2}] * 3
sd = random_flow_sd(specs, seed=5, scale=0.4)
sd64 = {k: (v.double() if v.is_floating_point() else v) for k, v in sd.items()}
prog = load_flow_model(specs, sd, return_intermediates=False)._program()
prog.plan("cuda", 2)  # packs the parameters (Glow assembly) before launches are counted
CHECK = 1 << 16


def median_ms(fn, iters=20):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
    for a, b in evs:
        a.record()
        fn()
        b.record()
    torch.cuda.synchronize()
    return sorted(a.elapsed_time(b) for a, b in evs)[iters // 2]


out, saved = {"gpu": torch.cuda.get_device_name()}, {}
x_all = 2.0 * torch.randn((1 << 24) + 1, 2, device="cuda", generator=torch.Generator(device="cuda").manual_seed(0))
for name, rows, want_inter in (("inter_2^20", 1 << 20, True), ("inter_2^24", 1 << 24, True), ("odd_2^20+1", (1 << 20) + 1, False)):
    x = x_all[:rows]
    y, ld = torch.empty_like(x), torch.empty(rows, device="cuda")
    for inverse in (True, False):
        call = lambda: prog.run(x, inverse, want_inter=want_inter, out=y, log_det=ld)
        _lib.launch_stats(reset=True)
        call()
        torch.cuda.synchronize()
        sites = _lib.launch_stats()
        ms = median_ms(call)
        _, _, inter, _ = prog.run(x, inverse, want_inter=want_inter, out=y, log_det=ld)
        yg, ldg, _, _ = prog.run(x[:CHECK].contiguous(), inverse, kernel="generic")
        ref, ref_ld = flows_cpu.stack(sd64, specs, x[:CHECK].cpu().double(), inverse=inverse)
        key = f"{name}/{'inv' if inverse else 'fwd'}"
        out[key] = {"rows": rows, "sites": sites, "ms": ms, "gpts_s": rows / ms / 1e6,
                    "max_diff_vs_generic": float(torch.maximum((y[:CHECK] - yg).abs().max(), (ld[:CHECK] - ldg).abs().max())),
                    "max_diff_vs_fp64": float(max((y[:CHECK].cpu().double() - ref[-1]).abs().max(),
                                                  (ld[:CHECK].cpu().double() - ref_ld).abs().max()))}
        saved[key] = (y[:CHECK].cpu(), ld[:CHECK].cpu(), inter[:, :CHECK].cpu() if inter is not None else None)
        print(json.dumps({key: out[key]}), file=sys.stderr, flush=True)
        del inter
print(json.dumps(out))
if len(sys.argv) > 1:
    torch.save(saved, sys.argv[1])
