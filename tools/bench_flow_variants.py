"""Times the flow-stack kernel variants on the BASELINE shapes (scratch tool for tuning)."""
import os, sys, json
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "torch-mnf_b200"), ROOT]
import torch

torch.set_grad_enabled(False)  # inference kernels; training goes through mnf_flow_stack_backward
from tests.helpers import load_flow_model, random_flow_sd
from tests.test_flows_gpu import ORACLE_CASES


def time_prog(prog, x, inverse, kernel, iters=5):
    y = torch.empty_like(x); ld = torch.empty(x.size(0), device=x.device)
    for _ in range(2):
        prog.run(x, inverse, out=y, log_det=ld, kernel=kernel)
    torch.cuda.synchronize()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
    for a, b in evs:
        a.record(); prog.run(x, inverse, out=y, log_det=ld, kernel=kernel); b.record()
    torch.cuda.synchronize()
    ts = sorted(a.elapsed_time(b) for a, b in evs)
    return ts[0], ts[len(ts) // 2]


def main():
    n = int(os.environ.get("N", 1 << 24))
    out = {}
    for name in ("cfg2_shape", "cfg1_shape"):
        specs = ORACLE_CASES[name]
        model = load_flow_model(specs, random_flow_sd(specs, seed=0, scale=0.6 if name == "cfg2_shape" else 0.3),
                                return_intermediates=False)
        g = torch.Generator(device="cuda").manual_seed(0)
        x = 1.5 * torch.randn(n, 2, device="cuda", generator=g)
        prog = model._program()
        for kernel in (6, "generic"):
            xs = x if kernel != "generic" else x[: n // 16].contiguous()
            for inverse in (True, False):
                best, med = time_prog(prog, xs, inverse, kernel)
                key = f"{name}/{kernel}/{'inv' if inverse else 'fwd'}"
                out[key] = {"ms_best": best, "ms_med": med, "gpts_s": xs.size(0) / best / 1e6}
                print(key, out[key], flush=True)
    if name == "cfg1_shape":
        x4 = x[:4096].contiguous()
        for kernel in (6,):
            best, med = time_prog(prog, x4, True, kernel, iters=20)
            print("cfg1 B=4096", kernel, "us best", best * 1e3, "med", med * 1e3)
    os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
    json.dump(out, open(os.path.join(ROOT, "gpurun_out", "flow_variants.json"), "w"), indent=1)


if __name__ == "__main__":
    main()
