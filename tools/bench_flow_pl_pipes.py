"""Where the time of the table kernel goes: ablation builds of flow_pl_kernel timed against the product build.

    python tools/bench_flow_pl_pipes.py --build                      # variant libraries, next to the product one
    python tools/bench_flow_pl_pipes.py --run [--rounds 3] [--out F] [--lib NAME=PATH ...]

--build compiles the library once per variant of VARIANTS with its own object directory and .so suffix
(torch-mnf_b200/build.py, MNF_LIB_SUFFIX / MNF_NVCC_FLAGS).  The ablations (MNF_FPL_ABLATE in csrc/flow_pl.cu) remove
one part of the spline conditioner: their outputs are wrong by construction and only their time means something.
--run times the BASELINE config-2 log-prob step (bench.py's model and 2^24 points, one flow_pl_kernel<8, true> launch)
with each library in a process of its own, the variants alternating within every round, and prints one JSON line per
run and a summary with the card, its power limit and the SM clock read after each run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIBDIR = os.path.join(ROOT, "torch-mnf_b200", "lib")

# name -> extra nvcc flags; "product" is the library build() makes
VARIANTS = {
    "product": "",
    "no_xu_ex2": "-DMNF_FPL_ABLATE=1",     # every ex2 an FMUL
    "fixed_bin": "-DMNF_FPL_ABLATE=2",     # no bin selection
    "const_deriv": "-DMNF_FPL_ABLATE=3",   # no knot derivatives
}


def lib_path(name: str) -> str:
    return os.path.join(LIBDIR, "libmnf_b200.so" if name == "product" else f"libmnf_b200_{name}.so")


def build_all() -> None:
    for name, flags in VARIANTS.items():
        env = dict(os.environ, MNF_LIB_SUFFIX="" if name == "product" else f"_{name}", MNF_NVCC_FLAGS=flags)
        subprocess.run([sys.executable, os.path.join(ROOT, "torch-mnf_b200", "build.py")], env=env, check=True)
        print(name, lib_path(name), flush=True)


def gpu_state() -> dict:
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    vals = [v.strip() for v in r.stdout.splitlines()[0].split(",")] if r.returncode == 0 and r.stdout else []
    return dict(zip(q.split(","), vals))


def time_one(steps: int, warmup: int) -> None:
    """(child) kernel time of the config-2 step with the library MNF_B200_LIB names"""
    sys.path[:0] = [os.path.join(ROOT, "torch-mnf_b200"), ROOT]
    import torch

    torch.set_grad_enabled(False)
    import bench

    dev = torch.device("cuda:0")
    model = bench.build_model(dev)
    x = bench.make_points(1 << 24).to(dev)
    out = torch.empty(x.size(0), device=dev)
    for _ in range(warmup):
        model.log_prob(x, out=out)
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for a, b in ev:
        a.record()
        model.log_prob(x, out=out)
        b.record()
    torch.cuda.synchronize()
    ts = sorted(a.elapsed_time(b) for a, b in ev)
    print(json.dumps({"kernel_ms_mean": sum(ts) / len(ts), "kernel_ms_median": ts[len(ts) // 2]}))


def run_all(rounds: int, libs: dict, steps: int, out_path: str | None) -> None:
    res = {name: [] for name in libs}
    for r in range(rounds):
        for name, path in libs.items():
            env = dict(os.environ, MNF_B200_LIB=path)
            p = subprocess.run([sys.executable, os.path.abspath(__file__), "--time-one", "--steps", str(steps)], env=env,
                               capture_output=True, text=True)
            if p.returncode != 0:
                raise RuntimeError(f"{name}: {p.stdout}\n{p.stderr}")
            t = json.loads(p.stdout.strip().splitlines()[-1])
            t.update(gpu_state(), variant=name, round=r)
            res[name].append(t)
            print(json.dumps(t), flush=True)
    summary = {name: {"kernel_ms_mean": [t["kernel_ms_mean"] for t in ts], "min": min(t["kernel_ms_mean"] for t in ts),
                      "max": max(t["kernel_ms_mean"] for t in ts)} for name, ts in res.items()}
    summary["gpu"] = gpu_state()
    print(json.dumps(summary, indent=1))
    if out_path:
        os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
        with open(out_path, "w") as f:
            json.dump({"runs": res, "summary": summary}, f, indent=1)


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--build", action="store_true")
    ap.add_argument("--run", action="store_true")
    ap.add_argument("--time-one", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--lib", action="append", default=[], metavar="NAME=PATH", help="a further library to time (e.g. a parent build)")
    ap.add_argument("--only", default=None, help="comma-separated variant names to time (default: all)")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if a.time_one:
        return time_one(a.steps, warmup=5)
    if a.build:
        build_all()
    if a.run:
        names = a.only.split(",") if a.only else list(VARIANTS)
        libs = {n: lib_path(n) for n in names}
        for spec in a.lib:
            n, p = spec.split("=", 1)
            libs[n] = p
        run_all(a.rounds, libs, a.steps, a.out)


if __name__ == "__main__":
    main()
