#!/usr/bin/env python
"""bench.py -- flow log-prob throughput on the BASELINE.json headline configuration.

Workload ("cfg2"): [ActNormFlow, Glow, NSF_CL(K=8, B=3, n_h=16)] x 3 on synthetic 2-D points
x = 1.5 * randn(2^24, 2) (seed 0), one step = log p(x) for every point of the batch
(inverse pass + log-det + standard-normal base density, the quantity tests/test_flows.py:22-24
of the reference assembles).  One process per GPU; under torchrun each rank owns its own 2^24
points (weak scaling) and the per-point log-probs are all-gathered over NCCL, chunk by chunk,
overlapped with the next chunk's kernel.

    python bench.py --gpus 1 --steps 20 --warmup 3            # our arm
    python bench.py --impl reference --steps 3 --warmup 1      # CPU oracle port on host cores
    python bench.py --steps 20 --dump-outputs DIR              # also DIR/log_prob.npy: the last timed step's log-probs

Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for the meaning of every key.

The headline keys describe config 2.  The same line carries `configs`: BASELINE configs 1, 3, 4, 5 (and config 2 under
strong scaling when N > 1), each measured in this process with its own value / unit / ms / roofline / cpu_baseline /
e2e, so that every named configuration -- and the second named metric, MNF-LeNet MC predictive samples/s -- is
measured by the same run.  `--steps` is the number of timed steps of every timed loop, headline and configurations.
`--workload cfg2` prints the headline alone, `--workload cfg4` the MNF-LeNet line alone.
"""

from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (os.path.join(ROOT, "torch-mnf_b200"), ROOT):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

N_POINTS = 1 << 24
K_BINS, BOUND, N_H = 8, 3, 16
BYTES_PER_POINT = 12  # 8 B point in + 4 B log-prob out (z is not materialised in log-prob mode)
MLP_FMA_PER_POINT = 3 * 2 * (16 + 256 + 256 + 16 * 23)  # 5376 fused multiply-adds in the conditioners
TRAFFIC_FILE = os.path.join(ROOT, "profiles", "ncu_traffic.json")  # written by tools/ncu_traffic.py from an `ncu --set full` capture
METRIC = "flow log-prob points/s"
WORKLOAD = "cfg2: [ActNormFlow, Glow, NSF_CL(K=8,B=3,n_h=16)] x3, 2-D points, batch 2^24 per GPU"
DUMP_MAX_VALUES = 1 << 22  # --dump-outputs: 16 MB of float32 at most, whatever the batch and the number of GPUs


def specs():
    return [
        {"type": "ActNormFlow", "dim": 2, "scale": True, "shift": True},
        {"type": "Glow", "dim": 2},
        {"type": "NSF_CL", "dim": 2, "K": K_BINS, "B": BOUND, "n_h": N_H},
    ] * 3


def make_points(n, seed=0):
    g = torch.Generator().manual_seed(seed)
    return 1.5 * torch.randn(n, 2, generator=g)


def traffic_for(workload, units):
    """DRAM bytes per step of `workload` scaled to `units` work items, from the committed ncu capture summary
    (profiles/ncu_traffic.json: dram__bytes_read.sum + dram__bytes_write.sum summed over the step's launches), or
    None when no capture exists for it."""
    try:
        with open(TRAFFIC_FILE) as f:
            w = json.load(f)["workloads"][workload]
        return float(w["dram_bytes"]) * units / float(w["units"])
    except (OSError, KeyError, ValueError):
        return None


def kernels_of(fn):
    """{launch site: launches} of the library's own tally (mnf_launch_stats) while fn() runs."""
    from torch_mnf import _lib

    _lib.launch_stats(reset=True)
    fn()
    return _lib.launch_stats()


def timed_ms(fn, steps, warmup, dev, world=1):
    """CUDA-event time per step of fn() on the current stream: warm-up, barrier + synchronize on both sides, max over ranks."""
    import torch.distributed as dist

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for _ in range(warmup):
        fn()
    barrier()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        fn()
    b.record()
    barrier()
    ms = a.elapsed_time(b) / steps
    if world > 1:
        tt = torch.tensor([ms], device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms = float(tt)
    return ms


def dump_sample(values, seed=0):
    """`values` (1-D, on the device) on the host: all of them up to DUMP_MAX_VALUES, else one value drawn with a fixed
    seed from each of DUMP_MAX_VALUES equal consecutive blocks.  The indices depend only on the length, so runs with
    the same arguments sample the same points."""
    n = values.numel()
    if n <= DUMP_MAX_VALUES:
        return values.cpu()
    stride = n // DUMP_MAX_VALUES
    g = torch.Generator().manual_seed(seed)
    idx = torch.arange(DUMP_MAX_VALUES) * stride + torch.randint(stride, (DUMP_MAX_VALUES,), generator=g)
    return values[idx.to(values.device)].cpu()


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "MEASURED_PEAKS.json (measured)", d
    return 6650.0, "fallback (B200_PROFILING.md)", {}


class ClockSampler:
    """nvidia-smi sampler running during the timed region (B200_PROFILING.md clocks line)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50",
                 "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        rows = [r for ts, r in self.rows if t0 <= ts <= t1 + 0.06] or [r for _, r in self.rows[-3:]]
        sm = sorted(float(r[1]) for r in rows if r[1].replace(".", "").isdigit())
        mx = max((float(r[2]) for r in rows if r[2].replace(".", "").isdigit()), default=None)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in rows for n, v in zip(names, r[5:9]) if v.lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": reasons,
                "samples": len(rows)}


# ---------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle port on host cores
# ---------------------------------------------------------------------------------------
def cpu_model_state():
    """Weights for the CPU arm: same construction as the CUDA arm (seed 0, ActNorm init on the
    first 4096 points), produced by the oracle alone so the reference arm needs no GPU."""
    from tests.helpers import random_flow_sd

    from oracle import flows_cpu

    sp = specs()
    sd = random_flow_sd(sp, seed=0, scale=0.6)
    x0 = make_points(4096)
    v = x0
    for i in reversed(range(len(sp))):  # data-dependent init in inverse order (core.py:30)
        p = flows_cpu.sub(sd, f"flows.{i}.")
        if sp[i]["type"] == "ActNormFlow":
            s, t = flows_cpu.actnorm_init(p, sp[i], v)
            sd[f"flows.{i}.s"], sd[f"flows.{i}.t"] = s, t
            p = flows_cpu.sub(sd, f"flows.{i}.")
        v, _ = flows_cpu.apply_flow(p, sp[i], v, True)
    return sp, sd


def cpu_time_sample(sp, sd, n, reps=1):
    from oracle import flows_cpu

    x = make_points(n, seed=1)
    best = float("inf")
    with torch.no_grad():
        for _ in range(reps):
            t0 = time.perf_counter()
            flows_cpu.log_prob(sd, sp, x)
            best = min(best, time.perf_counter() - t0)
    return best


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    sp, sd = cpu_model_state()
    probe = cpu_time_sample(sp, sd, 1 << 16)
    budget = 90.0 / max(1, args.steps + args.warmup)
    n = 1 << 16
    while n < (1 << 22) and probe * (2 * n / (1 << 16)) < budget:
        n *= 2
    for _ in range(args.warmup):
        cpu_time_sample(sp, sd, n)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_time_sample(sp, sd, n)
    dt = (time.perf_counter() - t0) / args.steps
    value = n / dt
    sample = f"{n} points per step (2^{n.bit_length() - 1}) of the 2^24-point workload, torch CPU, {cores} threads"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": "points/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "sample": sample},
        "cpu_baseline": {"value": value, "unit": "points/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "points/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ---------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------
def build_model(device):
    from tests.helpers import load_flow_model, random_flow_sd

    sp = specs()
    model = load_flow_model(sp, random_flow_sd(sp, seed=0, scale=0.6), device=device, return_intermediates=False)
    for f in model.flows:  # re-arm the data-dependent init, as a fresh model would have it
        if hasattr(f, "data_dep_init_done"):
            f.data_dep_init_done = False
    model.inverse(make_points(4096).to(device))
    return model


def pin_to_gpu_numa_node(local: int) -> str:
    """Bind this rank's host threads to the cores next to its GPU before any pinned buffer is allocated (first touch
    then places the buffers on that NUMA node): with 8 ranks the host-to-host figure is limited by cross-socket
    traffic otherwise.  Best effort; returns a note for the JSON line."""
    try:
        import pynvml

        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local)
        n_cpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (n_cpu + 63) // 64)
        cpus = {64 * w + b for w, word in enumerate(words) for b in range(64) if (word >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return f"{len(cpus)} cores local to GPU {local}"
    except Exception as e:  # noqa: BLE001
        return f"unchanged ({type(e).__name__})"
    return "unchanged"


def run_ours(args):
    import torch.distributed as dist
    from torch_mnf import _lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback in the product path)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    affinity = pin_to_gpu_numa_node(local) if world > 1 else "unchanged (single rank)"
    if world > 1 and not dist.is_initialized():
        dist.init_process_group("nccl", device_id=dev)
    model = build_model(dev)
    n = args.points
    chunks = args.chunks if world > 1 else 1
    assert n % (2 * chunks) == 0
    cn = n // chunks
    x_host = make_points(n, seed=100 + rank).pin_memory()
    x = x_host.to(dev, non_blocking=True)
    # Result gather.  Preferred: NVLink peer memory -- the kernel stores each log-prob into every rank's gather
    # buffer while it computes (torch_mnf.distributed.PeerGather: NVLS multicast or per-peer stores), so the step
    # has no data-moving collective, only barriers.  Fallback (--gather nccl, or no symmetric memory): chunked
    # NCCL all-gather on a side stream; the kernel writes this rank's slice of the gather buffer directly.
    peer = None
    if world > 1 and args.gather == "peer":
        try:
            from torch_mnf.distributed import PeerGather

            peer = PeerGather(n, dev)
        except Exception as e:  # noqa: BLE001
            if rank == 0:
                print(f"[bench] peer-memory gather unavailable ({type(e).__name__}: {e}); using NCCL all-gather", file=sys.stderr)
            peer = None
    if peer is not None:
        chunks = 1
        cn = n
        gathered = peer.buffer.view(1, world, n)
        gather_out = peer.gather_out(use_multicast=not args.no_multicast)
    else:
        gathered = torch.empty((chunks, world, cn), device=dev, dtype=torch.float32)
        gather_out = None
    comm = torch.cuda.Stream(device=dev) if (world > 1 and peer is None) else None

    def step():
        cur = torch.cuda.current_stream(dev)
        if peer is not None:
            peer.barrier()  # peers are done reading the previous step's results
            model.log_prob(x, out=gathered[0, rank], gather=gather_out)
            peer.barrier()  # every rank's stores have landed everywhere
            return
        for c in range(chunks):
            model.log_prob(x[c * cn:(c + 1) * cn], out=gathered[c, rank])
            if world > 1:
                comm.wait_stream(cur)
                with torch.cuda.stream(comm):
                    dist.all_gather_into_tensor(gathered[c].view(-1), gathered[c, rank])
        if world > 1:
            cur.wait_stream(comm)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.15)
    barrier()
    launches0 = _lib.lib().mnf_launch_count()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    t_wall0 = time.time()
    ev[0].record()
    for i in range(args.steps):
        step()
        ev[i + 1].record()
    barrier()
    t_wall1 = time.time()
    launches = _lib.lib().mnf_launch_count() - launches0  # kernels launched by libmnf_b200.so in the timed region
    total_ms = ev[0].elapsed_time(ev[-1])
    if world > 1:
        tmax = torch.tensor([total_ms], device=dev)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        total_ms = float(tmax)
    clocks = sampler.stop(t_wall0, t_wall1) if rank == 0 else None
    gather_ok = True
    if world > 1:
        # every rank must now hold every rank's log-probs: compare a checksum per slice with an all-gather of the
        # owners' checksums
        mine = gathered.view(-1, world, cn)[:, rank].double().sum().reshape(1)
        sums = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(sums, mine)
        seen = torch.stack([gathered.view(-1, world, cn)[:, r].double().sum() for r in range(world)])
        gather_ok = bool(torch.allclose(seen, torch.cat(sums), rtol=1e-9, atol=1e-6))
    if args.dump_outputs and rank == 0:
        # what the last timed step handed its caller: every rank's log-probs, in rank order (before later legs reuse the buffer)
        import numpy as np

        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "log_prob.npy"), dump_sample(gathered.transpose(0, 1).reshape(-1)).numpy())
    ms_per_step = total_ms / args.steps
    value = world * n / (ms_per_step * 1e-3)

    # ---- kernel-only duration (same launches, no collective) for the roofline ----
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    _lib.launch_stats(reset=True)
    for a, b in kev:
        a.record()
        model.log_prob(x, out=gathered.view(-1)[:n])
        b.record()
    torch.cuda.synchronize(dev)
    k_sites = {k: v // len(kev) for k, v in _lib.launch_stats().items()}  # launch sites per step, from the library's tally
    k_ms = sum(a.elapsed_time(b) for a, b in kev) / len(kev)
    # the module call keeps the conditioner tables of the table kernel per parameter version (like the packed parameter
    # blob); the same step with the tables rebuilt from the weights inside EVERY call (explicit variant: no staging):
    k_ms_rebuild = None
    if any("flow_pl" in k for k in k_sites):
        prog, buf = model._program(), gathered.view(-1)[:n]
        for _ in range(2):
            prog.run(x, True, log_prob_only=True, kernel=6, log_prob_out=buf)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(args.steps):
            prog.run(x, True, log_prob_only=True, kernel=6, log_prob_out=buf)
        b.record()
        torch.cuda.synchronize(dev)
        k_ms_rebuild = a.elapsed_time(b) / args.steps

    # ---- end to end through the module API with HOST buffers (pinned), copies inside ----
    out_host = torch.empty(n, dtype=torch.float32).pin_memory()
    e_chunks = args.e2e_chunks
    ecn = n // e_chunks
    s_in, s_out = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
    xd = [torch.empty((ecn, 2), device=dev) for _ in range(2)]
    od = [torch.empty(ecn, device=dev) for _ in range(2)]

    # chunk buffers are double-buffered ACROSS steps too: the first copy-in of step k+1 overlaps the last kernels and
    # copy-outs of step k (every step still moves all of its input H2D and all of its output D2H inside the timed region)
    ready = [None, None]  # copy-out of the chunk that last used od[b] has finished
    freed = [None, None]  # kernel that last read xd[b] has finished

    def e2e_step():
        cur = torch.cuda.current_stream(dev)
        for c in range(e_chunks):
            b = c & 1
            with torch.cuda.stream(s_in):
                if freed[b] is not None:
                    s_in.wait_event(freed[b])
                xd[b].copy_(x_host[c * ecn:(c + 1) * ecn], non_blocking=True)
                e_in = torch.cuda.Event()
                e_in.record(s_in)
            cur.wait_event(e_in)
            if ready[b] is not None:
                cur.wait_event(ready[b])
            model.log_prob(xd[b], out=od[b])
            e_k = torch.cuda.Event()
            e_k.record(cur)
            freed[b] = e_k
            with torch.cuda.stream(s_out):
                s_out.wait_event(e_k)
                out_host[c * ecn:(c + 1) * ecn].copy_(od[b], non_blocking=True)
                e_o = torch.cuda.Event()
                e_o.record(s_out)
            ready[b] = e_o

    def e2e_join():
        cur = torch.cuda.current_stream(dev)
        cur.wait_stream(s_out)
        cur.wait_stream(s_in)

    for _ in range(2):
        e2e_step()
    e2e_join()
    barrier()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(args.steps):
        e2e_step()
    e2e_join()
    b.record()
    barrier()
    e_ms = a.elapsed_time(b) / args.steps
    if world > 1:
        tmax = torch.tensor([e_ms], device=dev)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        e_ms = float(tmax)
    e2e_value = world * n / (e_ms * 1e-3)
    # sanity: the e2e path produced finite log-probs equal to the resident path
    chk = torch.allclose(out_host[:4096], gathered.view(-1)[:4096].cpu(), rtol=1e-6, atol=1e-6) if chunks == 1 else True

    # ---- the same copies with NO kernel: the ceiling PCIe / the host side puts on the end-to-end figure ----
    def copies_only():
        for c in range(e_chunks):
            b = c & 1
            with torch.cuda.stream(s_in):
                xd[b].copy_(x_host[c * ecn:(c + 1) * ecn], non_blocking=True)
            with torch.cuda.stream(s_out):
                out_host[c * ecn:(c + 1) * ecn].copy_(od[b], non_blocking=True)

    copies_only()
    e2e_join()
    barrier()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    s_in.wait_stream(torch.cuda.current_stream(dev))
    s_out.wait_stream(torch.cuda.current_stream(dev))
    for _ in range(args.steps):
        copies_only()
    e2e_join()
    b.record()
    barrier()
    c_ms = a.elapsed_time(b) / args.steps
    if world > 1:
        tmax = torch.tensor([c_ms], device=dev)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        c_ms = float(tmax)

    del xd, od, out_host
    if rank != 0:
        return None

    hbm_peak, peak_src, _ = peaks()
    achieved = BYTES_PER_POINT * n / (k_ms * 1e-3) / 1e9
    sm_clock = (clocks or {}).get("sm_mhz") or 1965.0
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    fp32_peak = sms * 128 * 2 * sm_clock * 1e6 / 1e12
    mlp_tflops = 2 * MLP_FMA_PER_POINT * n / (k_ms * 1e-3) / 1e12
    out = {
        "metric": METRIC, "value": value, "unit": "points/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "points_per_gpu": n, "l2": "inputs (134 MB/GPU) larger than the 126 MB L2",
                   "collective": ("none (N=1)" if world == 1 else
                                  ("fused in the kernel: log-probs stored to every rank over NVLink peer memory ("
                                   + ("NVLS multicast multimem.st" if gather_out.multicast_ptr else "per-peer st.global")
                                   + "), 2 barriers per step") if peer is not None else
                                  f"NCCL all_gather of log-probs in {chunks} chunks overlapped with compute"), "parallelism": f"points sharded over {world} GPU(s), weights replicated"},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "points/s", "h2d_bytes_per_step": 8 * n, "d2h_bytes_per_step": 4 * n,
                "ms_per_step": e_ms, "matches_resident_path": bool(chk), "host_affinity": affinity,
                "copy_only_ceiling": {"value": world * n / (c_ms * 1e-3), "unit": "points/s", "ms_per_step": c_ms,
                                      "frac_of_ceiling": c_ms / e_ms,
                                      "note": "the same pinned-memory H2D + D2H copies per step on the same streams with NO kernel in between"},
                "how": f"pinned host -> {e_chunks} chunks double-buffered over 3 streams (pipelined across steps) -> NormalizingFlowModel.log_prob -> pinned host"},
        "gpu_launches": launches, "gather_verified": gather_ok,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                     "frac": achieved / hbm_peak, "traffic": traffic_for("cfg2", n),
                     "kernel": k_sites,
                     "kernel_ms": k_ms, "kernel_ms_tables_rebuilt_every_step": k_ms_rebuild,
                     "bytes_per_point": BYTES_PER_POINT, "peak_source": peak_src,
                     "note": ("ONE launch per step (flow_pl_kernel): every conditioner MLP is a piecewise-linear function of "
                              "its scalar input, evaluated as a binary search over its breakpoints in shared memory and one FMA per "
                              "output; the tables are built from the weights in fp64 once per parameter version (cached with the packed "
                              "parameter blob, checked every call) -- kernel_ms_tables_rebuilt_every_step is the same step with the "
                              "builder inside every call; DRAM traffic is the algorithmic "
                              "12 B/pt. The kernel is instruction-issue / MUFU bound on the spline arithmetic, not HBM bound: "
                              "profiles/r02_flow_pl.md"
                              if any("flow_pl" in k for k in k_sites) else
                              "one launch per step (flow_tc16_kernel): conditioner MLPs on tcgen05 as fp16-split 3-term products, "
                              "weights resident in shared memory, points in registers; DRAM traffic is the algorithmic 12 B/pt. "
                              "The kernel is instruction-issue bound (spline arithmetic + operand splitting), not HBM bound: "
                              "profiles/r02_flow_tc.md"
                              if any("flow_tc" in k for k in k_sites) else
                              "per STEP (6 segment launches): algorithmic 12 B/pt; the segmented stack moves ~113 B/pt "
                              "(ncu, profiles/r01_flow_cbank_ncu_full.md); kernel is fp32-FMA-pipe bound, not HBM "
                              "bound (DESIGN.md): see fma_pipe")},
        "fma_pipe": {"mlp_tflops": mlp_tflops, "fp32_peak_tflops_at_sampled_clock": fp32_peak,
                     "frac_mlp_only": mlp_tflops / fp32_peak, "fma_per_point_mlp": MLP_FMA_PER_POINT,
                     "note": ("the conditioner MLPs' NOMINAL multiply-adds per second (layer-by-layer count) against the fp32 FMA peak; "
                              "the table kernel does not execute them (one FMA per output per point), so this can exceed 1"
                              if any("flow_pl" in k for k in k_sites) else
                              "conditioner-MLP multiply-adds per second against the fp32 FMA peak, for comparison with the FFMA2 "
                              "kernel of round 1 (this kernel runs them on the tensor pipe)"
                              if any("flow_tc" in k for k in k_sites) else
                              "conditioner-MLP FMAs only; spline arithmetic shares the same pipe")},
    }
    if any("flow_pl" in k for k in k_sites):
        # what the table kernel is really bound by: the special-function (XU / MUFU) pipe next to the issue slots
        mufu_pt = 6 * 45  # per conditioner + spline: 32 EX2 (two softmaxes per axis), 4 RCP, 2 x (EX2 + LG2) softplus, 3 RCP, SQRT, LG2
        xu_peak = sms * 16 * sm_clock * 1e6 / 1e9  # 16 MUFU lanes per SM and clock
        out["xu_pipe"] = {"mufu_per_point": mufu_pt, "achieved": mufu_pt * n / (k_ms * 1e-3) / 1e9, "peak": xu_peak, "unit": "G MUFU/s",
                          "frac": mufu_pt * n / (k_ms * 1e-3) / 1e9 / xu_peak,
                          "note": "nominal count (a point outside [-B, B] skips the spline); ncu of the same kernel: XU pipe 71 %, issue "
                                  "slots 82 % (profiles/r02_flow_pl_ncu_full.md) -- the kernel is bound by the reference's spline "
                                  "parameterisation on these two pipes, not by HBM"}
    if world == 1:
        # The conditioner-free part of the same stack ([ActNormFlow, Glow] x 3) is the flow workload that IS HBM-bound:
        # reported next to the headline so that the HBM roofline of the streaming path can be read off this line too.
        try:
            from tests.helpers import load_flow_model, random_flow_sd

            sub_specs = [s_ for s_ in specs() if s_["type"] != "NSF_CL"]
            sub = load_flow_model(sub_specs, random_flow_sd(sub_specs, seed=0), device=dev, return_intermediates=False)
            ys, lds = torch.empty_like(x), torch.empty(n, device=dev)
            prog = sub._program()
            for _ in range(3):
                prog.run(x, True, out=ys, log_det=lds)
            a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a_.record()
            for _ in range(args.steps):
                prog.run(x, True, out=ys, log_det=lds)
            b_.record()
            torch.cuda.synchronize(dev)
            sub_ms = a_.elapsed_time(b_) / args.steps
            out["hbm_bound_substack"] = {
                "workload": "[ActNormFlow, Glow] x3 (the conditioner-free flows of the headline stack), inverse with z and log_det stored",
                "bytes_per_point": 20, "ms": sub_ms, "achieved": 20 * n / (sub_ms * 1e-3) / 1e9, "peak": hbm_peak,
                "unit": "GB/s", "frac": 20 * n / (sub_ms * 1e-3) / 1e9 / hbm_peak, "kernel": "affine_stream_kernel"}
            del ys, lds, sub
        except Exception as e:  # noqa: BLE001  (diagnostic extra, never fails the bench)
            out["hbm_bound_substack"] = {"error": f"{type(e).__name__}: {e}"}
    if world == 1 and not args.no_cpu:
        cores = os.cpu_count() or 1
        torch.set_num_threads(cores)
        sp, sd = cpu_model_state()
        probe = cpu_time_sample(sp, sd, 1 << 16)
        ncpu = 1 << 16
        while ncpu < (1 << 22) and probe * (2 * ncpu / (1 << 16)) < 8.0:
            ncpu *= 2
        t = cpu_time_sample(sp, sd, ncpu, reps=2)
        out["cpu_baseline"] = {"value": ncpu / t, "unit": "points/s", "cores": cores, "kind": "port",
                               "sample": f"{ncpu} points (2^{ncpu.bit_length() - 1}), best of 2, torch CPU oracle port, {cores} threads"}
    else:
        out["cpu_baseline"] = None
    return out


# ---------------------------------------------------------------------------------------
# the other BASELINE configurations (attached to the headline line as `configs`)
# ---------------------------------------------------------------------------------------
def _tf32_peak():
    """TF32 dense peak = half the measured bf16 peak (MEASURED_PEAKS.json sustained figure: these kernels are timed
    inside a long step)."""
    d = peaks()[2]
    return float(d.get("bf16_tflops_sustained", 1400.0)) / 2, ("MEASURED_PEAKS.json bf16_tflops_sustained / 2" if d else "fallback 1400 / 2")


def cfg_strong(args, dev, world, rank, model):
    """Config 2 as BASELINE words it: ONE batch of 2^24 points sharded over the N GPUs (strong scaling), log-probs
    gathered on every rank through the fused peer-memory stores."""
    import torch.distributed as dist
    from torch_mnf.distributed import PeerGather

    n_tot = N_POINTS
    n = n_tot // world
    x = make_points(n, seed=300 + rank).to(dev)
    try:
        peer = PeerGather(n, dev)
        gather_out = peer.gather_out(use_multicast=not args.no_multicast)
        how = "fused peer-memory stores (" + ("NVLS multicast" if gather_out.multicast_ptr else "per-peer st.global") + "), 2 barriers"

        def step():
            peer.barrier()
            model.log_prob(x, out=peer.local_slice(), gather=gather_out)
            peer.barrier()
    except Exception as e:  # noqa: BLE001
        buf = torch.empty(world * n, device=dev)
        how = f"NCCL all_gather ({type(e).__name__}: no peer memory)"

        def step():
            model.log_prob(x, out=buf[rank * n:(rank + 1) * n])
            dist.all_gather_into_tensor(buf, buf[rank * n:(rank + 1) * n])
    ms = timed_ms(step, args.steps, 3, dev, world)
    return {"metric": METRIC, "value": n_tot / (ms * 1e-3), "unit": "points/s", "ms_per_step": ms, "scaling": "strong",
            "n_gpus": world, "steps": args.steps, "warmup": 3,
            "config": {"workload": f"cfg2 stack, ONE batch of 2^24 points sharded over {world} GPUs ({n} points each)",
                       "collective": how, "l2": f"{8 * n / 1e6:.0f} MB of points per GPU per step"
                       + ("" if 8 * n > 126e6 else " (fits the 126 MB L2: steps re-read the same resident shard)")}}


def cfg1(args, dev):
    """BASELINE config 1: RNVP x9 (AffineHalfFlow) on 2-D half-moons, batch 4096, log_prob (inverse + log-det + base
    density) and forward, per call.  Launch-latency-bound: 80 KB of traffic per call."""
    from tests.helpers import golden_sd, golden_spec, load_flow_model, load_golden, t
    from torch_mnf import _lib

    g = load_golden("rnvp9_moons")  # the reference's own trained weights (tests/test_flows.py training loop)
    sd, specs = golden_sd(g), golden_spec(g)
    model = load_flow_model(specs, sd, device=dev, return_intermediates=False)
    try:
        from sklearn.datasets import make_moons

        x_host = torch.from_numpy(make_moons(4096, noise=0.05, random_state=0)[0]).float()  # data.py:21-24
        data = "make_moons(4096, noise=0.05, random_state=0)"
    except Exception:  # noqa: BLE001
        x_host = t(g, "inv/x").repeat(40, 1)[:4096].contiguous()
        data = "golden half-moon points tiled to 4096"
    x_pin = x_host.pin_memory()
    out_pin = torch.empty(4096).pin_memory()
    x = x_host.to(dev)
    lp = torch.empty(4096, device=dev)
    K = args.steps
    sites = kernels_of(lambda: model.log_prob(x, out=lp))
    ms = timed_ms(lambda: model.log_prob(x, out=lp), K, 20, dev)
    ms_fwd = timed_ms(lambda: model.forward(x), K, 20, dev)
    xd = torch.empty_like(x)

    def e2e():
        xd.copy_(x_pin, non_blocking=True)
        model.log_prob(xd, out=lp)
        out_pin.copy_(lp, non_blocking=True)

    e_ms = timed_ms(e2e, K, 20, dev)
    fast = None
    if hasattr(model, "log_prob_fn"):
        call = model.log_prob_fn(4096)
        ref_lp = model.log_prob(x).clone()
        ms_fast = timed_ms(lambda: call(x, lp), K, 20, dev)
        fast = {"us_per_call": ms_fast * 1e3, "value": 4096 / (ms_fast * 1e-3), "matches_module_call": bool(torch.equal(call(x), ref_lp)),
                "how": "NormalizingFlowModel.log_prob_fn: mnf_flow_handle_log_prob, the program bound once (no parameter "
                       "change check, allocation or descriptor marshalling per call)"}
    hbm_peak, peak_src, _ = peaks()
    res = {"metric": METRIC, "value": 4096 / (ms * 1e-3), "unit": "points/s", "us_per_call": ms * 1e3, "ms_per_step": ms,
           "forward_us_per_call": ms_fwd * 1e3, "steps": K, "warmup": 20, "dtype": "f32",
           "config": {"workload": "cfg1: RNVP x9 (AffineHalfFlow, h=24x3) on 2-D half-moons, batch 4096, log_prob per call",
                      "data": data, "l2": "32 KB per call: resident in L2 by construction of this configuration (latency-bound)"},
           "gpu_launches_per_call": sum(sites.values()), "kernels": sites,
           "roofline": {"bound": "hbm", "achieved": 12 * 4096 / (ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                        "frac": 12 * 4096 / (ms * 1e-3) / 1e9 / hbm_peak, "traffic": traffic_for("cfg1", 4096), "peak_source": peak_src,
                        "note": "49 KB of algorithmic traffic per call: the call is launch- and latency-bound (SURVEY 8d), "
                                "the HBM fraction is reported for completeness only; us_per_call is the figure of merit"},
           "e2e": {"value": 4096 / (e_ms * 1e-3), "unit": "points/s", "us_per_call": e_ms * 1e3, "h2d_bytes_per_step": 8 * 4096,
                   "d2h_bytes_per_step": 4 * 4096}}
    if fast:
        res["cached_handle"] = fast
    if not args.no_cpu:
        from oracle import flows_cpu

        cores = os.cpu_count() or 1
        torch.set_num_threads(cores)
        best = float("inf")
        for _ in range(20):
            t0 = time.perf_counter()
            flows_cpu.log_prob(sd, specs, x_host)
            best = min(best, time.perf_counter() - t0)
        res["cpu_baseline"] = {"value": 4096 / best, "unit": "points/s", "cores": cores, "kind": "port",
                               "sample": "the full 4096-point call, best of 20", "us_per_call": best * 1e6}
    return res


def cfg3(args, dev):
    """BASELINE config 3: MAF x9 (MADE 64-24-24-24-128) on 64-dim Gaussian data, batch 2^20, density evaluation."""
    from tests.helpers import golden_sd, golden_spec, load_flow_model, load_golden

    g = load_golden("maf9_d64")
    sd, specs = golden_sd(g), golden_spec(g)
    model = load_flow_model(specs, sd, device=dev, return_intermediates=False)
    n = 1 << 20
    x_pin = torch.randn(n, 64, generator=torch.Generator().manual_seed(0)).pin_memory()
    x = x_pin.to(dev)
    steps = args.steps
    res = {}
    rows = []
    for prec in ("auto", "fp32"):
        for f in model.flows:
            f.precision = prec
        sites = kernels_of(lambda: model.inverse(x))
        ms = timed_ms(lambda: model.inverse(x), steps, 3, dev)
        rows.append((prec, ms, sites))
    for f in model.flows:
        f.precision = "auto"
    prec, ms, sites = rows[0]
    lp_pin = torch.empty(n).pin_memory()
    xd = torch.empty_like(x)

    def e2e():
        xd.copy_(x_pin, non_blocking=True)
        lp_pin.copy_(model.log_prob(xd), non_blocking=True)

    e_ms = timed_ms(e2e, steps, 2, dev)
    hbm_peak, peak_src, _ = peaks()
    tf32_peak, tf32_src = _tf32_peak()
    flops_row = 9 * 2 * (64 * 24 + 24 * 24 + 24 * 24 + 24 * 128)  # 103 680 dense flops per row (SURVEY 8d)
    tflops = flops_row * n / (ms * 1e-3) / 1e12
    on_tc = any("made_fused" in k or "tf32_gemm" in k for k in sites)
    res = {"metric": METRIC, "value": n / (ms * 1e-3), "unit": "rows/s", "ms_per_step": ms, "steps": steps, "warmup": 3,
           "dtype": "tf32 tensor cores (MADE GEMMs, 2e-3 class), fp32 elsewhere" if on_tc else "f32",
           "config": {"workload": "cfg3: MAF x9 (MADE 64-24-24-24-128), 64-dim Gaussian data, batch 2^20, density (inverse: z and log_det stored)",
                      "l2": "268 MB of rows per step, larger than the 126 MB L2"},
           "gpu_launches_per_step": sum(sites.values()), "kernels": sites,
           "roofline": {"bound": "hbm", "achieved": 516 * n / (ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                        "frac": 516 * n / (ms * 1e-3) / 1e9 / hbm_peak, "traffic": traffic_for("cfg3", n), "peak_source": peak_src,
                        "bytes_per_row": 516},
           "tensor_pipe": {"dense_tflops": tflops, "peak": tf32_peak, "frac": tflops / tf32_peak, "peak_source": tf32_src,
                           "flops_per_row": flops_row, "note": "dense-equivalent MADE flops (masks ~50% zero) against the TF32 peak"},
           "exact_fp32_path": {"ms_per_step": rows[1][1], "value": n / (rows[1][1] * 1e-3), "kernels": rows[1][2]},
           "e2e": {"value": n / (e_ms * 1e-3), "unit": "rows/s", "ms_per_step": e_ms, "h2d_bytes_per_step": 256 * n,
                   "d2h_bytes_per_step": 4 * n, "how": "pinned host rows -> device -> NormalizingFlowModel.log_prob -> pinned host log-probs"}}
    if not args.no_cpu:
        from oracle import flows_cpu

        cores = os.cpu_count() or 1
        torch.set_num_threads(cores)
        xc = x_pin[: 1 << 16]
        best = float("inf")
        for _ in range(2):
            t0 = time.perf_counter()
            flows_cpu.stack(sd, specs, xc, True)
            best = min(best, time.perf_counter() - t0)
        res["cpu_baseline"] = {"value": (1 << 16) / best, "unit": "rows/s", "cores": cores, "kind": "port",
                               "sample": "2^16 rows of the 2^20-row batch, best of 2"}
    return res


def cfg4(args, dev, world, rank, total_samples=500, per_gpu_samples=None):
    """BASELINE config 4: MNF-LeNet Monte-Carlo predictive samples/s.  1024 synthetic 28x28 images x 500 MC samples per
    image; the MC-sample axis is sharded over the ranks (strong scaling: 500 samples in total), conv z shared through
    the common seed, per-row noise keyed by the global row; ranks reduce their samples to per-image class
    probabilities and all-reduce the [1024, 10] sums -- the raw samples never cross NVLink.
    per_gpu_samples: weak-scaling form (`--workload cfg4 --mc-samples S`)."""
    import torch.distributed as dist
    from tests.helpers import golden_sd, load_golden
    from torch_mnf import _lib
    from torch_mnf.distributed import shard_range
    from torch_mnf.models import MNFLeNet

    net = MNFLeNet()
    net.load_state_dict(golden_sd(load_golden("mnf_lenet")))  # the briefly trained fixture (tests/golden)
    net.to(dev)
    n_img, chunk = 1024, 25
    if per_gpu_samples is not None:
        s_lo, s_hi = rank * per_gpu_samples, (rank + 1) * per_gpu_samples
        total_s = per_gpu_samples * world
    else:
        s_lo, s_hi = shard_range(total_samples, world, rank)
        total_s = total_samples
    imgs_host = torch.rand(n_img, 1, 28, 28, generator=torch.Generator().manual_seed(0)).pin_memory()
    imgs = imgs_host.to(dev)
    probs_host = torch.empty(n_img, 10).pin_memory()
    counter = [0]

    def step(from_host=False):
        counter[0] += 1
        x = imgs_host.to(dev, non_blocking=True) if from_host else imgs
        # the public MC-prediction call (MNFLeNet.predict): this rank's samples, partial probability sums
        sums = net.predict(x, n_samples=total_s, chunk=chunk, seed=1000 + counter[0] * 131, sample_range=(s_lo, s_hi))
        if world > 1:
            dist.all_reduce(sums)
        probs = sums / total_s
        if from_host:
            probs_host.copy_(probs, non_blocking=True)
        return probs

    steps = args.steps
    sites = kernels_of(step)
    l0 = _lib.lib().mnf_launch_count()
    ms = timed_ms(step, steps, 3, dev, world)
    launches = (_lib.lib().mnf_launch_count() - l0) // (steps + 3)
    e_ms = timed_ms(lambda: step(True), steps, 1, dev, world)
    if rank != 0:
        return None
    total = n_img * total_s
    flops = 8.2e6 * total  # SURVEY 8d: ~8.2 MFLOP per sample (dense count, conv1 per sample)
    tf32_peak, tf32_src = _tf32_peak()
    ach = flops / (ms * 1e-3) / 1e12 / world
    res = {"metric": "MNF-LeNet MC predictive samples/s", "value": total / (ms * 1e-3), "unit": "samples/s", "n_gpus": world,
           "steps": steps, "warmup": 3, "ms_per_step": ms, "higher_is_better": True,
           "scaling": "weak" if per_gpu_samples is not None else "strong", "vs_baseline": None,
           "dtype": "tf32 tensor cores (conv2, fc1) / f32", "data": "synthetic",
           "config": {"workload": f"cfg4: MNF-LeNet (696,950 params), 1024 images x {total_s} MC samples per image in total",
                      "parallelism": f"MC samples sharded over {world} GPU(s) ({s_hi - s_lo} on rank 0); all_reduce of [1024,10] probability sums",
                      "l2": "activations (46 KB/sample before the pool of conv1, 11.5 KB/sample after it) far exceed L2"},
           "gpu_launches_per_step": launches, "kernels": sites,
           "e2e": {"value": total / (e_ms * 1e-3), "unit": "samples/s", "h2d_bytes_per_step": n_img * 784 * 4,
                   "d2h_bytes_per_step": n_img * 40, "ms_per_step": e_ms},
           "roofline": {"bound": "tensor", "achieved": ach, "peak": tf32_peak, "unit": "TFLOP/s", "frac": ach / tf32_peak,
                        "traffic": traffic_for("cfg4", total / world), "peak_source": tf32_src,
                        "note": "dense-equivalent 8.2 MFLOP/sample per GPU against the TF32 peak; the pipeline is co-bound by "
                                "operand generation in shared memory (implicit-GEMM conv2) and Philox noise (15.6 k normals/sample)"},
           "normals_per_s": 15630 * total / (ms * 1e-3),
           "cpu_baseline": None}
    if world == 1 and not args.no_cpu:
        # the reference's CPU path (oracle port: same ATen ops) on a bounded sample: 8 images x 250 MC samples
        from oracle import mnf_cpu
        from oracle.noise import FreshNoise

        cores = os.cpu_count() or 1
        torch.set_num_threads(cores)
        sd_cpu = {k: v.detach().cpu() for k, v in net.state_dict().items()}
        xc = imgs_host[:8].repeat(250, 1, 1, 1)
        best = float("inf")
        with torch.no_grad():
            for _ in range(3):
                t_0 = time.perf_counter()
                mnf_cpu.lenet_forward(sd_cpu, xc, FreshNoise())
                best = min(best, time.perf_counter() - t_0)
        res["cpu_baseline"] = {"value": xc.size(0) / best, "unit": "samples/s", "cores": cores, "kind": "port",
                               "sample": "8 images x 250 MC samples (2000 rows), best of 3"}
    return res


def cfg5(args, dev, world, rank):
    """BASELINE config 5: MNFLinear(4096, 4096), 64 input rows x 8192 MC samples + one kl_div() per step; the MC-sample
    axis is sharded over the ranks (strong scaling), MC mean and second moment [64, 4096] all-reduced -- never the raw
    [R, 4096] outputs (SURVEY 8e)."""
    import torch.distributed as dist
    from torch_mnf import _lib
    from torch_mnf.distributed import shard_range
    from torch_mnf.layers import MNFLinear
    from torch_mnf.layers import _train
    from torch_mnf.layers._mnf_ops import Noise

    torch.manual_seed(0)
    layer = MNFLinear(4096, 4096).to(dev)
    x_pin = torch.randn(64, 4096, generator=torch.Generator().manual_seed(0)).pin_memory()
    x64 = x_pin.to(dev)
    S_tot = args.cfg5_samples
    s_lo, s_hi = shard_range(S_tot, world, rank)
    S = s_hi - s_lo
    R = 64 * S
    stats_pin = torch.empty(2, 64 * 4096).pin_memory()
    counter = [0]

    def step(e2e=False):
        counter[0] += 1
        x = x_pin.to(dev, non_blocking=True) if e2e else x64
        y = layer.forward_mc(x, S, noise=Noise(None, dev, s_lo * 64, seed=17 + counter[0]))
        kl = layer.kl_div()
        if e2e or world > 1:
            flat = y.view(S, 64 * 4096)
            m1, m2 = _train.colsum(flat), _train.colsum(flat, flat)  # MC sums of y and y^2 over the sample axis
            st = torch.stack([m1, m2])
            if world > 1:
                dist.all_reduce(st)
            if e2e:
                stats_pin.copy_(st / S_tot, non_blocking=True)
        return kl

    steps = args.steps
    sites = kernels_of(step)
    ms = timed_ms(step, steps, 2, dev, world)
    fwd_ms = timed_ms(lambda: layer.forward_mc(x64, S, noise=Noise(None, dev, s_lo * 64, seed=5)), steps, 1, dev, world)
    kl_ms = timed_ms(lambda: layer.kl_div(), steps, 3, dev, world)
    e_ms = timed_ms(lambda: step(True), steps, 1, dev, world)
    if rank != 0:
        return None
    R_tot = 64 * S_tot
    h = 64  # conditioner width padded to one 64-wide tile
    executed = 2.0 * R * 4096 * 4096 + 2.0 * 64 * 4096 * 4096 + 2 * (2.0 * R * 4096 * h + 2.0 * R * h * 8192)
    tf32_peak, tf32_src = _tf32_peak()
    ach = executed / (fwd_ms * 1e-3) / 1e12
    hbm_peak, _, _ = peaks()
    res = {"metric": "MNFLinear MC rows/s (forward over all MC rows + one kl_div per step)", "value": R_tot / (ms * 1e-3),
           "unit": "rows/s", "n_gpus": world, "steps": steps, "warmup": 2, "ms_per_step": ms,
           "scaling": "strong", "dtype": "tf32 tensor cores (2e-3 class), fp32 accumulate",
           "config": {"workload": f"cfg5: MNFLinear(4096,4096), 64 rows x {S_tot} MC samples = {R_tot} rows, 2+2 RNVP flows (h=50), + kl_div()",
                      "parallelism": f"MC samples sharded over {world} GPU(s); all_reduce of the [2, 64, 4096] MC moment sums",
                      "l2": f"{R * 4096 * 4 / 1e9:.1f} GB of outputs per GPU per step, far larger than L2"},
           "forward_ms": fwd_ms, "forward_rows_per_s": R_tot / (fwd_ms * 1e-3), "kl_div_ms": kl_ms,
           "gpu_launches_per_step": sum(sites.values()), "kernels": sites,
           "roofline": {"bound": "tensor", "achieved": ach, "peak": tf32_peak, "unit": "TFLOP/s", "frac": ach / tf32_peak,
                        "traffic": traffic_for("cfg5", R), "peak_source": tf32_src,
                        "note": "EXECUTED flops of forward per GPU (mean GEMM per row, variance GEMM once per distinct input row, "
                                "RNVP q-flow GEMMs with the conditioner padded to 64) over the forward time, against the TF32 peak"},
           "kl_div_roofline": {"bound": "hbm", "achieved": 2 * 4096 * 4096 * 4 / (kl_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                               "frac": 2 * 4096 * 4096 * 4 / (kl_ms * 1e-3) / 1e9 / hbm_peak,
                               "note": "one read of W_mean and W_log_var (134 MB), eps_w from Philox; whole kl_div() call"},
           "e2e": {"value": R_tot / (e_ms * 1e-3), "unit": "rows/s", "ms_per_step": e_ms, "h2d_bytes_per_step": 64 * 4096 * 4,
                   "d2h_bytes_per_step": 2 * 64 * 4096 * 4,
                   "how": "pinned host x[64,4096] -> forward_mc -> MC mean / second moment over the samples (library kernel) -> pinned host"},
           "cpu_baseline": None}
    if world == 1 and not args.no_cpu:
        from oracle import mnf_cpu
        from oracle.noise import FreshNoise

        cores = os.cpu_count() or 1
        torch.set_num_threads(cores)
        sd5 = {k: v.detach().cpu() for k, v in layer.state_dict().items()}
        xc = x_pin.repeat(16, 1)  # 1024 rows
        best = float("inf")
        with torch.no_grad():
            for _ in range(2):
                t0 = time.perf_counter()
                mnf_cpu.linear_forward(sd5, xc, FreshNoise())
                best = min(best, time.perf_counter() - t0)
            t0 = time.perf_counter()
            mnf_cpu.linear_kl_div(sd5, FreshNoise())
            kl_cpu = time.perf_counter() - t0
        res["cpu_baseline"] = {"value": xc.size(0) / best, "unit": "rows/s", "cores": cores, "kind": "port",
                               "sample": "1024 rows (64 x 16 MC samples) of the forward, best of 2; kl_div once",
                               "kl_div_ms": kl_cpu * 1e3}
    return res


def run_all(args):
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback in the product path)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    t_start = time.time()
    out = run_ours(args)
    if args.workload == "all":
        extra = {}

        def attempt(name, fn):
            # a failing secondary configuration must never cost the headline line; every rank takes the same path
            t0 = time.time()
            try:
                r = fn()
            except Exception as e:  # noqa: BLE001
                r = {"error": f"{type(e).__name__}: {e}"[:400]}
                torch.cuda.synchronize(dev)
            if isinstance(r, dict):
                r["wall_s"] = round(time.time() - t0, 2)
            extra[name] = r
            torch.cuda.empty_cache()

        if world > 1:
            attempt("cfg2_strong", lambda: cfg_strong(args, dev, world, rank, build_model(dev)))
            for name in ("cfg1", "cfg3"):
                extra[name] = {"skipped": "single-GPU configuration (BASELINE names no multi-GPU form); measured at N=1"}
        else:
            attempt("cfg1", lambda: cfg1(args, dev))
            attempt("cfg3", lambda: cfg3(args, dev))
        attempt("cfg4", lambda: cfg4(args, dev, world, rank))
        attempt("cfg5", lambda: cfg5(args, dev, world, rank))
        if out is not None:
            out["configs"] = extra
            out["wall_s"] = round(time.time() - t_start, 2)
    if rank == 0 and out is not None:
        print(json.dumps(out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_lenet(args):
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    res = cfg4(args, dev, world, rank, per_gpu_samples=args.mc_samples)
    if rank == 0:
        sampler = None  # clocks are sampled on the headline line; this line is a secondary entry point
        print(json.dumps(res))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--points", type=int, default=N_POINTS, help="points per GPU (default 2^24)")
    ap.add_argument("--chunks", type=int, default=4, help="all-gather chunks per step when N>1")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline legs")
    ap.add_argument("--e2e-chunks", type=int, default=2, help="chunks per step of the host-to-host (e2e) pipeline")
    ap.add_argument("--gather", default="peer", choices=["peer", "nccl"],
                    help="N>1 result gather: fused peer-memory stores (default) or NCCL all-gather")
    ap.add_argument("--no-multicast", action="store_true", help="peer gather: per-peer stores even if NVLS multicast exists")
    ap.add_argument("--workload", default="all", choices=["all", "cfg2", "cfg4"],
                    help="all (default): the cfg2 headline line carrying every other configuration under `configs`; "
                         "cfg2: the headline alone; cfg4: the MNF-LeNet MC prediction line alone (weak scaling)")
    ap.add_argument("--mc-samples", type=int, default=64, help="--workload cfg4: MC samples per image per GPU per step")
    ap.add_argument("--cfg5-samples", type=int, default=8192, help="cfg5: MC samples (x 64 input rows) in total")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the headline's log-probs of the last step to DIR/log_prob.npy "
                         "(float32, every rank's points in rank order; above 2^22 values a fixed, seeded sample of them)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload == "cfg4"):
        ap.error("--dump-outputs writes the headline (cfg2) outputs: use it with --impl ours and --workload all or cfg2")
    torch.set_grad_enabled(False)  # the workload is density evaluation / prediction, not training
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "cfg4":
        run_lenet(args)
    else:
        run_all(args)


if __name__ == "__main__":
    main()
