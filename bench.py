#!/usr/bin/env python
"""bench.py -- the measurement contract (one JSON line on stdout from rank 0).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload NAME] [--no-secondary]
                    [--dump-outputs DIR]

N > 1 is launched by the driver as
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 ... bench.py --gpus N ...
one rank per GPU; the batch (independent sequences) is sharded across ranks with no data-path
collective; one NCCL all_gather of per-rank result checksums per step replaces the reference's
JSON-file + barrier gather (utils/caption_collect.py:7-37).  Timing is on the device (CUDA
events), max over ranks, barrier + synchronize on both sides.

The main line is BASELINE cfg 3 (benchmarks/workloads.py::InterleavedCfg3) through the reference surface
``MMInterleaved.forward``; the other BASELINE configurations that fit one GPU (cfg 2, cfg 4, cfg 5) are timed
afterwards with the same procedure at a few steps each and attached as ``"secondary": {name: {...}}`` objects.

``--dump-outputs DIR`` writes, after each workload's timed steps, what its last timed step (the last step of the
end-to-end loop) computed as ``DIR/<workload>.<output>.npy`` (float32, or float64 for float64 and integer outputs; an
output of more than 2**20
elements is reduced to a fixed seeded sample of them).  Inputs and weights are seeded, so two builds run with the same
arguments can be compared output for output.
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
sys.path.insert(0, ROOT)


DUMP_LIMIT_BYTES = 64 * 2 ** 20


def positive_int(text):
    n = int(text)
    if n < 1:
        raise argparse.ArgumentTypeError(f"must be >= 1, got {n}")
    return n


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=positive_int, default=10, help="timed steps of the main workload")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="auto")
    ap.add_argument("--local-batch", type=int, default=0, help="sequences per GPU per step (0 = workload default)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the cfg 2 / cfg 4 / cfg 5 secondary measurements")
    ap.add_argument("--secondary", default="", help="comma-separated subset of secondary workloads to run")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write each workload's last timed step's outputs to DIR/<workload>.<output>.npy")
    return ap.parse_args()


def dump_outputs(directory, workload, outputs, written):
    """Write ``outputs`` ({name: tensor}) as float32 / float64 .npy files; returns ``written`` + their bytes."""
    import numpy as np
    import torch
    os.makedirs(directory, exist_ok=True)
    for name, t in outputs.items():
        t = t.detach().cpu()
        a = (t.double() if t.dtype == torch.float64 or not t.is_floating_point() else t.float()).numpy()
        written += a.nbytes
        if written > DUMP_LIMIT_BYTES:
            raise SystemExit(f"--dump-outputs: more than {DUMP_LIMIT_BYTES} bytes at {workload}.{name}")
        np.save(os.path.join(directory, f"{workload}.{name}.npy"), a)
    return written


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (profiling recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [l for (t, l) in self.lines if t0 - 0.05 <= t <= t1 + 0.15] or [l for (_, l) in self.lines]
        sm, mx, reasons = [], [], set()
        for l in rows:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measure(wl, steps, warmup, dist, rank, world, local_rank, cpu_baseline):
    """The timing procedure of the contract for one workload; returns its result object."""
    import torch

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    warmup = max(warmup, 3) if wl.default_steps is None else max(warmup, 1)
    # ---------------- device-resident timing (`value`) ----------------
    for _ in range(warmup):
        wl.flush_l2()
        wl.step_device()
        wl.gather(dist)
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.25)
    wl.reset_counters()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    barrier()
    t_wall0 = time.time()
    for i in range(steps):
        wl.flush_l2()              # inputs (< L2 size) must not be served from a warm L2
        ev[i][0].record()
        wl.step_device()
        wl.gather(dist)
        ev[i][1].record()
    barrier()
    t_wall1 = time.time()
    step_ms = [a.elapsed_time(b) for a, b in ev]
    total_ms = torch.tensor([sum(step_ms)], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
    total_s = float(total_ms.item()) * 1e-3
    clocks = sampler.stop(t_wall0, t_wall1) if rank == 0 else None
    launches = wl.launch_count()
    kernel = wl.kernel_stats()      # dominant-kernel CUDA-event timings gathered inside the region
    roofline = wl.roofline(kernel)

    # ---------------- end-to-end timing through the public API with host buffers ----------------
    for _ in range(2 if wl.default_steps is None else 1):
        wl.step_e2e()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        wl.step_e2e()
        wl.gather(dist)
    e1.record()
    barrier()
    e2e_ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(e2e_ms, op=dist.ReduceOp.MAX)
    e2e_s = float(e2e_ms.item()) * 1e-3

    units = wl.units_per_step() * world      # whole job: one rank-local step per rank
    value = units * steps / total_s
    e2e_value = units * steps / e2e_s
    line = {
        "metric": wl.metric, "value": value, "unit": wl.unit, "n_gpus": world, "steps": steps,
        "warmup": warmup, "ms_per_step": total_s * 1e3 / steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": wl.dtype_name, "data": "synthetic",
        "config": wl.config(),
        "e2e": dict({"value": e2e_value, "unit": wl.unit, "h2d_bytes_per_step": wl.h2d_bytes(),
                     "d2h_bytes_per_step": wl.d2h_bytes()}, **{k: (v * e2e_value / value if k.endswith("_per_s") and v else v)
                                                               for k, v in wl.extras(value).items() if k.endswith("_per_s")}),
        "gpu_launches": launches,
        "clocks": clocks,
        "roofline": roofline,
    }
    line.update(wl.extras(value))
    if cpu_baseline and rank == 0 and world == 1:
        line["cpu_baseline"] = wl.cpu_baseline()
    return line


def main():
    args = parse_args()
    import torch

    from benchmarks import workloads

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        # the reference's own CPU implementation of the path, on the host cores; rank 0 only
        if rank != 0:
            return 0
        line = workloads.run_reference_arm(args, world)
        print(json.dumps(line), flush=True)
        return 0

    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    wl = workloads.make(args.workload, rank=rank, world=world, local_batch=args.local_batch)
    wl.setup()
    line = measure(wl, args.steps, args.warmup, dist, rank, world, local_rank, cpu_baseline=not args.no_cpu_baseline)
    dumped = 0
    if args.dump_outputs and rank == 0:
        dumped = dump_outputs(args.dump_outputs, wl.name, wl.outputs(), dumped)
    wl.teardown()

    main_name = workloads.AUTO if args.workload == "auto" else args.workload
    if main_name == workloads.AUTO and not args.no_secondary:
        names = [n for n in workloads.SECONDARY if not args.secondary or n in args.secondary.split(",")]
        line["secondary"] = {}
        for name in names:
            try:
                sw = workloads.make(name, rank=rank, world=world, local_batch=0)
                sw.setup()
                line["secondary"][name] = measure(sw, sw.default_steps, sw.default_warmup, dist, rank, world, local_rank,
                                                  cpu_baseline=False)
                if args.dump_outputs and rank == 0:
                    dumped = dump_outputs(args.dump_outputs, name, sw.outputs(), dumped)
                sw.teardown()
            except Exception as e:          # a secondary must never take the main line down
                import traceback
                line["secondary"][name] = {"error": f"{type(e).__name__}: {e}", "trace": traceback.format_exc()[-1500:]}
            torch.cuda.empty_cache()
    if rank == 0:
        print(json.dumps(line), flush=True)
    if dist is not None:
        try:
            dist.destroy_process_group()
        except Exception:
            pass
    return 0


if __name__ == "__main__":
    sys.exit(main())
