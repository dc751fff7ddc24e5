#!/usr/bin/env python
"""bench_inference.py -- what the forward-only path (DESIGN.md section 11) saves when the headline model (bench.py's
73 x 720 x 1440 configuration, bf16, eval mode) runs without gradients.

    python tools/bench_inference.py [--iters 10] [--warmup 3] [--rounds 3] [--out profiles/inference]

Workloads, each timed with CUDA events over `--iters` calls after `--warmup` untimed ones:
  * fwd_b1 / fwd_b8: one forward at batch 1 and 8;
  * rollout4_b1: a 4-step MultiStepWrapper rollout at batch 1 (orography + the two land-mask channels re-appended every step).
Each runs under torch.no_grad() twice: on the forward-only path and, as the baseline, with the path choice forced to the
training Functions -- exactly the kernels and allocations no_grad ran before the forward-only path existed.  (Running with
gradients enabled and dropping the graph issues the same kernels, but at batch 8 it would also hold ~150 GB of saved
activations.)
The two arms alternate, `--rounds` times each, in one process.  Recorded per workload and arm: times, the peak of
torch.cuda.max_memory_allocated above what was allocated before the timed calls, kernel launches per call
(_lib.LAUNCH_COUNT), and whether the outputs of the two arms are bitwise equal.  GPU name, power limit and SM clocks are
read in the same run.  The JSON goes to OUT/bench_inference.json and to stdout.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
from types import SimpleNamespace

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from bench import make_model  # noqa: E402
from swin_v2_weather_b200 import _lib  # noqa: E402
from swin_v2_weather_b200.networks import swinv2_global as SG  # noqa: E402
from swin_v2_weather_b200.networks.helpers import MultiStepWrapper  # noqa: E402


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        info["power_limit_sm_clock_max_sm_clock"] = r.stdout.strip().splitlines()[0] if r.returncode == 0 else None
    except (OSError, subprocess.SubprocessError, IndexError):
        info["power_limit_sm_clock_max_sm_clock"] = None
    return info


def timed(fn, training_kernels: bool, iters: int, warmup: int):
    saved = SG._forward_only
    if training_kernels:
        SG._forward_only = lambda *t: False
    try:
        with torch.no_grad():
            for _ in range(warmup):
                out = fn()
            torch.cuda.synchronize()
            torch.cuda.reset_peak_memory_stats()
            base = torch.cuda.memory_allocated()
            n0 = _lib.LAUNCH_COUNT
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
            ev[0].record()
            for _ in range(iters):
                fn()
            ev[1].record()
            torch.cuda.synchronize()
    finally:
        SG._forward_only = saved
    return out, {"ms": ev[0].elapsed_time(ev[1]) / iters, "peak_mib": (torch.cuda.max_memory_allocated() - base) / 2**20,
                 "launches": (_lib.LAUNCH_COUNT - n0) / iters}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "inference"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_inference.py needs a CUDA device")
    dev = torch.device("cuda:0")
    model = make_model(dev, "bf16").eval()
    gen = torch.Generator().manual_seed(1234)
    x1 = torch.randn(1, 73, 720, 1440, generator=gen).to(dev)
    x8 = torch.randn(8, 73, 720, 1440, generator=gen).to(dev)
    # rollout: 73 prognostic channels + the 3 invariant channels (orography 1, land mask 2) in, 73 out; the invariants are
    # re-appended to the prediction every step
    roll_model = make_model(dev, "bf16", in_chans=76).eval()
    wrap = MultiStepWrapper(SimpleNamespace(n_future=3, add_orography=True, add_landmask=True), lambda p: roll_model)
    stat = torch.randn(1, 3, 720, 1440, generator=gen).to(dev)
    workloads = {
        "fwd_b1": lambda: model(x1),
        "fwd_b8": lambda: model(x8),
        "rollout4_b1": lambda: wrap([x1, stat]),
    }
    result = {"gpu": gpu_info(), "iters": args.iters, "warmup": args.warmup, "rounds": args.rounds, "workloads": {}}
    for name, fn in workloads.items():
        rounds, same = [], True
        for _ in range(args.rounds):
            ref, base = timed(fn, True, args.iters, args.warmup)
            out, fo = timed(fn, False, args.iters, args.warmup)
            same = same and bool(torch.equal(out, ref))
            rounds.append({"training_kernels": base, "forward_only": fo})
            del ref, out
        base_ms = sorted(r["training_kernels"]["ms"] for r in rounds)
        fo_ms = sorted(r["forward_only"]["ms"] for r in rounds)
        result["workloads"][name] = {"rounds": rounds, "training_kernels_ms_min_max": [base_ms[0], base_ms[-1]],
                                     "forward_only_ms_min_max": [fo_ms[0], fo_ms[-1]], "bitwise_equal": same}
        torch.cuda.empty_cache()
    result["gpu_after"] = gpu_info()
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "bench_inference.json"), "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
