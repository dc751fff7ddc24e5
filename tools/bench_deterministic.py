#!/usr/bin/env python
"""bench_deterministic.py -- what deterministic mode (torch.use_deterministic_algorithms(True), DESIGN.md section 10) costs on
the headline training step of bench.py (73 x 720 x 1440 synthetic fields, 'squared geometric l2', batch 1, bf16), and whether
it delivers equal bits.

    python tools/bench_deterministic.py [--steps 10] [--warmup 3] [--rounds 3] [--out profiles/deterministic]

In one call it
  * times zero_grad + forward + loss + backward with the flag off and on, alternating, `--rounds` times each (CUDA events);
  * times the flag-on step once more with torch.utils.deterministic.fill_uninitialized_memory = False: under the flag torch
    fills every torch.empty with NaN, traffic that the kernels do not cause;
  * runs one training step in three fresh processes -- two with the flag on, one without -- and writes their outputs with
    bench.dump_outputs; asserts that the two deterministic dumps are bitwise identical and reports the relative L2 distance
    between the deterministic and the default dump;
  * records the GPU's name and power limit.
The JSON result goes to OUT/bench_deterministic.json and to stdout.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
os.environ.setdefault("CUBLAS_WORKSPACE_CONFIG", ":4096:8")     # torch-side cuBLAS calls (none in the headline config)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from bench import dump_outputs, make_loss, make_model  # noqa: E402


def setup(dev):
    model = make_model(dev, "bf16")
    lossf = make_loss(dev)
    gen = torch.Generator().manual_seed(1234)
    x = torch.randn(1, 73, 720, 1440, generator=gen).to(dev)
    t = torch.randn(1, 73, 720, 1440, generator=gen).to(dev)
    params = list(model.parameters())

    def step():
        for p in params:
            p.grad = None
        torch.manual_seed(5)          # DropPath draws
        pred = model(x)
        loss = lossf(pred, t, x)
        loss.backward()
        return loss, pred

    return model, step


def time_steps(step, steps, warmup):
    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    for _ in range(steps):
        step()
    ev[1].record()
    torch.cuda.synchronize()
    return ev[0].elapsed_time(ev[1]) / steps


def worker(out_dir, det):
    dev = torch.device("cuda", 0)
    torch.use_deterministic_algorithms(det)
    model, step = setup(dev)
    step()
    loss, pred = step()
    torch.cuda.synchronize()
    dump_outputs(out_dir, loss, pred, model)


def load_dump(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d)) if f.endswith(".npy")}


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        info["power_limit_and_max_sm_clock"] = r.stdout.strip().splitlines()[0] if r.returncode == 0 else None
    except (OSError, subprocess.SubprocessError, IndexError):
        info["power_limit_and_max_sm_clock"] = None
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "deterministic"))
    ap.add_argument("--worker", default=None, help=argparse.SUPPRESS)
    ap.add_argument("--det", type=int, default=1, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_deterministic.py needs a CUDA device")
    if args.worker:
        worker(args.worker, bool(args.det))
        return

    dev = torch.device("cuda", 0)
    _, step = setup(dev)
    off, on = [], []
    for _ in range(args.rounds):
        torch.use_deterministic_algorithms(False)
        off.append(time_steps(step, args.steps, args.warmup))
        torch.use_deterministic_algorithms(True)
        on.append(time_steps(step, args.steps, args.warmup))
    torch.utils.deterministic.fill_uninitialized_memory = False
    on_nofill = time_steps(step, args.steps, args.warmup)
    torch.utils.deterministic.fill_uninitialized_memory = True
    torch.use_deterministic_algorithms(False)
    torch.cuda.synchronize()

    dumps = {}
    with tempfile.TemporaryDirectory(prefix="swinb200_det_") as tmp:
        for name, det in (("det_a", 1), ("det_b", 1), ("default", 0)):
            d = os.path.join(tmp, name)
            subprocess.run([sys.executable, os.path.abspath(__file__), "--worker", d, "--det", str(det)], check=True)
            dumps[name] = load_dump(d)
    a, b, ref = dumps["det_a"], dumps["det_b"], dumps["default"]
    unequal = sorted(k for k in a if a[k].tobytes() != b[k].tobytes())
    rel = {k: float(np.linalg.norm(a[k].astype(np.float64) - ref[k]) / max(np.linalg.norm(ref[k].astype(np.float64)), 1e-30)) for k in a}
    worst = sorted(rel.items(), key=lambda kv: -kv[1])[:5]

    res = {
        "workload": "bench.py headline training step (bf16, batch 1, 73 x 720 x 1440)",
        "gpu": gpu_info(),
        "steps": args.steps, "warmup": args.warmup, "rounds": args.rounds,
        "ms_per_step_default": [round(v, 2) for v in off],
        "ms_per_step_deterministic": [round(v, 2) for v in on],
        "ms_per_step_deterministic_no_fill": round(on_nofill, 2),
        "dump_arrays": len(a),
        "deterministic_dumps_bitwise_equal": not unequal,
        "unequal_arrays": unequal,
        "rel_l2_deterministic_vs_default_max": max(rel.values()),
        "rel_l2_deterministic_vs_default_worst": worst,
        "loss_deterministic": float(a["loss"].reshape(-1)[0]), "loss_default": float(ref["loss"].reshape(-1)[0]),
    }
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "bench_deterministic.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res), flush=True)
    assert not unequal, f"deterministic dumps differ: {unequal[:5]}"


if __name__ == "__main__":
    main()
