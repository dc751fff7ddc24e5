#!/usr/bin/env python
"""bench_wide.py -- training throughput of the largest shipped configuration,
swin_73var_geo_depth24_e2048_mlp2_chweight_invar (embed_dim 2048, 8 heads of 256, depth 24, mlp_ratio 2; 943,347,904
parameters at 73 channels), on one GPU with the headline's synthetic data and loss (bench.py): 73 x 721 x 1440 N(0,1)
fields cropped to 720 rows, 'squared geometric l2', batch 1, zero_grad + forward + loss + backward per timed step.

    python tools/bench_wide.py [--steps 5] [--warmup 2] [--checkpoint-stages] [--batch 1]

Prints one JSON line: samples/s and ms/step (CUDA events), per-family device time and GEMM variants (CUDA events around
every launch, bench.KernelTimer), attention forward / backward against the tensor and HBM peaks, peak memory (the fused
Adam's moments are allocated before the timed steps, so the figure covers the whole training state), the model's FLOP
rate from shapes, and the GPU's name, power limit and clocks read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from bench import FIELD_ROWS, ClockSampler, KernelTimer, make_loss, read_peaks  # noqa: E402

WIDE = dict(img_size=(720, 1440), patch_size=4, depth=24, num_heads=8, in_chans=73, out_chans=73, embed_dim=2048,
            window_ratio=80, drop_path_rate=0.1, full_pos_embed=True, rel_pos=False, mlp_ratio=2.0)


def model_flops_per_sample(cfg=WIDE):
    """fwd + bwd FLOPs of one sample, from shapes: every GEMM 2 M N K, window attention 4 nW h L^2 d (S = Q K^T and P V), and the
    backward counted as twice the forward (dgrad + wgrad; dQ, dK, dV, dP for attention)."""
    H, W = cfg["img_size"][0] // cfg["patch_size"], cfg["img_size"][1] // cfg["patch_size"]
    T, C = H * W, cfg["embed_dim"]
    hid = int(C * cfg["mlp_ratio"])
    Wh, Ww = cfg["img_size"][0] // cfg["window_ratio"], cfg["img_size"][1] // cfg["window_ratio"]
    L, nW = Wh * Ww, (H // Wh) * (W // Ww)
    pp = cfg["patch_size"] ** 2
    block = 2.0 * T * C * (3 * C + C + 2 * hid) + 4.0 * nW * cfg["num_heads"] * L * L * (C // cfg["num_heads"])
    fwd = cfg["depth"] * block + 2.0 * T * cfg["in_chans"] * pp * C + 2.0 * T * C * cfg["out_chans"] * pp
    return 3.0 * fwd


def gpu_identity(index):
    """Name, power limit and clocks of the card, from nvidia-smi in this run (None where it is unavailable)."""
    fields = "name,power.limit,power.max_limit,clocks.sm,clocks.max.sm,clocks.mem"
    try:
        r = subprocess.run(["nvidia-smi", "-i", str(index), f"--query-gpu={fields}", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        vals = [v.strip() for v in r.stdout.strip().split(",")]
        if r.returncode == 0 and len(vals) == len(fields.split(",")):
            return dict(zip(fields.split(","), vals))
    except Exception:
        pass
    return {"name": torch.cuda.get_device_name(index), "power.limit": None}


def build_model(dev, mode, checkpoint_stages):
    from swin_v2_weather_b200.networks.swinv2_global import SwinTransformerV2Cr
    torch.manual_seed(0)
    with torch.device(dev):     # 943 M parameters: initialised on the device
        m = SwinTransformerV2Cr(img_size=WIDE["img_size"], patch_size=4, depths=(WIDE["depth"],), num_heads=(WIDE["num_heads"],),
                                in_chans=WIDE["in_chans"], out_chans=WIDE["out_chans"], embed_dim=WIDE["embed_dim"],
                                img_window_ratio=WIDE["window_ratio"], drop_path_rate=WIDE["drop_path_rate"],
                                full_pos_embed=WIDE["full_pos_embed"], rel_pos=WIDE["rel_pos"], mlp_ratio=WIDE["mlp_ratio"],
                                checkpoint_stages=checkpoint_stages, compute_mode=mode)
    with torch.no_grad():       # the reference zero-inits norm1/2.weight (every block the identity); bench.py does the same
        g = torch.Generator(device=dev).manual_seed(1)
        for blk in m.stages[0].blocks:
            blk.norm1.weight.copy_(1 + 0.1 * torch.randn(WIDE["embed_dim"], generator=g, device=dev))
            blk.norm2.weight.copy_(1 + 0.1 * torch.randn(WIDE["embed_dim"], generator=g, device=dev))
    return m.train()


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--batch", type=int, default=1)
    ap.add_argument("--mode", default="bf16", help="compute mode: bf16 | bf16_simt | fp32")
    ap.add_argument("--checkpoint-stages", action="store_true", help="activation checkpointing of the stage (recomputed forward)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 1:
        ap.error("--steps and --warmup must be >= 1")
    if not torch.cuda.is_available():
        sys.exit("bench_wide.py measures on a CUDA device; none is visible")

    from swin_v2_weather_b200 import _lib, ops
    from swin_v2_weather_b200.optim import Adam
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    _lib.load()
    peaks = read_peaks()
    B = args.batch
    model = build_model(dev, args.mode, args.checkpoint_stages)
    lossf = make_loss(dev)
    params = list(model.parameters())
    opt = Adam(params, lr=0.0, betas=(0.9, 0.95))        # lr 0: the moments exist (memory), the weights do not move

    gen = torch.Generator().manual_seed(1234)
    x = torch.randn(B, 73, FIELD_ROWS, 1440, generator=gen)[:, :, :720].contiguous().to(dev)
    t = torch.randn(B, 73, FIELD_ROWS, 1440, generator=gen)[:, :, :720].contiguous().to(dev)

    def step():
        for p in params:
            p.grad = None
        loss = lossf(model(x), t, x)
        loss.backward()
        return loss

    for _ in range(args.warmup):
        step()
        opt.step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    opt.step()
    e1.record()
    torch.cuda.synchronize()
    opt_ms = e0.elapsed_time(e1)

    timer = KernelTimer()
    _lib.PROFILE_HOOK = timer.hook
    ident = gpu_identity(0)
    sampler = ClockSampler(0)
    sampler.start()
    timer.enabled = True
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    torch.cuda.synchronize()
    ev[0].record()
    for _ in range(args.steps):
        loss = step()
    ev[1].record()
    torch.cuda.synchronize()
    timer.enabled = False
    _lib.PROFILE_HOOK = None
    clocks = sampler.stop()
    ms = ev[0].elapsed_time(ev[1])
    fam = timer.summary()

    T = 180 * 360
    C = WIDE["embed_dim"]
    value = args.steps * B / (ms / 1e3)
    flops = model_flops_per_sample()
    families = {k: {"ms_per_step": round(v["ms"] / args.steps, 3), "launches_per_step": v["launches"] / args.steps}
                for k, v in sorted(fam.items(), key=lambda kv: -kv[1]["ms"])}
    gemm_variants = {k: {"launches_per_step": v["launches"] / args.steps, "gflop": round(v["flops"] / v["launches"] / 1e9, 1),
                         "us": round(v["ms"] / v["launches"] * 1e3, 1), "tflops": round(v["flops"] / (v["ms"] / 1e3) / 1e12, 1),
                         "frac_of_sustained": round(v["flops"] / (v["ms"] / 1e3) / 1e12 / peaks["tf_sust"], 3)}
                     for k, v in sorted(timer.variants.items(), key=lambda kv: -kv[1]["ms"]) if v["ms"] > 0}
    attn = {}
    # algorithmic bytes: forward reads q^, k^, v and writes o; backward reads q^, k^, v, o, dO and writes dq, dk, dv (bf16)
    for key, nbytes in (("attn_fwd", 4 * T * C * 2), ("attn_bwd", 8 * T * C * 2)):
        a = fam.get(key)
        if a and a["ms"] > 0:
            tf = a["flops"] / (a["ms"] / 1e3) / 1e12
            gbs = nbytes * B * a["launches"] / (a["ms"] / 1e3) / 1e9
            attn[key] = {"us_per_launch": round(a["ms"] / a["launches"] * 1e3, 1), "tflops": round(tf, 1),
                         "frac_of_tc_peak_sustained": round(tf / peaks["tf_sust"], 4), "hbm_gbs": round(gbs, 0),
                         "frac_of_hbm_peak": round(gbs / peaks["hbm"], 4)}
    mode = ops.MODES[args.mode]
    out = {
        "metric": "samples/s (fwd+bwd) 73ch 721x1440 SwinV2 e2048 depth 24", "value": round(value, 4), "unit": "samples/s",
        "ms_per_step": round(ms / args.steps, 2), "steps": args.steps, "warmup": args.warmup, "batch": B,
        "config": {"workload": "swin_73var_geo_depth24_e2048_mlp2_chweight_invar: embed_dim 2048, 8 heads of 256, depth 24, "
                               "mlp_ratio 2, window 9x18, 64,800 tokens/sample; zero_grad + forward + 'squared geometric l2' + backward",
                   "compute_mode": args.mode, "checkpoint_stages": args.checkpoint_stages,
                   "parameters": sum(p.numel() for p in params),
                   "attention_backend": "tcgen05" if ops.attn_backend_for(mode, C, WIDE["num_heads"], 9, 18) == 1 else "cuda-core"},
        "gpu": ident, "clocks_during_timed_steps": clocks,
        "kernel_families": families, "gemm_variants": gemm_variants, "attn": attn,
        "model_tflop_per_sample": round(flops / 1e12, 1),
        "model_tflops": round(value * flops / 1e12, 1),
        "model_frac_of_sustained_peak": round(value * flops / 1e12 / peaks["tf_sust"], 4),
        "peaks": {"tf_sust": peaks["tf_sust"], "hbm_gbs": peaks["hbm"], "source": peaks["src"]},
        "peak_mem_gib": round(torch.cuda.max_memory_allocated(dev) / 2 ** 30, 2),
        "peak_reserved_gib": round(torch.cuda.max_memory_reserved(dev) / 2 ** 30, 2),
        "optimizer_step_ms": round(opt_ms, 2),
        "last_loss": float(loss.detach()),
    }
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
