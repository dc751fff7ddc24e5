#!/usr/bin/env python
"""bench.py -- headline benchmark: training samples/s (fwd + loss + bwd) of the 73-channel, depth-12 SwinV2
weather model on synthetic 73x721x1440 fields (cropped to 720 rows exactly as the reference loaders do),
batch 1 per GPU, data-parallel over N B200s.

    python bench.py --gpus 1 --steps 10 --warmup 3                    # our CUDA path (one JSON line)
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...                               # the reference algorithm on the host CPU cores
    python bench.py --gpus 1 --steps 10 --warmup 3 --dump-outputs DIR  # + the last timed step's results as DIR/*.npy

`value`      : whole-job samples/s with inputs already resident in HBM (CUDA events, max over ranks).
`e2e`        : same metric through the public model API from pinned HOST buffers: per step the H2D copy of that
               step's input + target and the D2H read of the loss are inside the timed region.
`roofline`   : the dominant kernel family, timed live with CUDA events inside the timed region.
`cpu_baseline`: the CPU oracle (a port of the reference algorithm) on the host cores, bounded sample (1/10 sample: all 12 blocks
               on 40 of the 400 windows).  `gpu_eager_baseline`: the same oracle as eager PyTorch on the GPU under bf16 autocast.
`gemm_variants` / `attn_pct_tc_peak`: per-shape GEMM table and the attention kernels against tensor and HBM peaks.
"""
from __future__ import annotations

import argparse
import contextlib
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

# ---- workload (BASELINE.json configs[1]: swin_73var_geo_depth12, config/swin.yaml:145-150 over :2-16) ----
CFG = dict(img_size=(720, 1440), patch_size=4, depth=12, num_heads=8, in_chans=73, out_chans=73, embed_dim=768,
           window_ratio=80, drop_path_rate=0.1, full_pos_embed=True, rel_pos=False, mlp_ratio=4.0, residual=False)
FIELD_ROWS = 721          # ERA5 rows on disk; the loaders crop [:720] (data_loader_era5.py:163-165)
T = 180 * 360             # tokens per sample
FLOPS_FWD_BWD = 34.96e12  # per sample, SURVEY section 8(a)


def read_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sust=d["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src="fallback")


# ---- clocks sampler ----------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.path = index, None, None

    def start(self):
        try:
            self.path = tempfile.mktemp(prefix="clocks_", suffix=".csv")
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in open(self.path):
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for n, v in zip(names, parts[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        os.unlink(self.path)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---- kernel-family timer (CUDA events on the launching stream, no syncs inside the timed region) ------------------
class KernelTimer:
    FAMILY = {"swinb200_gemm": "gemm", "swinb200_window_attn_fwd": "attn_fwd", "swinb200_window_attn_bwd": "attn_bwd",
              "swinb200_ln_residual_fwd": "ln_fwd", "swinb200_ln_residual_bwd": "ln_bwd", "swinb200_colsum": "colsum",
              "swinb200_patchify": "patchify", "swinb200_unpatchify": "unpatchify", "swinb200_latw_l2_fwd": "loss",
              "swinb200_latw_l2_bwd": "loss", "swinb200_transpose_f32": "transpose", "swinb200_pos_embed_grad": "transpose",
              "swinb200_cast_f32_to_bf16": "cast", "swinb200_linear_ln_residual": "gemm_ln",
              "swinb200_linear_wgrad": "gemm_wgrad"}

    def __init__(self):
        self.records = []   # (family, flops, bytes, start_event, end_event)
        self.enabled = False

    @contextlib.contextmanager
    def hook(self, name, args):
        fam = self.FAMILY.get(name)
        if not self.enabled or fam is None:
            yield
            return
        flops = bytes_ = 0.0
        variant = None
        if fam in ("attn_fwd", "attn_bwd"):
            # window attention FLOPs with the UNPADDED window length (SURVEY 8(a)): fwd 4 nW h L^2 d, bwd 10 nW h L^2 d
            if fam == "attn_fwd":
                Bq, H, W, C, heads, Wh, Ww = args[7:14]
            else:
                Bq, H, W, C, heads, Wh, Ww = args[13:20]
            L = Wh * Ww
            flops = (4.0 if fam == "attn_fwd" else 10.0) * Bq * (H // Wh) * (W // Ww) * heads * L * L * (C // heads)
        if fam == "gemm_ln":
            # proj / fc2 + LayerNorm + residual in one kernel: GEMM operands + z (bf16) + x_in, x_out (fp32) + bf16 shadow
            M, N, K = args[1], args[2], args[3]
            fam = "gemm_tcgen05"
            flops = 2.0 * M * N * K
            bytes_ = 2.0 * (M * K + N * K) + 12.0 * M * N
            variant = f"M{M}_N{N}_K{K}_a0b0_bias_ln_residual"
        if fam == "gemm_wgrad":
            # weight + bias gradient in one kernel: dW (n_out, n_in) += dY^T X, dbias += column sums of dY (read from the staged tiles)
            M, N, K = args[1], args[2], args[3]
            fam = "gemm_tcgen05"
            flops = 2.0 * M * N * K
            bytes_ = 2.0 * (M * K + N * K) + 4.0 * M * N
            variant = f"M{M}_N{N}_K{K}_a1b1_f32_colsum" + (f"_splitk{args[11]}" if args[11] > 1 else "")
        if fam == "gemm":
            backend, M, N, K = args[0], args[1], args[2], args[3]
            fam = "gemm_tcgen05" if backend == 1 else "gemm_simt"
            flops = 2.0 * M * N * K
            # algorithmic bytes: both operands once + every output / epilogue operand once (swinb200_gemm argument order)
            esz = 2 if args[10] == 1 else 4
            epi = args[11]
            out_b = {0: esz, 1: 2 * esz, 2: 2 * esz, 3: 8, 4: 4, 5: esz}.get(epi, esz)    # per output element
            bytes_ = float(esz) * (M * K + N * K) + float(out_b) * M * N
            epi_name = {0: "bias", 1: "bias_gelu", 2: "dgelu", 3: "add_f32", 4: "f32", 5: "bias_qknorm"}.get(epi, str(epi))
            variant = f"M{M}_N{N}_K{K}_a{args[5]}b{args[8]}_{epi_name}" + (f"_splitk{args[20]}" if args[20] > 1 else "")
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        yield
        e.record()
        self.records.append((fam, flops, bytes_, s, e, variant))

    def summary(self):
        fam, var = {}, {}
        for f, fl, by, s, e, v in self.records:
            ms = s.elapsed_time(e)
            for key, table in ((f, fam), (v, var)):
                if key is None:
                    continue
                d = table.setdefault(key, dict(ms=0.0, flops=0.0, bytes=0.0, launches=0))
                d["ms"] += ms
                d["flops"] += fl
                d["bytes"] += by
                d["launches"] += 1
        self.variants = var
        return fam


def gemm_traffic(B, mode):
    """DRAM bytes per GEMM launch from the committed ncu capture (never a literal): profiles/gemm_traffic.json is written
    by tools/traffic_summary.py from the ncu CSV named inside it."""
    p = os.path.join(ROOT, "profiles", "gemm_traffic.json")
    if not (B == 1 and mode == "bf16" and os.path.exists(p)):
        return {"traffic": None, "traffic_source": None}
    d = json.load(open(p))
    return {"traffic": d["bytes_per_launch"], "traffic_source": f"{d['source']} ({d['when']}; {d['launches']} launches, "
            f"{d['read_mb_per_launch']:.1f} MB read + {d['write_mb_per_launch']:.1f} MB written per launch)"}


def make_model(device, compute_mode="bf16", in_chans=None, residual=False):
    from swin_v2_weather_b200.networks.swinv2_global import SwinTransformerV2Cr
    torch.manual_seed(0)
    m = SwinTransformerV2Cr(img_size=CFG["img_size"], patch_size=4, depths=(CFG["depth"],), num_heads=(CFG["num_heads"],),
                            in_chans=in_chans or CFG["in_chans"], out_chans=CFG["out_chans"], embed_dim=CFG["embed_dim"],
                            img_window_ratio=CFG["window_ratio"], drop_path_rate=CFG["drop_path_rate"],
                            full_pos_embed=True, rel_pos=False, mlp_ratio=CFG["mlp_ratio"], residual=residual,
                            compute_mode=compute_mode)
    with torch.no_grad():   # SURVEY F7: the reference zero-inits norm1/2.weight, which makes every block the identity
        g = torch.Generator().manual_seed(1)
        for blk in m.stages[0].blocks:
            blk.norm1.weight.copy_(1 + 0.1 * torch.randn(768, generator=g))
            blk.norm2.weight.copy_(1 + 0.1 * torch.randn(768, generator=g))
    return m.to(device).train()


CHANNEL_NAMES_73 = (["u10m", "v10m", "u100m", "v100m", "t2m", "sp", "msl", "tcwv"]      # config/swin.yaml:60-133
                    + [f"{v}{lev}" for v in "uvztq" for lev in (50, 100, 150, 200, 250, 300, 400, 500, 600, 700, 850, 925, 1000)])


def make_loss(device, config4=False):
    from types import SimpleNamespace
    from swin_v2_weather_b200.utils.losses import LossHandler
    p = SimpleNamespace(n_future=0, img_shape_x=720, img_shape_y=1440, loss='squared geometric l2', channel_weights='none',
                        n_out_channels=73, channel_names=[], out_channels=list(range(73)), dt=1, model_grid_type='equiangular')
    if config4:   # BASELINE config 4 / SURVEY 8(d): 'auto' channel table x (sigma_global / sigma_dt)^2, synthetic statistics
        import numpy as np
        d = tempfile.mkdtemp(prefix="swinb200_stats_")
        np.save(os.path.join(d, "gs.npy"), np.ones((1, 73, 1, 1), dtype=np.float32))
        np.save(os.path.join(d, "ts.npy"), np.random.default_rng(7).uniform(0.2, 1.0, size=(1, 73, 1, 1)).astype(np.float32))
        p.loss, p.channel_weights, p.channel_names = 'weighted absolute temp-std squared geometric l2', 'auto', list(CHANNEL_NAMES_73)
        p.global_stds_path, p.time_diff_stds_path = os.path.join(d, "gs.npy"), os.path.join(d, "ts.npy")
    return LossHandler(p).to(device).train()


DUMP_GRAD_ELEMS = 1 << 17     # per gradient; larger ones are sampled (51 of the 162 tensors of the headline model)
DUMP_PRED_ELEMS = 1 << 21     # of the (B, 73, 720, 1440) prediction
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir, loss, pred, model):
    """What one training step hands its caller -- the loss, the prediction and every parameter gradient -- as float32
    DIR/loss.npy, DIR/pred.npy and DIR/grad.<parameter name>.npy.  An array above its element cap is replaced by the
    elements at a fixed set of flat positions (seeded by the array's size, sorted), the same in every run, so the files of
    two builds compare element for element."""
    import numpy as np
    arrays = {"loss": (loss, 1), "pred": (pred, DUMP_PRED_ELEMS)}
    arrays.update({f"grad.{k}": (p.grad, DUMP_GRAD_ELEMS) for k, p in model.named_parameters() if p.grad is not None})
    host = {}
    for name, (t, cap) in arrays.items():
        a = t.detach()
        if a.numel() > cap:
            idx = torch.randint(0, a.numel(), (cap,), generator=torch.Generator().manual_seed(a.numel())).sort().values
            a = a.reshape(-1)[idx.to(a.device)]
        host[name] = a.float().cpu().numpy()
    total = sum(a.nbytes for a in host.values())
    assert total <= DUMP_MAX_BYTES, f"output dump of {total} bytes exceeds {DUMP_MAX_BYTES}"
    os.makedirs(out_dir, exist_ok=True)
    for name, a in host.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


# ==============================================================================================================
# our arm
# ==============================================================================================================
def run_ours(args):
    from swin_v2_weather_b200 import _lib, distributed as D
    rank, world, local = D.init_from_env()
    numa_bound = D.bind_to_gpu_numa_node(local) if os.environ.get("SWINB200_NUMA_BIND", "1") != "0" else False
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    _lib.load()
    peaks = read_peaks()
    B = args.batch_per_gpu

    config4 = args.workload == "config4"
    model = make_model(dev, args.mode, in_chans=77 if config4 else None, residual=config4)
    lossf = make_loss(dev, config4)
    static = None
    if config4:   # zenith angle per sample + batch-shared one-hot land mask (2) and standardised orography (1): channel groups,
        gs = torch.Generator().manual_seed(99)          # read in place by the PatchEmbed im2col (no 77-channel concatenation)
        lsm = torch.nn.functional.one_hot((torch.rand(720, 1440, generator=gs) > 0.7).long()).permute(2, 0, 1).float()[None]
        oro = torch.randn(1, 1, 720, 1440, generator=gs)
        static = torch.cat([lsm, (oro - oro.mean()) / (oro.std() + 1e-6)], dim=1).to(dev).contiguous()
    ddp = D.wrap_ddp(model, local)
    params = [p for p in model.parameters()]

    gen = torch.Generator().manual_seed(1234 + rank)
    host_x = torch.randn(B, 73, FIELD_ROWS, 1440, generator=gen).pin_memory()
    host_t = torch.randn(B, 73, FIELD_ROWS, 1440, generator=gen).pin_memory()
    x_res = host_x[:, :, :720].contiguous().to(dev)     # resident copies for the `value` leg (crop as the loaders do)
    t_res = host_t[:, :, :720].contiguous().to(dev)

    zen_res = (torch.rand(B, 1, 720, 1440, generator=gen) * 2 - 1).to(dev) if config4 else None
    last = {}                   # --dump-outputs: the latest step's loss and prediction

    def step(x, t, t_ready=None):
        for p in params:
            p.grad = None
        pred = ddp((x, zen_res, static)) if config4 else ddp(x)
        if t_ready is not None:     # the target is only needed by the loss: its host -> device copy may still run under the forward
            torch.cuda.current_stream().wait_event(t_ready)
        loss = lossf(pred, t, x)
        loss.backward()
        if args.dump_outputs:
            last.update(loss=loss, pred=pred)
        return loss

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    if args.profile_step:
        # one warmed-up step bracketed by cudaProfilerStart/Stop, for `ncu --profile-from-start off`
        step(x_res, t_res)
        torch.cuda.synchronize()
        torch.cuda.cudart().cudaProfilerStart()
        step(x_res, t_res)
        torch.cuda.synchronize()
        torch.cuda.cudart().cudaProfilerStop()
        return

    timer = KernelTimer()
    _lib.PROFILE_HOOK = timer.hook

    # ---- leg 1: inputs resident in HBM -------------------------------------------------------------------------
    for _ in range(args.warmup):
        step(x_res, t_res)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = _lib.LAUNCH_COUNT
    timer.enabled = True
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    barrier()
    ev[0].record()
    for _ in range(args.steps):
        step(x_res, t_res)
    ev[1].record()
    barrier()
    timer.enabled = False
    ms_total = D.max_over_ranks(ev[0].elapsed_time(ev[1]), dev)
    launches = _lib.LAUNCH_COUNT - launches0
    clocks = sampler.stop() if rank == 0 else None
    fam = timer.summary()
    peak_mem = torch.cuda.max_memory_allocated(dev) / 2 ** 30
    if args.dump_outputs and rank == 0:     # the gradients are all-reduced; the prediction is rank 0's sample
        dump_outputs(args.dump_outputs, last["loss"], last["pred"], model)

    # ---- leg 2: end to end from pinned host buffers (prefetch on a copy stream, double-buffered) ---------------
    from swin_v2_weather_b200.utils.host_io import copy_cropped_async
    copy_stream = torch.cuda.Stream(dev)
    bufs = [(torch.empty(B, 73, 720, 1440, device=dev), torch.empty(B, 73, 720, 1440, device=dev)) for _ in range(2)]
    ready = [torch.cuda.Event(enable_timing=True) for _ in range(2)]        # the step's target has landed (its input landed before)
    ready_x = [torch.cuda.Event() for _ in range(2)]                       # the step's input has landed
    copy_begin = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]
    h2d_bytes = 2 * B * 73 * 720 * 1440 * 4
    copy_ms = []          # duration of each step's host -> device copies, measured on the copy stream while the previous step runs

    def prefetch(i):
        slot = i % 2
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[slot])
            copy_begin[slot].record(copy_stream)
            dx, dt = bufs[slot]
            # crop [:720]: each plane's first 720 rows are one contiguous 4.1 MB run -> one strided copy per tensor
            copy_cropped_async(dx, host_x, copy_stream)
            ready_x[slot].record(copy_stream)
            copy_cropped_async(dt, host_t, copy_stream)
            ready[slot].record(copy_stream)

    loss_host = [torch.empty((), dtype=torch.float32).pin_memory() for _ in range(2)]
    # blocking events: the host thread sleeps while it waits for the previous step's loss instead of spinning on a core that the
    # other ranks' launch threads need (8 ranks share the node's CPUs)
    loss_ready = [torch.cuda.Event(blocking=True) for _ in range(2)]

    def e2e_loop(n):
        # Per step: wait for the step's inputs (copied host -> device on the copy stream while the previous step ran),
        # enqueue the NEXT step's copies (they run under this step), enqueue the step, then read the PREVIOUS step's loss on the host (async D2H into
        # pinned memory + event).  Every step's loss reaches the host inside the timed region; the host just does not
        # stall the launch queue waiting for it (the reference logs loss.item() per step, train.py:289-296).
        for s in range(2):
            consumed[s].record()
        prefetch(0)
        last = None
        for i in range(n):
            slot = i % 2
            if i >= 1 and ready[slot ^ 1].query():      # duration of step i-1's copies, before their events are recorded again
                copy_ms.append(copy_begin[slot ^ 1].elapsed_time(ready[slot ^ 1]))
            if i + 1 < n:       # next step's copies first: they only wait for the step before this one and run under this step
                prefetch(i + 1)
            torch.cuda.current_stream().wait_event(ready_x[slot])
            loss = step(*bufs[slot], t_ready=ready[slot])
            consumed[slot].record()
            loss_host[slot].copy_(loss.detach().reshape(()), non_blocking=True)
            loss_ready[slot].record()
            if i > 0:
                loss_ready[slot ^ 1].synchronize()
                last = float(loss_host[slot ^ 1])

        loss_ready[(n - 1) % 2].synchronize()
        last = float(loss_host[(n - 1) % 2])
        return last

    e2e_loop(max(2, min(args.warmup, 3)))
    barrier()
    ev2 = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev2[0].record()
    last_loss = e2e_loop(args.steps)
    ev2[1].record()
    barrier()
    ms_e2e = D.max_over_ranks(ev2[0].elapsed_time(ev2[1]), dev)
    _lib.PROFILE_HOOK = None

    if rank != 0:
        if world > 1:
            torch.distributed.barrier()
            torch.distributed.destroy_process_group()
        return

    samples = args.steps * B * world
    value = samples / (ms_total / 1e3)
    e2e_value = samples / (ms_e2e / 1e3)
    # dominant kernel family by device time inside the timed region
    dom = max(fam.items(), key=lambda kv: kv[1]["ms"]) if fam else ("none", dict(ms=0, flops=0, launches=1))
    gemm = fam.get("gemm_tcgen05")
    roof = None
    if gemm and gemm["ms"] > 0:
        achieved = gemm["flops"] / (gemm["ms"] / 1e3) / 1e12
        roof = {"kernel": "gemm_tc_kernel (tcgen05 bf16 GEMM family: qkv/proj/fc1/fc2/patch-embed/head fwd, dgrad, wgrad)",
                "bound": "tensor", "achieved": round(achieved, 1), "peak": peaks["tf_sust"], "unit": "TFLOP/s",
                "frac": round(achieved / peaks["tf_sust"], 4), "peak_source": f"{peaks['src']} sustained bf16 (kernel timed inside a long step)",
                # DRAM bytes per launch: ncu dram__bytes_read.sum + dram__bytes_write.sum averaged over the GEMM launches of one
                # step (tools/ncu_gemm_traffic.sh -> tools/traffic_summary.py -> profiles/gemm_traffic.json), next to the
                # algorithmic bytes per launch
                **gemm_traffic(B, args.mode),
                "algorithmic_bytes_per_launch": round(gemm["bytes"] / gemm["launches"], 1),
                "launches_per_step": gemm["launches"] / args.steps / 1.0,
                "avg_launch_ms": round(gemm["ms"] / gemm["launches"], 4), "flops_per_launch": gemm["flops"] / gemm["launches"],
                "share_of_step": round(gemm["ms"] / ms_total, 4)}
    families = {k: {"ms_per_step": round(v["ms"] / args.steps, 3), "launches_per_step": v["launches"] / args.steps}
                for k, v in sorted(fam.items(), key=lambda kv: -kv[1]["ms"])}
    # every GEMM template variant / shape on its own line, so a slow epilogue cannot hide inside the family average
    gemm_variants = {k: {"launches_per_step": v["launches"] / args.steps, "gflop": round(v["flops"] / v["launches"] / 1e9, 1),
                         "us": round(v["ms"] / v["launches"] * 1e3, 1), "tflops": round(v["flops"] / (v["ms"] / 1e3) / 1e12, 1),
                         "frac_of_sustained": round(v["flops"] / (v["ms"] / 1e3) / 1e12 / peaks["tf_sust"], 3)}
                     for k, v in sorted(timer.variants.items(), key=lambda kv: -kv[1]["ms"]) if v["ms"] > 0}
    # BASELINE metric, second half: attention as % of the tensor-core peak (and of its HBM roofline, which bounds it)
    attn = {}
    for key, nbytes in (("attn_fwd", 4 * T * 768 * 2), ("attn_bwd", 8 * T * 768 * 2)):
        a = fam.get(key)
        if a and a["ms"] > 0:
            tf = a["flops"] / (a["ms"] / 1e3) / 1e12
            gbs = nbytes * B * a["launches"] / (a["ms"] / 1e3) / 1e9
            attn[key] = {"us_per_launch": round(a["ms"] / a["launches"] * 1e3, 1), "tflops": round(tf, 1),
                         "pct_tc_peak_sustained": round(100 * tf / peaks["tf_sust"], 2), "pct_tc_peak_burst": round(100 * tf / peaks["tf_burst"], 2),
                         "hbm_gbs": round(gbs, 0), "frac_of_hbm_peak": round(gbs / peaks["hbm"], 3)}

    # ---- optimizer step, reported separately (SURVEY 8(d): "optimizer step reported separately"; 8(f) rank 1) ----------
    optimizer = None
    if world == 1:
        from swin_v2_weather_b200.functional import SHADOWS
        from swin_v2_weather_b200.optim import Adam
        inner = model.module if hasattr(model, "module") else model
        prm = [p for p in inner.parameters() if p.grad is not None]
        n_elem = sum(p.numel() for p in prm)
        n_shadow = sum(p.numel() for p in prm if SHADOWS.peek(p) is not None)

        def time_steps(opt, n=5):
            for _ in range(2):
                opt.step()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(n):
                opt.step()
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / n

        # lr = 0 keeps the benchmark weights unchanged while moving exactly the same bytes
        ours_ms = time_steps(Adam(prm, lr=0.0, betas=(0.9, 0.95)))
        torch_opt = torch.optim.Adam(prm, lr=0.0, betas=(0.9, 0.95), fused=True)
        torch_ms = time_steps(torch_opt)
        del torch_opt

        def recast():
            for p in prm:
                sh = SHADOWS.peek(p)
                if sh is not None:
                    from swin_v2_weather_b200 import ops as _ops
                    _ops.cast_bf16(p.detach(), sh)
        recast()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(5):
            recast()
        e1.record()
        torch.cuda.synchronize()
        recast_ms = e0.elapsed_time(e1) / 5
        alg_bytes = n_elem * 28 + n_shadow * 2
        optimizer = {"kernel": "adam_multi_kernel (fp32 masters + moments + bf16 shadows in one pass)", "ms": round(ours_ms, 3),
                     "bound": "hbm", "achieved_gbs": round(alg_bytes / ours_ms / 1e6, 1), "peak_gbs": peaks["hbm"],
                     "frac": round(alg_bytes / ours_ms / 1e6 / peaks["hbm"], 4), "algorithmic_bytes": alg_bytes,
                     "torch_fused_adam_ms": round(torch_ms, 3), "separate_shadow_recast_ms": round(recast_ms, 3),
                     "parameters": n_elem, "parameters_with_bf16_shadow": n_shadow,
                     "note": "not part of `value` (the metric is fwd+bwd); lr=0 so the timed weights do not move"}

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        cpu = cpu_reference_samples_per_s(steps=2, warmup=1)
    eager = None
    if world == 1 and not args.no_eager_baseline:
        del model, ddp, lossf, x_res, t_res, bufs
        torch.cuda.empty_cache()
        try:
            eager = gpu_eager_samples_per_s(dev, steps=3, warmup=1)
        except Exception as exc:   # the baseline must never take the main line down
            eager = {"error": f"{type(exc).__name__}: {exc}"[:300]}

    out = {
        "metric": "samples/s (fwd+bwd) 73ch 721x1440 SwinV2-d12", "value": round(value, 4), "unit": "samples/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms_total / args.steps, 3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16" if args.mode != "fp32" else "f32",
        "data": "synthetic N(0,1) 73x721x1440 fields cropped [:720]; random-init weights (norm1/2.weight ~ N(1,0.1))",
        "config": {"workload": ("swin_73var_geo_depth12 + conditioning (BASELINE config 4): 77 input channels as channel groups "
                                "(field 73 | zenith 1 | land mask 2 | orography 1), residual skip, 'weighted absolute temp-std squared "
                                f"geometric l2' loss with the 'auto' channel table, zero_grad + forward + loss + backward, batch {B}/GPU"
                                if config4 else
                                "swin_73var_geo_depth12: zero_grad + forward + 'squared geometric l2' loss + backward, "
                                f"batch {B}/GPU, C=768, 8 heads, window 9x18, 64,800 tokens/sample"),
                   "global_batch": B * world, "parallelism": f"dp{world}", "compute_mode": args.mode,
                   "l2_policy": "per-step working set (>= 19 GB of activations) is far larger than the 126 MB L2",
                   "attention_backend": "tcgen05" if ops_attn_is_tc(args.mode) else "cuda-core"},
        "clocks": clocks,
        "e2e": {"value": round(e2e_value, 4), "unit": "samples/s", "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 4,
                "ms_per_step": round(ms_e2e / args.steps, 3), "last_loss": last_loss, "numa_bound": bool(numa_bound),
                "h2d_copy_ms_per_step": round(statistics.median(copy_ms), 2) if copy_ms else None},
        "gpu_launches": launches,
        "roofline": roof,
        "kernel_families": families,
        "gemm_variants": gemm_variants,
        "attn_pct_tc_peak": attn,
        "gpu_eager_baseline": eager,
        "optimizer_step": optimizer,
        "model_tflops": round(value * FLOPS_FWD_BWD / 1e12 / world, 1),
        "model_frac_of_sustained_peak": round(value * FLOPS_FWD_BWD / 1e12 / world / peaks["tf_sust"], 4),
        "peak_mem_gib": round(peak_mem, 2),
        "cpu_baseline": cpu,
    }
    print(json.dumps(out), flush=True)
    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()


def ops_attn_is_tc(mode_name):
    from swin_v2_weather_b200 import ops
    return ops.MODES[mode_name].attn_backend == 1


# ==============================================================================================================
# reference arm / cpu baseline: the reference algorithm (oracle port) on the host CPU cores
# ==============================================================================================================
# The CPU sample: the FULL 12-block model on ten 72 x 144-pixel tiles of a 73-channel field (a batch of 10) = 10 x 4 = 40 of the
# 400 windows (6,480 of the 64,800 tokens) of a sample, same 9 x 18 windows and shift pattern.  Every operator of the path is
# per token or per window (PatchEmbed, LayerNorm, the MLP, window attention, head, loss rows), so one pass is exactly 1/10 of
# the work of one sample -- no intercept, no depth extrapolation -- and every timed step is the same real fwd + loss + bwd.
TILE = (72, 144)
TILES_PER_STEP = 10
BAND_FRACTION = TILES_PER_STEP * TILE[0] * TILE[1] / (720.0 * 1440.0)


def _band_problem(device="cpu"):
    from oracle import swinv2_oracle as O
    cfg = O.SwinConfig(**{**CFG, "img_size": TILE, "window_ratio": 8, "drop_path_rate": 0.0})
    assert cfg.window == (9, 18) and cfg.grid == (18, 36) and abs(BAND_FRACTION - 0.1) < 1e-12
    sd = {k: v.to(device) for k, v in O.init_state_dict(cfg, seed=0).items()}
    g = torch.Generator().manual_seed(1234)
    x = torch.randn(TILES_PER_STEP, 73, *TILE, generator=g).to(device)
    t = torch.randn(TILES_PER_STEP, 73, *TILE, generator=g).to(device)
    return O, cfg, sd, x, t, (torch.ones(73) / 73).to(device)


def _time_cpu_band(steps, warmup):
    """`steps` timed passes (after `warmup`) of the oracle on the band; returns (seconds per pass list, threads)."""
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    O, cfg, sd, x, t, chw = _band_problem()
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        O.loss_and_grads(x, t, sd, cfg, chw, relative=True)
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    return times, threads


CPU_SAMPLE = ("oracle (port of the reference algorithm, torch fp32 on the host cores): full 12-block model, fwd + 'squared geometric "
              "l2' loss + bwd, on ten 72x144-pixel tiles of a 73-channel field = 40 of the 400 windows of one sample; all "
              "operators are per token / per window, so one pass = 1/10 sample")


def cpu_reference_samples_per_s(steps=2, warmup=1):
    times, threads = _time_cpu_band(steps, warmup)
    sec = sum(times) / len(times)
    return {"value": round(BAND_FRACTION / sec, 5), "unit": "samples/s", "cores": threads, "kind": "port",
            "sample": CPU_SAMPLE + f"; {len(times)} timed passes of {sec:.2f} s after {warmup} warm-up"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warmup = max(1, args.steps), max(0, args.warmup)
    times, threads = _time_cpu_band(steps, warmup)
    total = sum(times)
    value = steps * BAND_FRACTION / total
    out = {"impl": "reference", "metric": "samples/s (fwd+bwd) 73ch 721x1440 SwinV2-d12", "value": round(value, 5),
           "unit": "samples/s", "n_gpus": args.gpus, "steps": steps, "warmup": warmup, "ms_per_step": round(total / steps * 1e3, 1),
           "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": "swin_73var_geo_depth12 fwd+loss+bwd on the host CPU; each step = 1/10 of a sample (ten 72x144 tiles = 40 "
                                  "windows, all 12 blocks)", "samples_per_step": BAND_FRACTION, "global_batch": 1, "parallelism": "cpu"},
           "step_seconds": [round(v, 3) for v in times],
           "cpu_baseline": {"value": round(value, 5), "unit": "samples/s", "cores": threads, "kind": "port", "sample": CPU_SAMPLE},
           "e2e": {"value": round(value, 5), "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out), flush=True)


def gpu_eager_samples_per_s(dev, steps=3, warmup=1):
    """The bar the reference itself would set on this GPU (SURVEY 8(d), BASELINE.md section 6): the same algorithm as plain
    eager PyTorch on the B200 under bf16 autocast -- the oracle port moved to the device (the reference tree does not exist
    on the GPU box), full 73x720x1440 sample, all 12 blocks, fwd + loss + bwd, CUDA-event timed."""
    from oracle import swinv2_oracle as O
    cfg = O.SwinConfig(**{**CFG, "drop_path_rate": 0.0})
    sd = {k: v.to(dev) for k, v in O.init_state_dict(cfg, seed=0).items()}
    g = torch.Generator().manual_seed(1234)
    x = torch.randn(1, 73, FIELD_ROWS, 1440, generator=g)[:, :, :720].contiguous().to(dev)
    t = torch.randn(1, 73, FIELD_ROWS, 1440, generator=g)[:, :, :720].contiguous().to(dev)
    chw = (torch.ones(73) / 73).to(dev)
    torch.cuda.reset_peak_memory_stats(dev)

    def one():
        with torch.autocast("cuda", dtype=torch.bfloat16):
            O.loss_and_grads(x, t, sd, cfg, chw, relative=True)

    for _ in range(warmup):
        one()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(dev)
    e0.record()
    for _ in range(steps):
        one()
    e1.record()
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / steps
    return {"value": round(1e3 / ms, 3), "unit": "samples/s", "ms_per_step": round(ms, 2), "steps": steps, "warmup": warmup,
            "kind": "oracle port, eager PyTorch on cuda under bf16 autocast (cuBLAS / cuDNN / ATen kernels, no kernels of this repo)",
            "peak_mem_gib": round(torch.cuda.max_memory_allocated(dev) / 2 ** 30, 1)}


def run_attn_sweep(args):
    """BASELINE config 5: windowed cosine attention (+ shift mask, with and without the CPB table) at 180 x 360 tokens, C = 768,
    over window sizes and head counts: forward + backward microseconds (CUDA events), achieved HBM GB/s on the algorithmic
    bytes (q, k, v, o read / written once forward; q, k, v, o, dO read and dq, dk, dv written backward) and % of the tensor peak
    on 4 / 10 nW h L^2 d FLOPs.  One JSON line per geometry; `backend` says which kernels ran."""
    from swin_v2_weather_b200 import _lib, ops
    from swin_v2_weather_b200._lib import BACKEND_TCGEN05
    _lib.load()
    peaks = read_peaks()
    dev = torch.device("cuda", 0)
    B, H, W, C = 1, 180, 360, 768
    T = B * H * W
    torch.manual_seed(0)
    qkv0 = torch.randn(T, 3 * C, device=dev).bfloat16()
    rows = []
    for window in ((9, 18), (6, 12), (12, 24), (18, 36)):
        for heads in (4, 8, 12, 16):
            for shift in ((0, 0), (window[0] // 2, window[1] // 2)):
                for cpb in (False, True):
                    L, d = window[0] * window[1], C // heads
                    rec = {"window": list(window), "heads": heads, "head_dim": d, "shifted": bool(shift[0]), "cpb": cpb}
                    try:
                        qkv = qkv0.clone()
                        inv = ops.qk_normalize_(qkv, C, heads)
                        scale = torch.full((heads,), 10.0, device=dev)
                        bias = (0.5 * torch.randn(heads, L, L, device=dev)) if cpb else None
                        be = ops.attn_backend_for(ops.MODE_BF16, C, heads, *window)
                        rec["backend"] = "tcgen05" if be == BACKEND_TCGEN05 else "cuda-core"
                        fwd = lambda: ops.window_attn_fwd(qkv, scale, bias, B, H, W, C, heads, window[0], window[1], shift[0], shift[1], ops.MODE_BF16)
                        o, lse = fwd()
                        d_o = torch.randn_like(o)
                        bwd = lambda: ops.window_attn_bwd(qkv, inv, scale, bias, o, d_o, lse, B, H, W, C, heads, window[0], window[1],
                                                          shift[0], shift[1], ops.MODE_BF16)
                        for name, fn, nbytes, nflop in (("fwd", fwd, 4 * T * C * 2, 4.0), ("bwd", bwd, 8 * T * C * 2, 10.0)):
                            for _ in range(max(1, args.warmup)):
                                fn()
                            ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
                            torch.cuda.synchronize()
                            ev[0].record()
                            for _ in range(args.steps):
                                fn()
                            ev[1].record()
                            torch.cuda.synchronize()
                            us = ev[0].elapsed_time(ev[1]) * 1e3 / args.steps
                            flops = nflop * (T // L) * heads * L * L * d
                            rec[name] = {"us": round(us, 1), "hbm_gbs": round(nbytes / us / 1e3, 0), "frac_of_hbm_peak": round(nbytes / us / 1e3 / peaks["hbm"], 3),
                                         "pct_tc_peak_sustained": round(100 * flops / us / 1e6 / peaks["tf_sust"], 2)}
                    except Exception as exc:
                        rec["error"] = f"{type(exc).__name__}: {exc}"[:200]
                    rows.append(rec)
                    print(json.dumps(rec), flush=True)
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "eager"])
    ap.add_argument("--mode", default="bf16", help="compute mode: bf16 | bf16_simt | fp32")
    ap.add_argument("--batch-per-gpu", type=int, default=1)
    ap.add_argument("--workload", default="headline", choices=["headline", "config4"],
                    help="headline = BASELINE configs[1] (the metric); config4 = conditioning inputs + channel-weighted temp-std loss")
    ap.add_argument("--sweep", default=None, choices=["attn"], help="attn: BASELINE config 5, the attention kernels over windows / head counts")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-eager-baseline", action="store_true")
    ap.add_argument("--profile-step", action="store_true", help="run one profiled step (for ncu) and exit")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps with resident inputs, write the last one's loss, prediction and parameter "
                         "gradients to DIR/*.npy (float32, large arrays as a fixed sample, <= 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.sweep or args.profile_step):
        ap.error("--dump-outputs applies to the timed steps of the default CUDA path")
    if args.sweep == "attn":
        run_attn_sweep(args)
    elif args.impl == "reference":
        run_reference(args)
    elif args.impl == "eager":
        print(json.dumps({"impl": "eager", **gpu_eager_samples_per_s(torch.device("cuda", 0), args.steps, args.warmup)}), flush=True)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
