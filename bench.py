#!/usr/bin/env python
"""bench.py -- denoising-UNet frames/sec of the CamAnimate denoising path on B200 (BASELINE.json configs 2-5).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config 2|3|4|5] [--impl native|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workloads (SURVEY.md 8d); default: config 2 on one GPU, config 4 under N > 1:
  config 2   1 clip, 24 frames of 768x576 (latent 96x72), CFG batch 2, no reference bank          96.30 TFLOP / step
  config 3   the same clip with the 16 ReferenceAttentionControl K/V banks                         105.71 TFLOP / step
  config 4   N independent config-3 clips, one per GPU, one final all-gather (weak scaling)        N x 105.71
  config 5   1 clip, 48 frames of 576x1024 (latent 72x128) = three 24-frame context windows per    3 x 152.11
             timestep, banks on; N > 1 splits the 6 (window x CFG-half) units over ranks (strong scaling)
A "step" is one per-timestep pass of the hot path for the clip(s): configs 2-4 one UNet3DConditionModel.forward on the
CFG-doubled batch; config 5 the three window forwards plus the on-device accumulate / CFG / DDIM glue.
value = frames of all clips / t_step.
--dump-outputs DIR writes what the last timed step returned as DIR/<name>.npy (float32); the inputs and weights are seeded, so two
builds run with the same arguments can be compared output for output.

  native arm     humanvid_b200 (hand-written sm_100a CUDA through the C ABI).  `value`: inputs resident in HBM, device time (CUDA
                 events) of K back-to-back steps, max over ranks.  `e2e`: the public Python call with the step's latents copied from
                 pinned host memory and the result read back to the host every step.  `oracle_gpu_eager`: the library bar -- the
                 reference-equivalent PyTorch path (the oracle) in fp16 eager on the same GPU and inputs.
  reference arm  (--impl reference) the oracle in fp32 on the host CPU cores, on a bounded sample of the same workload: 4 of the
                 step's frame-passes (2 frames x 2 CFG halves) at the full latent resolution, scaled linearly in frame-passes.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CH = (320, 640, 1280, 1280)
XDIM = 768
MM_KW = dict(num_attention_heads=8, num_transformer_block=1, attention_block_types=["Temporal_Self", "Temporal_Self"],
             temporal_position_encoding=True, temporal_position_encoding_max_len=32, temporal_attention_dim_div=1)
# frames of the clip, frames per window, latent h x w, banks, algorithmic TFLOP per UNet forward (SURVEY.md 8d), windows per step
CONFIGS = {
    2: dict(frames=24, fw=24, h=96, w=72, banks=False, tflop_fwd=96.30, windows=1, name="config2"),
    3: dict(frames=24, fw=24, h=96, w=72, banks=True, tflop_fwd=105.71, windows=1, name="config3"),
    4: dict(frames=24, fw=24, h=96, w=72, banks=True, tflop_fwd=105.71, windows=1, name="config4"),
    5: dict(frames=48, fw=24, h=72, w=128, banks=True, tflop_fwd=152.11, windows=3, name="config5"),
}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1421.9), d.get("bf16_tflops", 1668.4), d.get("hbm_gbs", 6586.4), "measured"
    return 1400.0, 1590.0, 6650.0, "fallback"


def measured_traffic():
    """DRAM bytes per launch of the dominant kernel family from the committed ncu pass of this command (profiles/)."""
    p = os.path.join(ROOT, "profiles", "r02_dram_traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p))
        except Exception:
            return None
    return None


def synthetic_init_(module, seed, device):
    """Seeded variance-controlled random init written straight on the device (no checkpoints exist offline; the
    reference's zero-inits are overridden so every branch does real work)."""
    import math

    import torch

    g = torch.Generator(device=device).manual_seed(seed)
    with torch.no_grad():
        for name, p in sorted(module.named_parameters()):
            if p.ndim >= 2:
                std = 1.0 / math.sqrt(p[0].numel())
                if any(k in name for k in ("conv2.", "to_out.0.", "ff.net.2.", "proj_out.", "block2.", "zero_conv")):
                    std *= 0.5
                p.copy_((torch.randn(p.shape, generator=g, device=device) * std).to(p.dtype))
            elif name.endswith("bias"):
                p.copy_((torch.randn(p.shape, generator=g, device=device) * 0.02).to(p.dtype))
            else:
                p.copy_((1.0 + 0.1 * torch.randn(p.shape, generator=g, device=device)).to(p.dtype))


class ClockSampler:
    def __init__(self, gpu_index):
        self.idx, self.rows, self.stop = gpu_index, [], threading.Event()
        self.th = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self.stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.idx)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self.stop.wait(0.2)

    def __enter__(self):
        self.th.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.th.join(timeout=3)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit())
        reasons = []
        for i, n in enumerate(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]):
            if any(len(r) > 3 + i and r[3 + i].lower().startswith("active") for r in self.rows):
                reasons.append(n)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": float(self.rows[0][1]) if self.rows[0][1].replace(".", "").isdigit() else None,
                "power_w_max": max((float(r[2]) for r in self.rows if r[2].replace(".", "").isdigit()), default=None), "reasons": reasons,
                "samples": len(self.rows)}


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(dirname, arrays):
    """Writes each tensor as dirname/<name>.npy in float32.  Every bench workload returns a few MB, well inside DUMP_LIMIT_BYTES."""
    import numpy as np

    total = sum(a.numel() * 4 for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise RuntimeError(f"outputs of {total} bytes exceed the {DUMP_LIMIT_BYTES}-byte dump limit")
    os.makedirs(dirname, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(dirname, name + ".npy"), a.detach().float().cpu().numpy())


# ------------------------------------------------------------------------------------------------ reference / CPU arm
def cpu_threads():
    """Pinned (not probed) thread count for the CPU arm, so that repeated runs time the same thing: the CPUs this process may use
    (affinity mask, cgroup quota), halved on large SMT boxes, capped at 64 -- more threads have run the oracle up to 20x SLOWER on
    the GPU boxes (OpenMP oversubscription), and a per-run probe made the round-1 baseline wander 3.3x."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except AttributeError:
        pass
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(int(q) / int(per))))
    except Exception:
        pass
    return max(1, min(64, n // 2 if n > 16 else n))


def cpu_reference_sample(cfg, samples=3, warmup=1, frames=2, cfg_batch=2):
    """Oracle (reference-equivalent PyTorch, fp32) on the host cores.  One sample = a UNet forward over `frames` frames of
    `cfg_batch` CFG halves at the config's full latent (and with its reference banks): frames * cfg_batch of the step's
    2 * fw * windows frame-passes.  frames/s counts a video frame as its CFG pair of passes, like the native arm."""
    import torch

    from oracle import hv_oracle as O

    nthreads = cpu_threads()
    torch.set_num_threads(nthreads)
    torch.set_flush_denormal(True)   # random-init activations reach denormals in places; the x86 slow path would understate the CPU
    H, W = cfg["h"], cfg["w"]
    m = O.UNet3DConditionModel(block_out_channels=CH, cross_attention_dim=XDIM).eval()
    synthetic_init_(m, 7, "cpu")
    g = torch.Generator().manual_seed(1)
    x = torch.randn(cfg_batch, 4, frames, H, W, generator=g)
    ehs = torch.randn(cfg_batch, 1, XDIM, generator=g)
    ehs[: cfg_batch // 2] = 0
    pose = torch.randn(cfg_batch, CH[0], frames, H, W, generator=g) * 0.5
    if cfg["banks"]:
        O.set_reference_banks(m, [torch.randn(cfg_batch, l, c, generator=g) for (l, c) in O.bank_shapes(m, H, W)], cfg=cfg_batch > 1)
    times = []
    with torch.no_grad():
        for i in range(warmup + samples):
            t0 = time.perf_counter()
            y = m(x, torch.tensor(500), ehs, pose_cond_fea=pose)[0]
            dt = time.perf_counter() - t0
            if i >= warmup:
                times.append(dt)
    t = statistics.median(times)
    passes = frames * cfg_batch
    # the step's windows overlap, so the clip's frames cost windows * fw * 2 passes per step
    passes_per_step = 2 * cfg["fw"] * cfg["windows"]
    fps = cfg["frames"] / (t * passes_per_step / passes)
    return {"output": y, "frames_per_s": fps, "s_per_sample": t, "cores": nthreads, "spread": (max(times) - min(times)) / t if len(times) > 1 else 0.0,
            "sample": f"oracle UNet forward (fp32, {nthreads} threads pinned by rule, denormals flushed) on {passes} of the step's {passes_per_step} "
                      f"frame-passes ({frames} frames x {cfg_batch} CFG halves) at the full {H}x{W} latent{' with the 16 reference banks' if cfg['banks'] else ''}; "
                      f"median of {len(times)} timed samples after {warmup} warm-up: {t:.1f} s (min {min(times):.1f}, max {max(times):.1f}); "
                      f"frames/s = {cfg['frames']} / (t * {passes_per_step} / {passes})"}


def workload_name(cfg, world):
    banks = ", 16 reference K/V banks" if cfg["banks"] else ", no reference bank"
    if cfg["name"] == "config5":
        return (f"config5: 1 clip x 48 frames 576x1024 (latent 72x128), 3 context windows of 24 frames per timestep (context.py), CFG batch 2{banks}, "
                f"random-init UNet3D 1.31B params" + (f"; the 6 (window x CFG-half) units split over {world} GPUs" if world > 1 else ""))
    per = "1 clip/GPU" if world > 1 else "1 clip"
    if cfg.get("single_clip"):
        per = f"ONE clip, its 2 CFG halves split over {world} GPUs (ranks beyond 2 idle),"
    return f"{cfg['name']}: {per} x 24 frames 768x576 (latent 96x72), CFG batch 2, random-init UNet3D 1.31B params{banks}"


def run_reference(args, rank, cfg):
    if rank != 0:
        return
    r = cpu_reference_sample(cfg, samples=args.steps, warmup=min(max(args.warmup, 0), 1))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"noise_pred": r["output"]})
    line = {"metric": "denoising-UNet frames/sec, 24x768x576, CFG", "value": r["frames_per_s"], "unit": "frames/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * cfg["frames"] / r["frames_per_s"], "higher_is_better": True,
            "scaling": "strong" if cfg["name"] == "config5" else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "reference",
            "config": {"workload": workload_name(cfg, 1),
                       "note": "reference = oracle restatement of the reference PyTorch path on the host CPU (diffusers not installable offline); "
                               "bounded sample scaled linearly in frame-passes"},
            "cpu_baseline": {"value": r["frames_per_s"], "unit": "frames/s", "cores": r["cores"], "kind": "port", "sample": r["sample"],
                             "run_to_run_spread": r["spread"]},
            "e2e": {"value": r["frames_per_s"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ native arm
def build_native(dev):
    import torch

    import humanvid_b200 as hv

    unet = hv.UNet3DConditionModel(block_out_channels=CH, cross_attention_dim=XDIM, use_motion_module=True, use_inflated_groupnorm=True,
                                   motion_module_resolutions=(1, 2, 4, 8), motion_module_mid_block=True, motion_module_type="Vanilla",
                                   motion_module_kwargs=MM_KW, unet_use_cross_frame_attention=False, unet_use_temporal_attention=False)
    unet = unet.to(dev, torch.float16)
    synthetic_init_(unet, 7, dev)
    unet.refresh_native()
    return unet


def time_oracle_eager(dev, x, ehs, pose, banks, native_ms, n=5):
    """The library bar (SURVEY 6 / BASELINE.md 4): the reference-equivalent PyTorch path in fp16 eager (cuDNN / cuBLAS / SDPA of
    torch 2.11) on the same B200, weights and inputs; CUDA-event median of n forwards after 2 warm-ups."""
    import torch

    from oracle import hv_oracle as O

    ora = O.UNet3DConditionModel(block_out_channels=CH, cross_attention_dim=XDIM).eval().to(dev, torch.float16)
    synthetic_init_(ora, 7, dev)
    if banks is not None:
        O.set_reference_banks(ora, banks, cfg=True)
    ts = []
    with torch.no_grad():
        for i in range(2 + n):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            y = ora(x, torch.tensor(500, device=dev), ehs, pose_cond_fea=pose)[0]
            e1.record()
            torch.cuda.synchronize()
            if i >= 2:
                ts.append(e0.elapsed_time(e1))
    ok = bool(torch.isfinite(y).all())
    del ora
    torch.cuda.empty_cache()
    ms = statistics.median(ts)
    return {"ms_per_forward": ms, "min_ms": min(ts), "max_ms": max(ts), "samples": n, "finite": ok, "native_ms_per_forward": native_ms,
            "native_speedup": ms / native_ms,
            "how": "oracle/hv_oracle.py UNet3DConditionModel (the reference's modules restated with plain torch ops; F.scaled_dot_product_attention, "
                   "nn.Conv2d, nn.Linear, nn.GroupNorm) in fp16 eager on the same GPU, same seeded weights and inputs as the native arm; CUDA events, "
                   f"median of {n} after 2 warm-ups"}


def time_cond_branches(dev, hbm_gbs, n=5):
    """PoseGuider (pose_guider.py:51-61) and CameraPoseEncoder (pose_adaptor.py:232-248) at the (1, ., 24, 768, 576) input of configs 2-4: the
    step-invariant conditioning branches the pipeline runs once per context window.  PoseGuider is HBM-bound small-channel convolution work:
    achieved GB/s on its ALGORITHMIC bytes (every conv reads its input and writes its output once at the true channel counts)."""
    import torch

    import humanvid_b200 as hv

    F_, H_, W_ = 24, 768, 576
    pg = hv.PoseGuider(320, block_out_channels=(16, 32, 96, 256)).to(dev, torch.float16)
    synthetic_init_(pg, 11, dev)
    pg.refresh_native()
    cam = hv.CameraPoseEncoder(downscale_factor=8, channels=[320], nums_rb=2, cin=384, ksize=1, sk=True, use_conv=False, compression_factor=1,
                               temporal_attention_nhead=8, attention_block_types=["Temporal_Self"], temporal_position_encoding=True,
                               temporal_position_encoding_max_len=24).to(dev, torch.float16)
    synthetic_init_(cam, 13, dev)
    cam.refresh_native()
    g = torch.Generator(device=dev).manual_seed(5)
    img = torch.rand(1, 3, F_, H_, W_, generator=g, device=dev).half()
    pl = torch.randn(1, 6, F_, H_, W_, generator=g, device=dev).half()
    K = torch.tensor([[[1.788079 * W_ * H_ / W_, 1.788079 * H_, 0.5 * W_, 0.5 * H_]]], device=dev).repeat(1, F_, 1)
    c2w = torch.eye(4, device=dev).repeat(1, F_, 1, 1)

    def timed(fn):
        ts = []
        for i in range(2 + n):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            if i >= 2:
                ts.append(e0.elapsed_time(e1))
        return statistics.median(ts)

    px = F_ * H_ * W_
    chans = [(3, 16, 1), (16, 16, 1), (16, 32, 2), (32, 32, 1), (32, 96, 2), (96, 96, 1), (96, 256, 2), (256, 320, 1)]
    nbytes, p = 0, px
    for cin, cout, st in chans:
        nbytes += p * cin * 2
        p //= st * st
        nbytes += p * cout * 2
    t_pg, t_cam, t_rays = timed(lambda: pg(img)), timed(lambda: cam(pl)), timed(lambda: cam.forward_cameras(K, c2w, H_, W_))
    return {"shape": "(1, ., 24, 768, 576)",
            "pose_guider": {"ms": t_pg, "algorithmic_gb": nbytes / 1e9, "gbs": nbytes / 1e6 / t_pg, "frac_of_hbm_peak": nbytes / 1e6 / t_pg / hbm_gbs,
                            "launches": pg.last_launch_count,
                            "note": "conv_in reads the planar image directly (mma.sync implicit GEMM, K = 27 -> 32); the 16/32-channel layers run at their true channel counts on "
                                    "the mma.sync small-channel kernel, the last three (96 -> 96 -> 256 -> 320 at <= 1/4 resolution) on the tcgen05 implicit GEMM"},
            "camera_encoder": {"ms": t_cam, "tflop": 2.18, "tflops": 2.18e3 / t_cam, "launches": cam.last_launch_count},
            "camera_encoder_from_cameras": {"ms": t_rays, "note": "Plucker embedding generated on the device inside the PixelUnshuffle producer (SURVEY 8f-3); "
                                            "the 127 MB (1,6,24,768,576) embedding is never built or copied"}}


def time_pipeline_clip(dev, unet, steps=25):
    """The real 25-step Pose2VideoPipeline call (on-device step glue, one CUDA graph per step) with stand-in VAE / CLIP modules (the reference's
    stay PyTorch and are out of scope) and a native writer UNet: clip latency for one 24-frame 768x576 clip."""
    import torch
    import torch.nn as nn
    import torch.nn.functional as Fn
    from types import SimpleNamespace

    import humanvid_b200 as hv
    from humanvid_b200.pipeline import Pose2VideoPipeline

    class StubVAE(nn.Module):
        def __init__(self):
            super().__init__()
            self.conv = nn.Conv2d(3, 4, 8, stride=8)
            self.config = SimpleNamespace(block_out_channels=(1, 2, 3, 4))

        def encode(self, x):
            return SimpleNamespace(latent_dist=SimpleNamespace(mean=self.conv(x)))

        def decode(self, z):
            return SimpleNamespace(sample=Fn.interpolate(z[:, :3], scale_factor=8.0))

    class StubCLIP(nn.Module):
        def __init__(self, dim):
            super().__init__()
            self.lin = nn.Linear(3, dim)

        def forward(self, pix):
            return SimpleNamespace(image_embeds=self.lin(pix.float().mean((2, 3)).to(self.lin.weight.dtype)))

    H_, W_, F_ = 768, 576, 24
    ref_unet = hv.UNet2DConditionModel(block_out_channels=CH, cross_attention_dim=XDIM).to(dev, torch.float16)
    synthetic_init_(ref_unet, 17, dev)
    ref_unet.refresh_native()
    pg = hv.PoseGuider(320, block_out_channels=(16, 32, 96, 256)).to(dev, torch.float16)
    synthetic_init_(pg, 11, dev)
    pg.refresh_native()
    cam = hv.CameraPoseEncoder(downscale_factor=8, channels=[320], nums_rb=2, cin=384, ksize=1, sk=True, use_conv=False, compression_factor=1,
                               temporal_attention_nhead=8, attention_block_types=["Temporal_Self"], temporal_position_encoding=True,
                               temporal_position_encoding_max_len=24).to(dev, torch.float16)
    synthetic_init_(cam, 13, dev)
    cam.refresh_native()
    pipe = Pose2VideoPipeline(vae=StubVAE().half().to(dev), image_encoder=StubCLIP(XDIM).half().to(dev), reference_unet=ref_unet, denoising_unet=unet,
                              pose_guider=pg, camera_pose_encoder=cam, scheduler=hv.DDIMScheduler()).to(dev, torch.float16)
    g = torch.Generator(device=dev).manual_seed(3)
    ref = torch.rand(3, H_, W_, generator=g, device=dev) * 2 - 1
    poses = [torch.rand(1, 3, H_, W_, generator=g, device=dev) for _ in range(F_)]
    camera = torch.randn(1, 6, F_, H_, W_, generator=g, device=dev).half()
    out = {}
    for label, n_steps in (("warmup", 2), ("first", steps), ("next", steps)):
        gen = torch.Generator(device=dev).manual_seed(42)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        lat = pipe(ref, poses, camera, W_, H_, F_, n_steps, 3.5, generator=gen, output_type="latent", return_dict=False)
        torch.cuda.synchronize()
        out[label] = time.perf_counter() - t0
    ok = bool(torch.isfinite(lat).all())
    del pipe, ref_unet, pg, cam
    torch.cuda.empty_cache()
    return {"steps": steps, "latency_s": out["next"], "first_clip_latency_s": out["first"], "frames_per_s_per_clip": F_ / out["next"],
            "denoise_frames_per_s": F_ * steps / out["next"], "finite": ok,
            "what": "humanvid_b200.pipeline.Pose2VideoPipeline.__call__ -> latents: CLIP/VAE stand-ins, native writer UNet2D once, PoseGuider + CameraPoseEncoder once, "
                    f"{steps} DDIM steps as {steps} replays of one captured CUDA graph (window gather + UNet forward with reference banks + accumulate/CFG/DDIM kernel). "
                    "first_clip_latency_s includes the warm-up step and the graph capture; latency_s is the next clip of the same shape, which reuses the captured step"}


HBM_WRITE_GBS = 3924.0   # write-only ceiling of this pool's B200 (profiles/r02_hbm_ceilings.txt, scripts/write_bw.py); reads: MEASURED_PEAKS hbm_gbs


def gemm_classes(trace_path, tensor_peak, hbm_peak):
    """Scores every launch of the dominant kernel family (gemm_kernel: linears, 1x1 / 3x3 / sub-pixel convs, V^T) against ITS OWN roofline:
    t_tensor = FLOPs / sustained tensor peak, t_hbm = compulsory reads / read bandwidth + compulsory writes / write-only bandwidth (fp16; A read
    once, residual read once, output written once; weights stay in L2).  The larger of the two is the launch's bound; launches are grouped by which
    one it is.  `frac_of_shape_roofline` = sum of the bounds / sum of the measured times over all launches."""
    import csv

    try:
        rows = list(csv.DictReader(open(trace_path)))
    except Exception:
        return None
    cls = {"tensor_bound": [0, 0.0, 0.0, 0.0, 0.0], "hbm_bound": [0, 0.0, 0.0, 0.0, 0.0]}   # launches, ms, bound ms, flops, bytes
    for r in rows:
        lb = r["label"]
        if int(r["cat"]) not in (0, 1) or not lb:
            continue
        M, Nn, K, ms = float(r["M"]), float(r["N"]), float(r["K"]), float(r["ms"])
        fl = 2 * M * Nn * K
        if lb == "gemm_vt":            # out[M rows][N tokens] = W[M][K] . X[N][K]^T
            rd, wr = 2 * Nn * K, 2 * M * Nn
        elif lb.startswith("conv3") or lb.startswith("upconv"):
            taps = 4 if lb.startswith("upconv") else 9
            rows_in = M / 4 if lb.startswith("upconv") else (M * 4 if lb.endswith("_s2") else M)
            rd, wr = 2 * (rows_in * K / taps + (M * Nn if lb.endswith("_res") else 0)), 2 * M * Nn
        else:
            n_out = Nn / 2 if lb == "gemm_geglu" else Nn
            rd, wr = 2 * (M * K + (M * n_out if lb == "gemm_res" else 0)), 2 * M * n_out
        t_tensor = fl / (tensor_peak * 1e9)                       # ms
        t_hbm = rd / (hbm_peak * 1e6) + wr / (HBM_WRITE_GBS * 1e6)
        c = cls["hbm_bound" if t_hbm > t_tensor else "tensor_bound"]
        c[0] += 1; c[1] += ms; c[2] += max(t_tensor, t_hbm); c[3] += fl; c[4] += rd + wr
    t, h = cls["tensor_bound"], cls["hbm_bound"]
    tot_ms, tot_bound = t[1] + h[1], t[2] + h[2]
    return {"hbm_read_gbs": hbm_peak, "hbm_write_gbs": HBM_WRITE_GBS, "hbm_write_source": "profiles/r02_hbm_ceilings.txt (scripts/write_bw.py, measured on this pool)",
            "frac_of_shape_roofline": tot_bound / tot_ms if tot_ms else None,
            "tensor_bound": {"launches": t[0], "ms": t[1], "bound_ms": t[2], "tflops": t[3] / 1e9 / t[1] if t[1] else None, "frac": t[2] / t[1] if t[1] else None},
            "hbm_bound": {"launches": h[0], "ms": h[1], "bound_ms": h[2], "gbs": h[4] / 1e6 / h[1] if h[1] else None, "tflops": h[3] / 1e9 / h[1] if h[1] else None,
                          "frac": h[2] / h[1] if h[1] else None}}


def run_native(args, rank, world, local_rank, cfg):
    import ctypes as C

    import torch

    import humanvid_b200 as hv
    from humanvid_b200 import _native as N
    from humanvid_b200.device_loop import DeviceDenoiseLoop
    from humanvid_b200.distributed import UnitExchange, gather_clip_latents, unit_list
    from humanvid_b200.pipeline import uniform

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)

    # one clip over all ranks (strong scaling): config 5 always; configs 2 / 3 with --single-clip (1 window x 2 CFG halves = the 2-GPU CFG split)
    is5 = cfg["name"] == "config5" or (args.single_clip and world > 1)
    F, Fw, H, W = cfg["frames"], cfg["fw"], cfg["h"], cfg["w"]
    unet = build_native(dev)
    # config 5 is ONE clip (same data on every rank); configs 2-4 are one clip per rank (seed 42 + rank)
    g = torch.Generator(device=dev).manual_seed(42 if is5 else 42 + rank)
    B = 2
    ehs = torch.randn(B, 1, XDIM, generator=g, device=dev).half()
    ehs[:1] = 0
    banks = None
    if cfg["banks"]:
        hv.ReferenceAttentionControl(unet, do_classifier_free_guidance=True, mode="read", fusion_blocks="full")
        lv = {320: H * W, 640: (H // 2) * (W // 2), 1280: (H // 4) * (W // 4)}
        names = {id(m): n for n, m in unet.named_modules()}
        banks = []
        for blk in unet.reader_blocks():
            c = blk.norm1.normalized_shape[0]
            L = (H // 8) * (W // 8) if names[id(blk)].startswith("mid_block") else lv[c]
            blk.bank = [torch.randn(B, L, c, generator=g, device=dev).half()]
            banks.append(blk.bank[0])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    windows = list(uniform(0, 25, F, Fw, 1, 4))
    assert len(windows) == cfg["windows"]
    sample = torch.randn(B, 4, Fw, H, W, generator=g, device=dev).half()          # one window's CFG-doubled UNet input
    poses = [(torch.randn(1, CH[0], Fw, H, W, generator=g, device=dev) * 0.5).half().repeat(2, 1, 1, 1, 1) for _ in windows]
    loop = None
    if is5:
        latents = torch.randn(1, 4, F, H, W, generator=g, device=dev).half()
        sched = hv.DDIMScheduler()
        sched.set_timesteps(max(args.steps, args.warmup, 3) + 1)
        kw = {}
        if world > 1:
            ex = UnitExchange(unit_list(len(windows), True))
            kw = dict(exchange=ex, my_units=ex.my_units, all_units=ex.units)
        loop = DeviceDenoiseLoop(unet, sched, latents, windows, ehs, poses, 3.5, True, **kw)
        lat0 = loop.latents.clone()

        def reset():
            loop.latents.copy_(lat0)
            loop.step_index.zero_()

        def step():
            loop._one_step()
            return loop.latents
    else:
        def reset():
            pass

        def step():
            return unet(sample, 500, ehs, pose_cond_fea=poses[0], return_dict=False)[0]

    for _ in range(max(args.warmup, 3)):
        out = step()
    torch.cuda.synchronize()
    if not torch.isfinite(out).all():
        raise RuntimeError("non-finite output")
    launches_fwd = unet.last_launch_count
    n_fwd = (len(loop.my_units) if (is5 and world > 1) else len(windows)) if is5 else 1
    launches_step = launches_fwd * n_fwd + ((n_fwd + 2) if is5 else 0)

    # ---- (N > 1) the same per-GPU workload on rank 0 ALONE, the other GPUs idle: the single-GPU reference point of THIS workload (no ratio is reported: the driver computes scaling itself)
    # (the default N = 1 run is config 2, the N > 1 runs are config 4 = N x config 3, which has 10 % more work per GPU)
    solo_ms = None
    if world > 1:
        reset()
        barrier()
        if rank == 0:
            s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s0.record()
            for _ in range(args.steps):
                if is5:   # one clip: the step's window forwards at the full CFG batch on this GPU alone (the N = 1 run minus its ~0.1 ms of glue)
                    for wi in range(len(windows)):
                        unet(sample, 500, ehs, pose_cond_fea=poses[wi], return_dict=False)
                else:
                    out = step()
            s1.record()
            torch.cuda.synchronize()
            solo_ms = s0.elapsed_time(s1) / args.steps
        barrier()

    # ---- kernel-only: inputs resident, K steps bracketed by barrier + synchronize, device-timed
    reset()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    with ClockSampler(local_rank) as cs:
        e0.record()
        for _ in range(args.steps):
            out = step()
        if world > 1 and not is5:
            gathered = gather_clip_latents(out[1:2].contiguous())   # config 4's single collective: reassemble the clips' latent-sized results
        e1.record()
        barrier()
    ms = e0.elapsed_time(e1) / args.steps
    clocks = cs.summary()
    if args.dump_outputs and rank == 0:
        # now, before the end-to-end loop below runs the same step again into the same buffers
        dumped = {"latents": out} if is5 else {"noise_pred": out}
        if world > 1 and not is5:
            dumped["gathered_noise_pred_cond"] = gathered
        dump_outputs(args.dump_outputs, dumped)

    # ---- end to end: the step's latents come from pinned host memory, the result goes back to the host
    src = loop.latents if is5 else sample
    h_in = torch.empty(src.shape, dtype=torch.float16).pin_memory()
    h_in.copy_(lat0.cpu() if is5 else sample.cpu())
    h_out = torch.empty(out.shape, dtype=torch.float16).pin_memory()
    reset()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        if is5:
            loop.latents.copy_(h_in, non_blocking=True)
            o = step()
        else:
            d_in = h_in.to(dev, non_blocking=True)
            o = unet(d_in, 500, ehs, pose_cond_fea=poses[0], return_dict=False)[0]
        h_out.copy_(o, non_blocking=True)
        torch.cuda.current_stream().synchronize()
    barrier()
    e2e_ms = (time.perf_counter() - t0) * 1000.0 / args.steps

    t = torch.tensor([ms, e2e_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, e2e_ms = float(t[0]), float(t[1])
    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    # ---- per-operator device time of one more UNet forward (events around every launch) -> roofline of the dominant kernel
    lib = N.lib()
    lib.hv_set_profiling(unet._handle, 1)
    if is5:
        loop.close()   # host timestep again
    x1 = sample
    if is5 and world > 1:   # a one-half unit, what this rank actually runs
        unet._forward_flags = 4
        unet(x1[1:], 500, ehs[1:], pose_cond_fea=poses[0][1:], return_dict=False)
        unet._forward_flags = None
    else:
        unet(x1, 500, ehs, pose_cond_fea=poses[0], return_dict=False)
    cat_ms, cat_fl, cat_n = (C.c_double * 6)(), (C.c_double * 6)(), (C.c_int64 * 6)()
    N.check(lib.hv_get_profile(unet._handle, cat_ms, cat_fl, cat_n, 6), unet._handle)
    trace_path = os.environ.get("HV_TRACE") or os.path.join("/tmp", f"hv_trace_{os.getpid()}.csv")
    lib.hv_dump_profile(unet._handle, trace_path.encode())
    lib.hv_set_profiling(unet._handle, 0)
    classes = gemm_classes(trace_path, *peaks()[:1], peaks()[2])
    names = ["tcgen05_gemm_linear", "tcgen05_implicit_gemm_conv3x3", "tcgen05_spatial_attention", "temporal_attention", "norms", "small_linear"]
    prof = {names[i]: {"ms": round(cat_ms[i], 3), "tflop": round(cat_fl[i] / 1e12, 3), "launches": int(cat_n[i]),
                       "tflops": round(cat_fl[i] / 1e9 / cat_ms[i], 1) if cat_ms[i] > 0 else None} for i in range(6)}
    sustained, burst, hbm, src_pk = peaks()
    gemm_ms, gemm_fl = cat_ms[0] + cat_ms[1], cat_fl[0] + cat_fl[1]
    gemm_n = int(cat_n[0] + cat_n[1])
    achieved = gemm_fl / 1e9 / gemm_ms if gemm_ms > 0 else 0.0
    executed_fl = sum(cat_fl[i] for i in range(6))   # counted by the runtime from the unpadded shapes of what it launched

    # ---- the library bar: the oracle in fp16 eager on this GPU, same inputs (one UNet forward)
    eager = None
    if not args.no_eager:
        torch.cuda.synchronize()
        if not (is5 and world > 1):   # (the unit split has no single-GPU forward to compare with)
            eager = time_oracle_eager(dev, sample, ehs, poses[0], banks, ms / len(windows) if is5 else ms)
    extras = {}
    if not args.no_extras and world == 1 and not is5:
        torch.cuda.synchronize()
        extras["cond_branches"] = time_cond_branches(dev, hbm)
        extras["pipeline_clip"] = time_pipeline_clip(dev, unet)
    cpu = cpu_reference_sample(cfg, samples=2 if args.quick_cpu else 3) if not args.no_cpu_baseline else None

    frames_total = F if is5 else world * F
    flops_step = cfg["tflop_fwd"] * 1e12 * (len(windows) if is5 else world)
    # executed = what the runtime launched, counted from the unpadded shapes of one profiled forward (rank 0's): the algorithmic count minus attn2's
    # to_q / to_out over all tokens (one-key cross-attention collapse, -2.07 TF at config 2) and minus 5/9 of the upsampler convs (sub-pixel form)
    n_fwd_total = (len(windows) if is5 else world)
    exec_step = executed_fl * n_fwd_total * (2.0 if (is5 and world > 1) else 1.0)   # (a profiled one-half unit is half a window forward)
    value = frames_total / (ms / 1000.0)
    traffic = measured_traffic()
    line = {
        "metric": "denoising-UNet frames/sec, 24x768x576, CFG", "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True, "scaling": "strong" if is5 else "weak", "vs_baseline": None,
        "dtype": "f16", "data": "synthetic", "impl": "native",
        "config": {"workload": workload_name(cfg, world), "global_batch_clips": 1 if is5 else world,
                   "parallelism": (f"(window x CFG-half) units over {world} ranks, one all_gather of unit predictions per step" if (is5 and world > 1)
                                   else f"clip-per-gpu x{world}" + (", final all_gather of predictions" if world > 1 else "")),
                   "l2": "working set per step (2.6 GB weights + multi-GB activations) >> 126 MB L2, no flush needed",
                   "cond_features": "pose_cond_fea resident (step-invariant; hoisted out of the step as the pipeline's feature cache does)"},
        "tflops_per_step": flops_step / 1e12, "executed_tflops_per_step": exec_step / 1e12,
        "achieved_tflops": exec_step / 1e9 / ms, "frac_of_tensor_roofline_sustained": exec_step / 1e9 / ms / sustained / world,
        "algorithmic_tflops": flops_step / 1e9 / ms,
        "flops_note": "tflops_per_step = algorithmic FLOPs of the reference's arithmetic (SURVEY 8d); executed = counted by the runtime from the shapes it launched: "
                      "no attn2 to_q/to_out over all tokens (one-key cross-attention collapse) and 4/9 of the upsampler-conv multiply-adds (sub-pixel form); "
                      "achieved_tflops and frac_of_tensor_roofline_sustained are on EXECUTED FLOPs",
        "e2e": {"value": frames_total / (e2e_ms / 1000.0), "unit": "frames/s", "ms_per_step": e2e_ms, "h2d_bytes_per_step": int(h_in.numel() * 2),
                "d2h_bytes_per_step": int(h_out.numel() * 2),
                "api": (f"humanvid_b200.device_loop.DeviceDenoiseLoop step (host latents -> {len(windows)} window forward(s) + glue -> host latents)" if is5 else
                        "humanvid_b200.UNet3DConditionModel.forward (host latents -> host prediction)")},
        "gpu_launches": int(launches_step) * args.steps,
        "roofline": {"bound": "tensor", "kernel": "gemm_kernel<128|160|256> (tcgen05 GEMM + implicit-GEMM conv3x3)", "achieved": achieved, "peak": sustained,
                     "unit": "TFLOP/s", "frac": achieved / sustained, "peak_source": f"MEASURED_PEAKS.json bf16_tflops_sustained ({src_pk})",
                     "launches_per_forward": gemm_n, "avg_launch_ms": gemm_ms / max(gemm_n, 1), "algorithmic_tflop_per_forward": gemm_fl / 1e12,
                     "traffic": (traffic or {}).get("gemm_kernel_avg_bytes_per_launch"), "traffic_source": (traffic or {}).get("source"),
                     "executed_tflop_per_forward_all_kernels": executed_fl / 1e12, "by_bound": classes},
        "op_profile": prof,
        "clocks": clocks,
    }
    line.update(extras)
    if solo_ms is not None and is5:
        line["solo_rank0"] = {"ms_per_step": solo_ms, "value": F / (solo_ms / 1000.0), "unit": "frames/s", "independent_units": len(windows) * 2,
                              "what": "the same clip's step (all window forwards at the full CFG batch) on rank 0 alone, the other GPUs idle, in this run"}
    elif solo_ms is not None:
        line["solo_rank0"] = {"ms_per_step": solo_ms, "value": F / (solo_ms / 1000.0), "unit": "frames/s",
                              "what": "the same per-GPU workload (one config-3 clip) timed on rank 0 with the other GPUs idle, in this run: the N = 1 reference of THIS "
                                      "workload (the default N = 1 bench line is config 2, 10 % less work per GPU)"}
    if eager is not None:
        eager["value"] = frames_total / (eager["ms_per_forward"] * (len(windows) if is5 else 1) / 1000.0)
        eager["unit"] = "frames/s"
        line["oracle_gpu_eager"] = eager
    if cpu is not None:
        line["cpu_baseline"] = {"value": cpu["frames_per_s"], "unit": "frames/s", "cores": cpu["cores"], "kind": "port", "sample": cpu["sample"],
                                "run_to_run_spread": cpu["spread"]}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--single-clip", action="store_true",
                    help="with --gpus N > 1 and --config 2|3: ONE clip over the ranks ((window x CFG-half) unit split, SURVEY 8f-4) instead of one clip per rank")
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--config", type=int, default=0, choices=[0, 2, 3, 4, 5], help="BASELINE config; default 2 on one GPU, 4 (= N x config 3) on N > 1")
    ap.add_argument("--banks", type=int, default=0, help="legacy: 1 = config 3")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-eager", action="store_true", help="skip the fp16-eager oracle timing on the GPU")
    ap.add_argument("--quick-cpu", action="store_true", help="2 instead of 3 timed CPU samples")
    ap.add_argument("--no-extras", action="store_true", help="skip the conditioning-branch timings and the 25-step pipeline clip")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    n = max(world, args.gpus)
    c = args.config or (3 if args.banks else (4 if n > 1 else 2))
    if c == 4 and n == 1:
        c = 3
    if c in (2, 3) and n > 1 and not args.single_clip:
        c = 4 if c == 3 else 2   # N > 1 with --config 2 keeps banks off (the round-1 scaling workload)
    cfg = dict(CONFIGS[c])
    if c == 2 and n > 1 and not args.single_clip:
        cfg["name"] = "config2 per GPU"
    if args.single_clip and n > 1 and c in (2, 3):
        cfg["single_clip"] = True
    if args.impl == "reference":
        run_reference(args, rank, cfg)
        return
    if world == 1 and args.gpus > 1:
        # launched without torchrun: re-exec under torch.distributed.run
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}", "--master-addr", "127.0.0.1",
               "--master-port", os.environ.get("MASTER_PORT", "29533"), os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    run_native(args, rank, world, local_rank, cfg)


if __name__ == "__main__":
    main()
