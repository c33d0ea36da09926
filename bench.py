#!/usr/bin/env python
"""bench.py — mel-spectrograms/sec of the DDPM sampling hot path (BASELINE.json metric).

A "step" is one denoising step (per-step noise draw + U-Net forward + fused DDPM update) over one batch of synthetic
input: config C2 of BASELINE.json — audio-diffusion-256 architecture (scripts/train_unet.py:115-137), 256x256x1, batch 64
per GPU, DDPM with 1000 steps per mel-spectrogram.  value = (batch * n_gpus) / (1000 * step time).

    python bench.py --gpus N --steps K --warmup W            # B200 arm (libb200ad.so)
    python bench.py --impl reference --gpus N ...            # CPU arm: oracle port of diffusers, host cores
    python bench.py --mode train ...                         # only the train_unet.py iteration (config C5)
    python bench.py ... --dump-outputs DIR                   # also save the sample the last timed step returned (.npy)

The JSON line of the default arm also carries
  e2e         whole `AudioDiffusionPipeline.__call__` (host noise in, PIL images + audio out): ONE complete 1000-step call
              (the `sustained` object); with --no-extras two short calls, per-step slope x 1000 + tail
  roofline    conv_tc_kernel, CUDA events around every launch of one step
  parity_check  one C2-shape fused step against the CPU oracle (2 of the 64 samples), outside the timed region
  sustained   one complete 1000-step call timed as a whole (what the power cap does to a 37 s run)
  configs     C3 (DDIM-50 whole call), C4 (latent pipeline), C5 (training iteration), Mel codec
Weights are random-init (no network for checkpoints), inputs synthetic (seed 42, as train_unet.py:314).
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True             # the tree may be read-only: no __pycache__ for the modules imported from it
if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
    os.environ["NCCL_DEBUG"] = "WARN"      # before torch loads NCCL: its version banner goes to STDOUT, next to the one JSON line

import torch  # noqa: E402

REF_ARCH = dict(
    in_channels=1, out_channels=1, layers_per_block=2, block_out_channels=(128, 128, 256, 256, 512, 512),
    down_block_types=("DownBlock2D",) * 4 + ("AttnDownBlock2D", "DownBlock2D"),
    up_block_types=("UpBlock2D", "AttnUpBlock2D", "UpBlock2D", "UpBlock2D", "UpBlock2D", "UpBlock2D"))
VAE_ARCH = dict(   # config/ldm_autoencoder_kl.yaml:18-28 as an AutoencoderKL: 1-channel image, 1-channel latent, /8
    in_channels=1, out_channels=1, latent_channels=1, layers_per_block=2, block_out_channels=(128, 256, 512, 512),
    down_block_types=("DownEncoderBlock2D",) * 4, up_block_types=("UpDecoderBlock2D",) * 4)
GFLOP_PER_SAMPLE_FWD = 496.415145984   # analytic, oracle.unet_oracle.unet_flops(256, 256); SURVEY §8(d)
GFLOP_PER_LATENT_FWD = 7.76            # same architecture at 32x32 (SURVEY §8a)
DDPM_STEPS = 1000
TRAFFIC_FILE = "traffic_r02.json"      # profiles/: ncu dram bytes per conv_tc launch of this same command (round tag)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1439.1), d.get("hbm_gbs", 6572.5), "measured"
    return 1400.0, 6650.0, "fallback"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md clocks line)."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index = index
        self.rows = []
        self._halt = threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self._halt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i",
                                      str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self._halt.wait(0.1)

    def stop(self):
        self._halt.set()
        self.join(timeout=3)
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            for k, nm in enumerate(names):
                if len(r) > 2 + k and r[2 + k].lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.rows)}


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


# ------------------------------------------------------------------------------------------------ CPU arm
def cpu_step_rate(batch: int, hw: int, steps: int, warmup: int):
    """Oracle (port of diffusers UNet2DModel + DDPMScheduler.step) on the host cores.
    Returns (mel-spec/s from the median step, list of per-step seconds)."""
    from oracle.schedulers_oracle import OracleDDPM
    from oracle.unet_oracle import UNetConfig, init_weights, unet_forward
    cfg = UNetConfig(sample_size=(hw, hw))
    w = init_weights(cfg, seed=0)
    sch = OracleDDPM()
    sch.set_timesteps(DDPM_STEPS)
    g = torch.Generator().manual_seed(42)
    x = torch.randn(batch, 1, hw, hw, generator=g)
    ts = sch.timesteps
    per = []
    with torch.no_grad():
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            eps = unet_forward(w, cfg, x, ts[i])
            x = sch.step(eps, ts[i], x, generator=g)["prev_sample"]
            if i >= warmup:
                per.append(time.perf_counter() - t0)
    med = sorted(per)[len(per) // 2]
    return batch / (DDPM_STEPS * med), per


def _cpu_threads():
    """Threads of the CPU arm.  The oracle port (torch CPU convolutions) stops scaling early: on the pool's 128-cpu hosts a
    denoise step at batch 4 takes 4.8 s with 16 or 32 threads, 6.6 s with torch's default 64 and 55 s with 128
    (profiles/cpu_threads_r02.txt), so the baseline runs on the count that is FASTEST for it, not on the largest."""
    want = max(1, min(32, os.cpu_count() or 1))
    if torch.get_num_threads() != want:
        torch.set_num_threads(want)
    return torch.get_num_threads()


def run_reference(args):
    rank, world, local = dist_env()
    if rank != 0:
        return
    cores = _cpu_threads()
    batch, hw = 4, 256
    steps = max(3, min(args.steps, 10))
    warmup = 1
    val, per = cpu_step_rate(batch, hw, steps, warmup)
    med = sorted(per)[len(per) // 2]
    line = {
        "impl": "reference", "metric": "mel-spectrograms/sec (1000-step DDPM, 256x256x1)", "value": val,
        "unit": "mel-spectrograms/s", "n_gpus": args.gpus, "steps": steps, "warmup": warmup,
        "ms_per_step": med * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic (random-init weights, seed-42 noise)",
        "config": {"workload": "audio-diffusion-256 DDPM 1000-step, 256x256x1 (C2 architecture)",
                   "note": "CPU arm: bounded sample; value from the MEDIAN step"},
        "step_seconds": {"min": min(per), "median": med, "max": max(per), "n": len(per)},
        "cpu_baseline": {"value": val, "unit": "mel-spectrograms/s", "cores": cores, "kind": "port",
                         "sample": f"batch {batch} x {steps} denoise steps of 1000 at 256x256 (median step), oracle port of "
                                   f"diffusers UNet2DModel+DDPMScheduler (diffusers/librosa not installable), "
                                   f"{cores} torch threads of {os.cpu_count()} cpus"},
        "e2e": {"value": val, "unit": "mel-spectrograms/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ helpers (B200 arm)
def _sync(dist_on):
    if dist_on:
        import torch.distributed as dist
        dist.barrier()
    torch.cuda.synchronize()


def _wall(fn, dist_on):
    """Wall time of fn() bracketed by barrier + synchronize on both sides (seconds)."""
    _sync(dist_on)
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    return dt, out


def _pipe(unet, sch, res, dev, vae=None, hop=512):
    from audio_diffusion_b200.mel import Mel
    from audio_diffusion_b200.pipeline import AudioDiffusionPipeline
    p = AudioDiffusionPipeline(vqvae=vae, unet=unet, mel=Mel(x_res=res, y_res=res, hop_length=hop), scheduler=sch)
    p.set_progress_bar_config(disable=True)
    return p


def whole_call(pipe, batch, steps_a, steps_b, dev, dist_on, latent_hw=None):
    """Time pipe(batch_size, steps) end to end for two step counts (host pinned noise in, PIL images + audio out) and split
    the wall time into per-step and once-per-call parts: T(k) = k * step + tail."""
    c = pipe.unet.in_channels
    hw = latent_hw or pipe.unet.sample_size
    hw = (hw, hw) if isinstance(hw, int) else hw
    noise = torch.randn(batch, c, hw[0], hw[1]).pin_memory()
    gen = torch.Generator(device=dev).manual_seed(42)
    call = lambda k: pipe(batch_size=batch, steps=k, noise=noise, step_generator=gen)     # noqa: E731
    call(2)                                                                                # warm-up: workspaces, constants
    ta, _ = _wall(lambda: call(steps_a), dist_on)
    tb, out = _wall(lambda: call(steps_b), dist_on)
    step = (tb - ta) / (steps_b - steps_a)
    tail = max(ta - steps_a * step, 0.0)
    d2h = len(out.images) * out.images[0].size[0] * out.images[0].size[1] + out.audios.nbytes
    return {"step_s": step, "tail_s": tail, "t_a": ta, "t_b": tb, "steps": [steps_a, steps_b],
            "h2d_bytes_per_call": noise.numel() * 4, "d2h_bytes_per_call": int(d2h)}


# ------------------------------------------------------------------------------------------------ B200 arm
def run_b200(args):
    rank, world, local = dist_env()
    from audio_diffusion_b200 import _lib
    from audio_diffusion_b200.schedulers import DDPMScheduler
    from audio_diffusion_b200.unet import UNet2DModel
    _lib.require_cuda()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    use_dist = world > 1
    if use_dist:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    B, HW = args.batch, args.res
    torch.manual_seed(0)
    model = UNet2DModel(sample_size=(HW, HW), seed=0, **REF_ARCH).to(dev)
    if use_dist:
        # batched sampling shards over GPUs: ONE broadcast of the weights at init, no per-step collective
        from audio_diffusion_b200.parallel import broadcast_parameters
        broadcast_parameters(model.parameters(), src=0)
    sch = DDPMScheduler()
    sch.set_timesteps(DDPM_STEPS)
    g = torch.Generator(device=dev).manual_seed(42 + rank)
    x = torch.randn(B, 1, HW, HW, generator=g, device=dev)
    ts = sch.timesteps
    K, W = args.steps, max(args.warmup, 3)

    def step(i, xin, xout):
        t = ts[i % DDPM_STEPS]
        # as scheduler.step does: a fresh full-batch noise draw per step from the caller's generator (t > 0)
        z = torch.randn(xin.shape, generator=g, device=dev) if int(t) > 0 else None
        return model.forward_step(xin, t, sch.step_coef(t), noise=z, out=xout)

    extras, sustained, parity = {}, None, None
    with torch.no_grad():
        for i in range(W):
            step(i, x, x)
        _sync(use_dist)
        sampler = ClockSampler(local)
        sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(K):
            step(W + i, x, x)
        e1.record()
        _sync(use_dist)
        ms = e0.elapsed_time(e1) / K
        clocks = sampler.stop()
        launches = model.last_launch_count * K
        if args.dump_outputs and rank == 0:
            # the sample the last timed step returned, before the passes below reuse its buffer
            dump_outputs(args.dump_outputs, {"sample": x})

        # ---- e2e: AudioDiffusionPipeline.__call__ — pinned host noise in (H2D inside), K denoise steps incl. the per-step
        # noise draw, float->uint8, D2H, PIL, batched Griffin-Lim, audio D2H.  Two step counts separate the per-step cost
        # from the once-per-call tail; the metric is quoted for the 1000-step call.
        pipe = _pipe(model, DDPMScheduler(), HW, dev)
        Ke = max(4, min(K, 20))
        e2e = whole_call(pipe, B, Ke, 2 * Ke, dev, use_dist)

        # ---- roofline of the dominant kernel (conv_tc_kernel), CUDA events around every launch of one step
        L = _lib.lib()
        maxops = 1024
        op_ms = (C.c_float * maxops)()
        op_kind = (C.c_int * maxops)()
        op_fl = (C.c_double * maxops)()
        t = ts[5]
        tt = model._timesteps(t, B, dev)
        coef = sch.step_coef(t)
        z = torch.randn(B, 1, HW, HW, generator=g, device=dev)
        x.copy_(torch.randn(B, 1, HW, HW, generator=g, device=dev))
        model.forward_step(x, t, coef, noise=z, out=x)          # make sure the plan is bound for this batch / shape
        tot = {}
        for rep in range(3):
            n = L.b200ad_unet_profile_step(model._h, x.data_ptr(), tt.data_ptr(), z.data_ptr(), C.byref(coef),
                                           x.data_ptr(), op_ms, op_kind, op_fl, maxops, _lib.stream_ptr())
            if n < 0:
                raise RuntimeError(L.b200ad_last_error().decode())
            if rep == 0:
                continue
            for i in range(n):
                k = op_kind[i]
                a = tot.setdefault(k, [0.0, 0.0, 0])
                a[0] += op_ms[i] / 2
                a[1] += op_fl[i] / 2
                a[2] += 0.5
        prof = {"ops": n, "by_kind": tot,
                "per_op": [(int(op_kind[i]), float(op_ms[i]), float(op_fl[i])) for i in range(n)]}

        # ---- parity of what was just timed: one fused step at the benchmarked shape vs the CPU oracle on 2 of the B samples
        if rank == 0 and not args.no_cpu and HW == 256:
            parity = parity_check(model, sch, B, HW, dev)

        # ---- the other BASELINE configs, on every rank (C5 all-reduces gradients); max over ranks below
        if not args.no_extras:
            extras = run_extras(args, model, dev, rank, world, use_dist)
            pipe = _pipe(model, DDPMScheduler(), HW, dev)
            sustained = sustained_call(pipe, B, local, dev, use_dist)

    # max over ranks of every time that enters a reported rate
    keys = sorted(k for k, v in extras.items() if isinstance(v, float))
    vec = [ms, e2e["step_s"], e2e["tail_s"]] + [extras[k] for k in keys]
    vec += [sustained["call_s"], sustained["loop_ms"]] if sustained else []
    ms_t = torch.tensor(vec, device=dev, dtype=torch.float64)
    if use_dist:
        dist.all_reduce(ms_t, op=dist.ReduceOp.MAX)
    vec = ms_t.tolist()
    ms, e2e["step_s"], e2e["tail_s"] = vec[:3]
    for i, k in enumerate(keys):
        extras[k] = vec[3 + i]
    if sustained:
        sustained["call_s"], sustained["loop_ms"] = vec[3 + len(keys):]
        sustained["value"] = B * world / sustained["call_s"]
    if rank != 0:
        if use_dist:
            dist.destroy_process_group()
        return

    peak_tf, peak_hbm, how = peaks()
    value = B * world / (DDPM_STEPS * ms * 1e-3)
    e2e_call_s = DDPM_STEPS * e2e["step_s"] + e2e["tail_s"]
    names = {0: "temb", 1: "conv_in", 2: "gn_finalize", 3: "conv_tc", 4: "upsample", 5: "parity_split", 6: "attention", 7: "conv_out",
             15: "gn_apply"}
    conv = prof["by_kind"].get(3, [0.0, 0.0, 0])
    step_prof_ms = sum(v[0] for v in prof["by_kind"].values())
    conv_tf = conv[1] / (conv[0] * 1e-3) / 1e12 if conv[0] > 0 else 0.0
    # DRAM bytes per conv_tc launch: ncu launch list of this same command, committed under profiles/ with the round tag;
    # valid for the default workload only (batch 64, 256x256), null otherwise
    traffic, traffic_src = None, None
    tpath = os.path.join(ROOT, "profiles", TRAFFIC_FILE)
    if os.path.exists(tpath) and HW == 256 and B == 64:
        with open(tpath) as f:
            tj = json.load(f)
        tk = tj["kernels"].get("conv_tc_kernel")
        if tk:
            traffic = tk["dram_read_bytes_per_launch"] + tk["dram_write_bytes_per_launch"]
            traffic_src = (f"profiles/{TRAFFIC_FILE} (ncu dram__bytes_read.sum + dram__bytes_write.sum, mean over "
                           f"{tk.get('launches', '?')} launches)")
    roof = {"bound": "tensor", "kernel": "conv_tc_kernel", "achieved": conv_tf, "peak": peak_tf, "unit": "TFLOP/s",
            "frac": conv_tf / peak_tf, "peak_source": f"{how} bf16 sustained (MEASURED_PEAKS.json)",
            "traffic": traffic, "traffic_source": traffic_src,
            "launches_per_step": int(conv[2]), "avg_launch_ms": conv[0] / max(conv[2], 1),
            "algorithmic_gflop_per_launch": conv[1] / max(conv[2], 1) / 1e9,
            "algorithmic_gflop_note": "conv / linear MACs only; identity-residual K-segments carry no algorithmic FLOPs",
            "kernel_share_of_step": conv[0] / step_prof_ms if step_prof_ms else None,
            "whole_step_tflops": GFLOP_PER_SAMPLE_FWD * B / (ms * 1e-3) / 1e3 if HW == 256 else None,
            "whole_step_frac": (GFLOP_PER_SAMPLE_FWD * B / (ms * 1e-3) / 1e3 / peak_tf) if HW == 256 else None,
            "ms_by_kernel": {names.get(k, f"kind{k}"): round(v[0], 4) for k, v in sorted(prof["by_kind"].items())}}
    cpu = None
    if not args.no_cpu and world == 1:
        cores = _cpu_threads()
        v, per = cpu_step_rate(4, HW, 5, 1)
        cpu = {"value": v, "unit": "mel-spectrograms/s", "cores": cores, "kind": "port",
               "step_seconds": {"min": min(per), "median": sorted(per)[len(per) // 2], "max": max(per)},
               "sample": f"batch 4 x 5 denoise steps (of 1000) at {HW}x{HW} on {cores} torch threads "
                         f"({os.cpu_count()} cpus), median step; oracle port of diffusers UNet2DModel + DDPMScheduler.step"}
    line = {
        "metric": "mel-spectrograms/sec (1000-step DDPM, 256x256x1)", "value": value, "unit": "mel-spectrograms/s",
        "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16 operands, fp32 accumulate (fp32 master weights, fp64 GroupNorm sums)",
        "data": "synthetic (random-init weights seed 0, noise seed 42)",
        "config": {"workload": f"audio-diffusion-256 DDPM 1000-step, batch={B} per GPU, {HW}x{HW}x1, {world}xB200",
                   "global_batch": B * world, "parallelism": f"dp{world} (batch sharded, weights broadcast once)",
                   "l2": "activations per step (>10 GB) far exceed the 126 MB L2; no explicit flush",
                   "step": "one denoise step = per-step randn + UNet2DModel forward + fused DDPMScheduler.step"},
        "clocks": clocks, "gpu_launches": launches,
        "e2e": {"value": (sustained["value"] if sustained else B * world / e2e_call_s), "unit": "mel-spectrograms/s",
                "source": ("one COMPLETE 1000-step call timed as a whole (the `sustained` object)" if sustained else
                           "two short calls (steps a, b): per-step slope x 1000 + once-per-call tail"),
                "api": "AudioDiffusionPipeline.__call__(batch_size, steps, noise=<pinned host>, step_generator): H2D of the "
                       "noise, denoise loop with per-step randn, float->uint8, D2H, PIL images, batched Griffin-Lim, audio D2H",
                "call_s_1000_steps": e2e_call_s, "ms_per_step": e2e["step_s"] * 1e3, "tail_s": e2e["tail_s"],
                "measured": {"steps": e2e["steps"], "wall_s": [e2e["t_a"], e2e["t_b"]]},
                "h2d_bytes_per_step": e2e["h2d_bytes_per_call"] / DDPM_STEPS,
                "d2h_bytes_per_step": e2e["d2h_bytes_per_call"] / DDPM_STEPS,
                "h2d_bytes_per_call": e2e["h2d_bytes_per_call"], "d2h_bytes_per_call": e2e["d2h_bytes_per_call"]},
        "roofline": roof, "cpu_baseline": cpu, "parity_check": parity, "sustained": sustained,
    }
    if extras:
        line["configs"] = format_extras(extras, world, peak_tf, peak_hbm)
    if args.dump_ops:
        os.makedirs(os.path.dirname(args.dump_ops) or ".", exist_ok=True)
        json.dump(prof["per_op"], open(args.dump_ops, "w"))
    print(json.dumps(line), flush=True)
    if use_dist:
        dist.destroy_process_group()


MAX_DUMP_BYTES = 64 << 20


def dump_outputs(d, arrays):
    """Write each tensor as d/<name>.npy in float32.  A tensor over MAX_DUMP_BYTES keeps a fixed, seeded choice of whole
    samples along dim 0 (the same rows on every run), so that two builds can be compared output for output."""
    import numpy as np
    os.makedirs(d, exist_ok=True)
    for name, t in arrays.items():
        per = t[0].numel() * 4
        if t.shape[0] * per > MAX_DUMP_BYTES:
            keep = max(MAX_DUMP_BYTES // per, 1)
            rows = torch.randperm(t.shape[0], generator=torch.Generator().manual_seed(0))[:keep].sort().values
            t = t[rows.to(t.device)]
        np.save(os.path.join(d, name + ".npy"), t.float().cpu().numpy())


def parity_check(model, sch, B, HW, dev):
    """One fused step at the benchmarked shape (batch B, HW x HW) against the CPU oracle on samples 0 and B-1."""
    from oracle.schedulers_oracle import OracleDDPM
    from oracle.unet_oracle import UNetConfig, unet_forward
    _cpu_threads()
    cfg = UNetConfig(sample_size=(HW, HW))
    w = {k: v.detach().cpu() for k, v in model.state_dict().items()}
    gq = torch.Generator().manual_seed(123)
    x = torch.randn(B, 1, HW, HW, generator=gq)
    z = torch.randn(B, 1, HW, HW, generator=gq)
    t = sch.timesteps[300]
    got, eps = model.forward_step(x.to(dev), t, sch.step_coef(t), noise=z.to(dev), want_eps=True)
    idx = [0, B - 1]
    osch = OracleDDPM()
    osch.set_timesteps(DDPM_STEPS)
    with torch.no_grad():
        e_ref = unet_forward(w, cfg, x[idx], t)
    a_t = osch.alphas_cumprod[int(t)]
    coef = sch.step_coef(t)
    x0 = ((x[idx] - (1 - a_t) ** 0.5 * e_ref) / a_t ** 0.5).clamp(-1, 1)
    ref = coef.c_x0 * x0 + coef.c_xt * x[idx] + coef.c_z * z[idx]

    def rel(a, b):
        d = a - b
        return {"max_rel": d.abs().max().item() / b.abs().max().item(),
                "rms_rel": (d.pow(2).mean().sqrt() / b.pow(2).mean().sqrt()).item()}
    r_eps, r_x = rel(eps.cpu()[idx], e_ref), rel(got.cpu()[idx], ref)
    return {"shape": [B, 1, HW, HW], "samples_checked": idx, "timestep": int(t), "eps": r_eps, "x_prev": r_x,
            "max_rel": r_eps["max_rel"], "rms_rel": r_eps["rms_rel"],
            "tolerance": {"max_rel": 0.06, "rms_rel": 0.015},
            "ok": bool(r_eps["max_rel"] <= 0.06 and r_eps["rms_rel"] <= 0.015)}


def sustained_call(pipe, B, local, dev, dist_on):
    """ONE complete DDPM-1000 call through the public API, timed as a whole (clocks sampled throughout): the number a 37 s
    run really gets under the board power cap, next to the K-step headline."""
    gen = torch.Generator(device=dev).manual_seed(7)
    noise = torch.randn(B, 1, *pipe.unet.sample_size).pin_memory()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    orig = pipe._denoise

    def timed_denoise(*a, **k):
        e0.record()
        r = orig(*a, **k)
        e1.record()
        return r
    pipe._denoise = timed_denoise
    sampler = ClockSampler(local)
    sampler.start()
    dt, out = _wall(lambda: pipe(batch_size=B, steps=DDPM_STEPS, noise=noise, step_generator=gen), dist_on)
    clocks = sampler.stop()
    pipe._denoise = orig
    return {"call_s": dt, "loop_ms": e0.elapsed_time(e1) / DDPM_STEPS, "steps": DDPM_STEPS, "batch_per_gpu": B,
            "value": B / dt, "unit": "mel-spectrograms/s", "clocks": clocks,
            "what": "AudioDiffusionPipeline.__call__(batch_size=B, steps=1000) incl. H2D noise, uint8, PIL, Griffin-Lim"}


def run_extras(args, model, dev, rank, world, dist_on):
    """C3 / C4 / C5 / Mel codec measurements (BASELINE.json configs[2..4], SURVEY §8d). Returns flat {name: seconds}."""
    from audio_diffusion_b200.mel import Mel
    from audio_diffusion_b200.schedulers import DDIMScheduler, DDPMScheduler
    from audio_diffusion_b200.unet import UNet2DModel
    from audio_diffusion_b200.vae import AutoencoderKL
    ex = {}
    HW, B = args.res, args.batch
    # ---- C3: DDIM 50 steps, batch 64 per GPU (512 over 8), whole call
    pipe = _pipe(model, DDIMScheduler(), HW, dev)
    r = whole_call(pipe, B, 25, 50, dev, dist_on)
    ex["c3_step_s"], ex["c3_tail_s"], ex["c3_call50_s"] = r["step_s"], r["tail_s"], r["t_b"]
    # ---- Mel codec alone (batch 64): encode 64 slices, decode 64 images
    mel = Mel(x_res=HW, y_res=HW)
    gcpu = torch.Generator().manual_seed(0)
    n = 64
    audio = (0.1 * torch.randn(n, mel.slice_size, generator=gcpu)
             + 0.5 * torch.sin(2 * torch.pi * 440.0 * torch.arange(mel.slice_size) / 22050.0)[None]).to(dev)
    imgs = mel.audio_slices_to_images(audio)
    mel.images_to_audio(imgs)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    _sync(dist_on)
    e0.record()
    for _ in range(3):
        imgs = mel.audio_slices_to_images(audio)
    e1.record()
    torch.cuda.synchronize()
    ex["mel_encode_s"] = e0.elapsed_time(e1) / 3 * 1e-3
    dt, _ = _wall(lambda: [mel.images_to_audio(imgs) for _ in range(3)], dist_on)
    ex["mel_decode_s"] = dt / 3          # incl. the D2H of the audio (images_to_audio returns numpy)
    del audio, imgs
    # ---- C4: latent audio diffusion, batch 128: latent U-Net (32x32) loop + VAE decode + Griffin-Lim tail
    if HW == 256:
        lat = HW // 8
        lunet = UNet2DModel(sample_size=(lat, lat), seed=1, **REF_ARCH).to(dev)
        vae = AutoencoderKL(seed=2, **VAE_ARCH).to(dev)
        lpipe = _pipe(lunet, DDPMScheduler(), HW, dev, vae=vae)
        r = whole_call(lpipe, 128, 50, 100, dev, dist_on, latent_hw=(lat, lat))
        ex["c4_step_s"], ex["c4_tail_s"] = r["step_s"], r["tail_s"]
        zl = torch.randn(128, 1, lat, lat, device=dev)
        vae.decode(zl)
        dt, _ = _wall(lambda: vae.decode(zl), dist_on)
        ex["c4_vae_decode_s"] = dt
        del lpipe, lunet, vae, zl
        torch.cuda.empty_cache()
    # ---- batch 1 (the reference facade hard-codes batch_size=1, audiodiffusion/__init__.py:59): device time per step and the
    # host time it takes to ENQUEUE a step (if the host is faster than the GPU, launch overhead is hidden and a CUDA graph
    # would not shorten the step)
    if HW == 256:
        sch1 = DDPMScheduler()
        sch1.set_timesteps(DDPM_STEPS)
        g1 = torch.Generator(device=dev).manual_seed(5)
        x1 = torch.randn(1, 1, HW, HW, generator=g1, device=dev)

        def step1(i):
            t = sch1.timesteps[i]
            z = torch.randn(x1.shape, generator=g1, device=dev)
            model.forward_step(x1, t, sch1.step_coef(t), noise=z, out=x1)
        for i in range(5):
            step1(i)
        _sync(dist_on)
        nb1 = 30
        t0 = time.perf_counter()
        e0.record()
        for i in range(nb1):
            step1(5 + i)
        e1.record()
        host = time.perf_counter() - t0           # all steps enqueued (no synchronisation yet)
        torch.cuda.synchronize()
        ex["b1_step_s"] = e0.elapsed_time(e1) / nb1 * 1e-3
        ex["b1_host_enqueue_s"] = host / nb1
        ex["b1_launches"] = float(model.last_launch_count)
        # the same steps as CUDA-graph replays (what AudioDiffusionPipeline does for batches <= 8)
        stepper = model.graph_stepper(x1)       # owns its sample buffer (initialised from x1)

        def gstep(i):
            t = sch1.timesteps[i]
            stepper.step(t, sch1.step_coef(t), torch.randn(x1.shape, generator=g1, device=dev))
        for i in range(5):
            gstep(40 + i)
        _sync(dist_on)
        e0.record()
        for i in range(nb1):
            gstep(45 + i)
        e1.record()
        torch.cuda.synchronize()
        ex["b1_graph_step_s"] = e0.elapsed_time(e1) / nb1 * 1e-3
        del stepper
    # ---- C5: one train_unet.py iteration (fwd + bwd + all-reduce + clip + AdamW + EMA), batch 16 per GPU
    from audio_diffusion_b200.training import EMAModel, FusedAdamW, train_step
    tb = 16
    tmodel = UNet2DModel(sample_size=(HW, HW), seed=0, **REF_ARCH).to(dev).train()
    if dist_on:
        from audio_diffusion_b200.parallel import broadcast_parameters
        broadcast_parameters(tmodel.parameters(), src=0)
    opt = FusedAdamW(tmodel.parameters(), lr=1e-4, betas=(0.95, 0.999), weight_decay=1e-6, eps=1e-8, max_grad_norm=1.0)
    ema = EMAModel(tmodel.parameters(), inv_gamma=1.0, power=0.75, max_value=0.9999)
    opt.attach_ema(ema)
    tsch = DDPMScheduler()
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    xb = (torch.randint(0, 256, (tb, 1, HW, HW), device=dev, generator=gen).float() / 255.0 - 0.5) / 0.5
    with torch.enable_grad():
        for _ in range(3):
            train_step(tmodel, opt, tsch, xb, ema=ema, generator=gen)

        def timed(nsteps, sync=True):
            _sync(dist_on)
            e0.record()
            for _ in range(nsteps):
                if sync:
                    train_step(tmodel, opt, tsch, xb, ema=ema, generator=gen)
                else:
                    with tmodel.no_sync():
                        train_step(tmodel, opt, tsch, xb, ema=ema, generator=gen)
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / nsteps * 1e-3
        ex["c5_step_s"] = timed(5)
        ex["c5_step_nosync_s"] = timed(5, sync=False) if dist_on else ex["c5_step_s"]
    ex["c5_launches"] = float(tmodel.last_launch_count + tmodel.last_backward_launch_count + 4)
    del tmodel, opt, ema, xb
    torch.cuda.empty_cache()
    return ex


def format_extras(ex, world, peak_tf, peak_hbm):
    B = 64
    out = {}
    c3_call = 50 * ex["c3_step_s"] + ex["c3_tail_s"]
    out["C3_ddim50"] = {"workload": f"audio-diffusion-ddim-256 DDIM 50-step, batch 64 per GPU ({64 * world} over {world} GPUs), whole call",
                        "value": B * world / c3_call, "unit": "mel-spectrograms/s", "call_s": c3_call,
                        "measured_call50_s": ex["c3_call50_s"], "ms_per_step": ex["c3_step_s"] * 1e3,
                        "tail_s": ex["c3_tail_s"]}
    if "c4_step_s" in ex:
        c4_call = DDPM_STEPS * ex["c4_step_s"] + ex["c4_tail_s"]
        out["C4_latent"] = {"workload": "latent-audio-diffusion-256: 32x32 latent U-Net DDPM-1000 + VAE decode + Griffin-Lim, batch 128 per GPU",
                            "value": 128 * world / c4_call, "unit": "mel-spectrograms/s", "call_s_1000_steps": c4_call,
                            "loop_ms_per_step": ex["c4_step_s"] * 1e3, "tail_s": ex["c4_tail_s"],
                            "vae_decode_s_batch128": ex["c4_vae_decode_s"],
                            "loop_tflops": GFLOP_PER_LATENT_FWD * 128 / ex["c4_step_s"] / 1e3}
    if "b1_step_s" in ex:
        out["B1_latency"] = {"workload": "audio-diffusion-256 denoise step at batch 1 (the reference facade's batch_size=1 path)",
                             "ms_per_step": ex["b1_graph_step_s"] * 1e3, "eager_ms_per_step": ex["b1_step_s"] * 1e3,
                             "eager_host_enqueue_ms_per_step": ex["b1_host_enqueue_s"] * 1e3,
                             "gpu_launches_per_step": int(ex["b1_launches"]),
                             "value": 1.0 / (DDPM_STEPS * ex["b1_graph_step_s"]), "unit": "mel-spectrograms/s",
                             "tflops": GFLOP_PER_SAMPLE_FWD / ex["b1_graph_step_s"] / 1e3,
                             "note": "ms_per_step = the step replayed as one CUDA graph (UNet2DModel.graph_stepper, what the pipeline "
                                     "does for batches <= 8); eager = ~120 launches per step enqueued from Python"}
    tf = 3 * GFLOP_PER_SAMPLE_FWD * 16 / ex["c5_step_s"] / 1e3
    out["C5_train"] = {"workload": f"train_unet.py iteration 256x256, batch 16 per GPU, dp{world}: fwd + bwd + all-reduce + clip + AdamW + EMA",
                       "value": 16 * world / ex["c5_step_s"], "unit": "images/s", "ms_per_step": ex["c5_step_s"] * 1e3,
                       "exposed_allreduce_ms": max(ex["c5_step_s"] - ex["c5_step_nosync_s"], 0.0) * 1e3,
                       "tflops_per_gpu": tf, "frac_of_peak": tf / peak_tf, "flops_model": "3 x 496.42 GFLOP per sample",
                       "gpu_launches_per_step": int(ex["c5_launches"])}
    # Mel codec: algorithmic bytes (DESIGN.md §3, Mel codec): encode reads the slice (fp32) and writes the image;
    # decode per Griffin-Lim iteration reads + writes the complex128 spectrum (1025 x 256 x 16 B) and the fp64 audio twice
    n, L, F, T = 64, 131071, 1025, 256
    enc_bytes = n * (L * 4 + 256 * 256)
    dec_bytes = n * (32 * (3 * F * T * 16 + 2 * (T - 1) * 512 * 8) + F * T * 8 + 256 * 256)
    out["mel_codec"] = {"batch": n,
                        "encode_ms": ex["mel_encode_s"] * 1e3, "encode_gbs": enc_bytes / ex["mel_encode_s"] / 1e9,
                        "decode_ms": ex["mel_decode_s"] * 1e3, "decode_gbs": dec_bytes / ex["mel_decode_s"] / 1e9,
                        "hbm_peak_gbs": peak_hbm, "encode_frac": enc_bytes / ex["mel_encode_s"] / 1e9 / peak_hbm,
                        "decode_frac": dec_bytes / ex["mel_decode_s"] / 1e9 / peak_hbm,
                        "algorithmic_bytes": {"encode": enc_bytes, "decode": dec_bytes}}
    return out


# ------------------------------------------------------------------------------------------------ training mode (extra)
def run_train(args):
    """`--mode train`: one iteration of scripts/train_unet.py:238-267 per step (config C5 of SURVEY §8: 256x256, bf16
    activations, data parallel). Not the headline metric — a separate JSON line with its own metric name."""
    rank, world, local = dist_env()
    from audio_diffusion_b200 import _lib
    from audio_diffusion_b200.parallel import broadcast_parameters
    from audio_diffusion_b200.schedulers import DDPMScheduler
    from audio_diffusion_b200.training import EMAModel, FusedAdamW, train_step
    from audio_diffusion_b200.unet import UNet2DModel
    _lib.require_cuda()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    use_dist = world > 1
    if use_dist:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    B = args.batch if args.batch != 64 else 16          # per-GPU batch (C5 states it): default 16
    HW = args.res
    model = UNet2DModel(sample_size=(HW, HW), seed=0, **REF_ARCH).to(dev).train()
    if use_dist:
        broadcast_parameters(model.parameters(), src=0)
    opt = FusedAdamW(model.parameters(), lr=1e-4, betas=(0.95, 0.999), weight_decay=1e-6, eps=1e-8, max_grad_norm=1.0)
    ema = EMAModel(model.parameters(), inv_gamma=1.0, power=0.75, max_value=0.9999)
    opt.attach_ema(ema)
    sch = DDPMScheduler()
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    # synthetic dataset batch: uint8 images through ToTensor + Normalize(.5, .5) (train_unet.py:73-78), resident on the GPU
    x = (torch.randint(0, 256, (B, 1, HW, HW), device=dev, generator=gen).float() / 255.0 - 0.5) / 0.5
    W = max(args.warmup, 3)
    for _ in range(W):
        train_step(model, opt, sch, x, ema=ema, generator=gen)
    torch.cuda.synchronize()
    if use_dist:
        dist.barrier()
    sampler = ClockSampler(local)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        loss = train_step(model, opt, sch, x, ema=ema, generator=gen)
    e1.record()
    torch.cuda.synchronize()
    clocks = sampler.stop()
    ms = e0.elapsed_time(e1) / args.steps
    ms_t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if use_dist:
        dist.all_reduce(ms_t, op=dist.ReduceOp.MAX)
        dist.barrier()
    ms = ms_t.item()
    if rank == 0:
        peak_tf, _, how = peaks()
        gf = GFLOP_PER_SAMPLE_FWD if HW == 256 else None
        tf = 3 * gf * B / ms if gf else None
        print(json.dumps({
            "metric": "images/sec (train_unet.py step: fwd + bwd + clip + AdamW + EMA, 256x256x1)", "mode": "train",
            "value": B * world / ms * 1e3, "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": W,
            "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16 activations and activation gradients, fp32 parameters / parameter gradients / optimizer",
            "data": "synthetic (uint8 images -> [-1,1], random-init weights seed 0)",
            "config": {"workload": f"train_unet.py iteration, batch={B} per GPU, {HW}x{HW}x1, {world}xB200",
                       "global_batch": B * world, "parallelism": f"dp{world} (one all-reduce of the flat gradient buffer per step)"},
            "clocks": clocks, "gpu_launches": (model.last_launch_count + model.last_backward_launch_count + 4) * args.steps,
            "roofline": {"bound": "tensor", "achieved": tf, "peak": peak_tf, "unit": "TFLOP/s",
                         "frac": tf / peak_tf if tf else None, "peak_source": f"{how} bf16 sustained (MEASURED_PEAKS.json)",
                         "traffic": None, "flops_model": "3 x 496.42 GFLOP per sample (SURVEY §8d)"},
            "loss": float(loss)}))
    if use_dist:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mode", default="sample", choices=["sample", "train"],
                    help="sample = the headline metric (default); train = one train_unet.py iteration per step")
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--res", type=int, default=256)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline and parity_check legs (both run the CPU oracle)")
    ap.add_argument("--no-extras", action="store_true", help="skip the C3/C4/C5/Mel sub-benchmarks and the sustained call")
    ap.add_argument("--dump-ops", default=None, help="write the per-launch profile (kind, ms, flops) to this JSON")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed steps write the sample the last one returned (rank 0) as DIR/sample.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.mode != "sample"):
        ap.error("--dump-outputs writes the outputs of the B200 sampling path (--impl b200 --mode sample)")
    if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
        os.environ["NCCL_DEBUG"] = "WARN"      # keep stdout to the one JSON line (NCCL prints its version banner to stdout)
    if args.impl == "reference":
        run_reference(args)
    elif args.mode == "train":
        run_train(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
