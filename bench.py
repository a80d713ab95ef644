#!/usr/bin/env python
"""Benchmark of the hot path named by BASELINE.json: `LatentToVideoPipeline.__call__` for one 16-frame 512x512 clip,
50 DDIM steps, CFG 9, random-init full-size UNet3D (1.41 B params) + SD VAE, bf16, synthetic inputs (config 2).

  python bench.py --gpus N --steps K --warmup W          # this repo (sm_100a kernels)
  python bench.py --impl reference --gpus N ...          # the reference's CPU path (oracle port) on the host cores

A "step" of this bench = one whole pipeline call (50 denoising steps + VAE decode) = 16 denoised frames per rank.
N > 1 (torchrun, one rank per GPU): weak scaling — every rank generates its own clip (prompts / CFG pairs are sharded
with both halves of a pair co-located, SURVEY.md 8e), decoded frames are all-gathered with ONE NCCL collective.

JSON line: `value` = frames/s with inputs resident in HBM (CUDA events, max over ranks); `e2e` = the same through the
public API with pinned HOST inputs copied H2D every step and the decoded video read back D2H; `roofline` = achieved
tensor TFLOP/s of the dominant kernel (tcgen05 implicit GEMM, all launches of one UNet forward timed with CUDA events)
against the measured bf16 peak; `cpu_baseline` = the oracle timed on the host cores on a bounded sample.
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

METRIC = "denoised_frames_per_sec_16f_512x512_50ddim"
UNIT = "frames/s"
FRAMES, HW, LAT, STEPS_DDIM, GUIDANCE = 16, 512, 64, 50, 9.0
SCHED = dict(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear", clip_sample=False,
             set_alpha_to_one=False, steps_offset=1)


def _peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return p["bf16_tflops_sustained"], p["hbm_gbs"], "measured (MEASURED_PEAKS.json, sustained)"
    except Exception:
        return 1400.0, 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.stop_flag = False

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                parts = [x.strip() for x in out.strip().split(",")]
                if len(parts) >= 6:
                    self.samples.append(parts)
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(int(float(s[0])) for s in self.samples)
        reasons = []
        for name, col in (("hw_slowdown", 2), ("hw_thermal_slowdown", 3), ("sw_thermal_slowdown", 4), ("sw_power_cap", 5)):
            if any(s[col].lower().startswith("active") for s in self.samples):
                reasons.append(name)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": int(float(self.samples[0][1])), "reasons": reasons}


# ------------------------------------------------------------------------------------------------ reference arm
def _usable_cores():
    """Host cores this process may actually use: affinity mask and cgroup CPU quota (os.cpu_count() reports the whole
    host inside a container; 128 torch threads on a 16-core quota ran the oracle 14x SLOWER than 8 threads)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, -(-int(q) // int(per))))
    except Exception:
        pass
    try:
        q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
        per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
        if q > 0:
            n = min(n, max(1, -(-q // per)))
    except Exception:
        pass
    return max(1, n)


def _oracle_unet_sample(threads=None):
    """Bounded CPU sample of the workload: one oracle UNet3D forward (fp32) for ONE batch element of the CFG pair.
    Picks the thread count (<= usable cores) that runs a small calibration forward fastest, then the largest frame count
    whose estimated time stays under ~25 s.  Returns (unet, fwd, frames_in_sample, description, threads_used)."""
    import torch
    from oracle.composition import OracleUNet3D
    usable = threads or _usable_cores()
    torch.manual_seed(0)
    unet = OracleUNet3D(motion_mask=True, motion_strength=True).eval()
    g = torch.Generator().manual_seed(1)

    def fwd(f, hw):
        s = torch.randn(1, 4, f, hw, hw, generator=g)
        c = torch.randn(1, 4, 1, hw, hw, generator=g)
        e = torch.randn(1, 77, 1024, generator=g)
        m = torch.ones(1, 1, 1, hw, hw)
        t0 = time.perf_counter()
        with torch.no_grad():
            unet(s, 500, e, c, m, motion=torch.tensor([4.0]))
        return time.perf_counter() - t0

    best_t, best_n = None, usable
    for n in sorted({usable, min(usable, 64), min(usable, 32), min(usable, 16), min(usable, 8)}, reverse=True):
        torch.set_num_threads(n)
        t = fwd(1, 16)                                  # T=2 at 16x16 latents: ~0.1 TFLOP, sub-second
        if best_t is None or t < best_t:
            best_t, best_n = t, n
    torch.set_num_threads(best_n)
    cal = fwd(2, 32)                                    # calibration: T=3 at 32x32 (0.9 TFLOP)
    est_full = cal * (17 / 3) * 4
    f_sample = 16
    for f in (16, 4, 1):
        f_sample = f
        if est_full * (f + 1) / 17 <= 25:
            break
    if f_sample == 16:
        desc = "1 oracle UNet3D forward, fp32, B=1 (one CFG half), T=17, 64x64 latents"
    else:
        desc = (f"1 oracle UNet3D forward, fp32, B=1, T={f_sample + 1} of 17 frames, 64x64 latents; scaled linearly in T "
                f"(all ops but the 0.1%-FLOP temporal attention are linear in T)")
    return unet, fwd, f_sample, desc + f"; {best_n} torch threads (fastest of the tried counts, {usable} usable cores)", best_n


def cpu_frames_per_sec(sample_s, f_sample):
    per_fwd_b1 = sample_s * (17.0 / (f_sample + 1))
    clip_s = per_fwd_b1 * 2 * STEPS_DDIM                    # CFG pair x 50 steps; VAE decode (1.8 % of FLOPs) ignored
    return FRAMES / clip_s


def run_reference(args):
    import torch
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    unet, fwd, f_sample, desc, threads = _oracle_unet_sample()
    for _ in range(args.warmup):
        fwd(f_sample, LAT)
    times = [fwd(f_sample, LAT) for _ in range(max(1, args.steps))]
    t = sum(times) / len(times)
    v = cpu_frames_per_sec(t, f_sample)
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": FRAMES / v * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "config2: pipeline.__call__ 16x512x512, 50 DDIM steps, CFG 9 (CPU: extrapolated from "
                                   "a bounded sample)", "sample_seconds": t},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": "port", "sample": desc},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ product arm
def build_models(device, dtype):
    import torch
    from animate_anything_b200.autoencoder_kl import AutoencoderKL
    from animate_anything_b200.pipeline import LatentToVideoPipeline
    from animate_anything_b200.schedulers import DDIMScheduler
    from animate_anything_b200.unet_3d_condition_mask import UNet3DConditionModel
    torch.manual_seed(0)
    with torch.device(device):
        unet = UNet3DConditionModel(sample_size=LAT, motion_mask=True, motion_strength=True)
        vae = AutoencoderKL()
    # the reference zero-inits these; re-draw so they are exercised (BASELINE.md section 3)
    with torch.no_grad():
        for n, p in unet.named_parameters():
            if p.abs().max() == 0:
                p.normal_(0.0, 0.02)
    unet = unet.to(dtype).eval()
    vae = vae.to(dtype).eval()
    pipe = LatentToVideoPipeline(vae=vae, text_encoder=None, tokenizer=None, unet=unet, scheduler=DDIMScheduler(**SCHED))
    return pipe


def synth_inputs(rank, pinned=True):
    import torch
    g = torch.Generator().manual_seed(100 + rank)
    d = {"latents": torch.randn(1, 4, FRAMES, LAT, LAT, generator=g),
         "condition_latent": torch.randn(1, 4, 1, LAT, LAT, generator=g),
         "prompt_embeds": torch.randn(1, 77, 1024, generator=g),
         "negative_prompt_embeds": torch.randn(1, 77, 1024, generator=g),
         "mask": torch.ones(1, 1, 1, LAT, LAT)}
    d = {k: v.to(torch.bfloat16) for k, v in d.items()}
    if pinned:
        d = {k: v.pin_memory() for k, v in d.items()}
    return d


def _stack_inputs(n_prompts, dev=None, pinned=False):
    import torch
    per = [synth_inputs(i, pinned=False) for i in range(n_prompts)]
    d = {k: torch.cat([p[k] for p in per]) for k in per[0] if k != "mask"}
    d["mask"] = per[0]["mask"]
    if pinned:
        d = {k: v.pin_memory() for k, v in d.items()}
    if dev is not None:
        d = {k: v.to(dev) for k, v in d.items()}
    return d


def _ev_ms(fn, reps=1, warm=1):
    """CUDA-event time of fn() on the current stream, ms per call."""
    import torch
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """Writes each named tensor as `<out_dir>/<name>.npy`, float64 kept, every other dtype as float32, at most
    DUMP_LIMIT_BYTES in all.  A tensor too large for its share of that limit is written as a fixed seeded sample of its
    flattened elements (1-D): the positions depend only on its shape, so dumps of two builds compare element for
    element."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    items = sorted(arrays.items(), key=lambda kv: kv[1].numel())
    budget = DUMP_LIMIT_BYTES - 1024 * len(items)        # room for the .npy headers
    for i, (name, t) in enumerate(items):
        dt = torch.float64 if t.dtype == torch.float64 else torch.float32
        share = budget // (len(items) - i)
        n = share // dt.itemsize
        if t.numel() > n:
            idx = np.sort(np.random.default_rng(0).integers(0, t.numel(), size=n))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        a = t.detach().to("cpu", dt).numpy()
        np.save(os.path.join(out_dir, name + ".npy"), a)
        budget -= a.nbytes


def parity_check(pipe, devin, dev, kw):
    """2 DDIM steps of the BENCHMARKED configuration (same weights, same inputs, graph replay as timed) against the fp32
    oracle and the stock bf16 torch execution on the same GPU.  Returns the dict stored under config.parity_check and
    the (bf16) oracle modules for the torch-eager leg."""
    import torch
    from oracle.composition import (AutoencoderKL as OVAE, DDIMScheduler as ODDIM, OracleUNet3D, oracle_sampling_loop)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    with torch.device(dev):
        ounet = OracleUNet3D(motion_mask=True, motion_strength=True).eval()
        ovae = OVAE().eval()
    ounet.load_state_dict({k: v.float() for k, v in pipe.unet.state_dict().items()})
    ovae.load_state_dict({k: v.float() for k, v in pipe.vae.state_dict().items()})
    kw2 = dict(kw, num_inference_steps=2)
    video, lat = pipe(prompt_embeds=devin["prompt_embeds"], negative_prompt_embeds=devin["negative_prompt_embeds"],
                      latents=devin["latents"], condition_latent=devin["condition_latent"], mask=devin["mask"], **kw2)
    f32 = {k: v.float() for k, v in devin.items()}
    _, rl = oracle_sampling_loop(ounet, ODDIM(**SCHED), f32["latents"], f32["prompt_embeds"],
                                 f32["negative_prompt_embeds"], f32["condition_latent"], f32["mask"], [4], GUIDANCE, 2,
                                 vae=None)
    ounet, ovae = ounet.to(torch.bfloat16), ovae.to(torch.bfloat16)
    _, sl = oracle_sampling_loop(ounet, ODDIM(**SCHED), devin["latents"], devin["prompt_embeds"],
                                 devin["negative_prompt_embeds"], devin["condition_latent"], devin["mask"], [4],
                                 GUIDANCE, 2, vae=None)
    # VAE decode compared on IDENTICAL latents (the product's): a random-init decoder amplifies the few-percent latent
    # difference of two bf16 loops into decorrelated pixels, which would say nothing about the decoder kernels
    from oracle.composition import oracle_decode_latents
    with torch.no_grad():
        sv = oracle_decode_latents(ovae, lat)
        rv = oracle_decode_latents(ovae.float(), lat.float())
    ovae = ovae.to(torch.bfloat16)

    def rel(a, b):
        return float((a.float() - b.float()).abs().max() / b.float().abs().mean())

    def relmean(a, b):
        return float((a.float() - b.float()).abs().mean() / b.float().abs().mean())
    res = {"what": "2 DDIM steps (CFG 9) of config 2 (bf16, CUDA-graph replay) vs the fp32 oracle on the same GPU, same "
                   "random-init weights and inputs; video = VAE decode of the SAME (product) latents by both; 'stock' = "
                   "the same ops through cuDNN/cuBLAS/SDPA in bf16",
           "latents_max_err_over_mean_ref": rel(lat, rl), "latents_mean_err_over_mean_ref": relmean(lat, rl),
           "video_max_err_over_mean_ref": rel(video, rv), "video_mean_err_over_mean_ref": relmean(video, rv),
           "stock_latents_max_err_over_mean_ref": rel(sl, rl), "stock_latents_mean_err_over_mean_ref": relmean(sl, rl),
           "stock_video_max_err_over_mean_ref": rel(sv, rv), "stock_video_mean_err_over_mean_ref": relmean(sv, rv)}
    res["ok"] = bool(res["latents_mean_err_over_mean_ref"] <= 2.0 * res["stock_latents_mean_err_over_mean_ref"] + 1e-3
                     and res["video_mean_err_over_mean_ref"] <= 2.0 * res["stock_video_mean_err_over_mean_ref"] + 1e-3)
    return res, ounet, ovae


def torch_eager_leg(ounet, ovae, devin, dev, e2e_value):
    """The comparison the north star names: the reference's op sequence through stock torch (cuDNN / cuBLAS / SDPA) in
    bf16 on the SAME GPU (the oracle modules; real diffusers is not installable).  Outside the timed region."""
    import torch
    from oracle.composition import DDIMScheduler as ODDIM, oracle_decode_latents, oracle_sampling_loop
    sample = devin["latents"].expand(2, -1, -1, -1, -1).contiguous()
    cond2 = torch.cat([devin["condition_latent"]] * 2)
    ehs = torch.cat([devin["negative_prompt_embeds"], devin["prompt_embeds"]])
    mot = torch.tensor([4.0], device=dev)
    with torch.no_grad():
        unet_ms = _ev_ms(lambda: ounet(sample, 500, ehs, cond2, devin["mask"], motion=mot), reps=3, warm=1)
        vae_ms = _ev_ms(lambda: oracle_decode_latents(ovae, devin["latents"]), reps=2, warm=1)
        clip_ms = _ev_ms(lambda: oracle_sampling_loop(ounet, ODDIM(**SCHED), devin["latents"], devin["prompt_embeds"],
                                                      devin["negative_prompt_embeds"], devin["condition_latent"],
                                                      devin["mask"], [4], GUIDANCE, STEPS_DDIM, vae=ovae), reps=1, warm=0)
    fps = FRAMES / (clip_ms / 1e3)
    return {"what": "oracle modules (the reference's op sequence) in bf16 through stock torch on the same GPU, device-"
                    "resident inputs, 1 clip", "unet_fwd_ms": unet_ms, "vae_decode_16f_ms": vae_ms,
            "clip_s": clip_ms / 1e3, "frames_per_s": fps, "this_repo_e2e_over_torch_eager": e2e_value / fps}


def kernel_rooflines(pipe, devin, dev):
    """Per-kernel CUDA-event timing of ONE eager UNet forward (config 2): tensor roofline of the implicit GEMM (dominant)
    and of flash attention, HBM roofline of the norm / temporal-attention kernels (algorithmic bytes, SURVEY 8d)."""
    import torch
    from animate_anything_b200 import ops
    peak_tf, peak_hbm, peak_src = _peaks()
    sample = devin["latents"].expand(2, -1, -1, -1, -1)
    cond2 = torch.cat([devin["condition_latent"]] * 2)
    ehs = torch.cat([devin["negative_prompt_embeds"], devin["prompt_embeds"]])
    tt = torch.tensor([500.0], device=dev)
    mot = torch.tensor([4.0], device=dev)

    def fwd():
        pipe.unet(sample, tt, ehs, condition_latent=cond2, mask=devin["mask"], motion=mot, _raw_eps=True)
    unet_ms = _ev_ms(fwd, reps=3, warm=2)
    ops.IGEMM_PROFILE = []
    fwd()
    torch.cuda.synchronize()
    prof = ops.IGEMM_PROFILE
    ops.IGEMM_PROFILE = None
    tot_ms = sum(p["ev"][0].elapsed_time(p["ev"][1]) for p in prof)
    tot_fl = sum(p["flops"] for p in prof)
    achieved = tot_fl / (tot_ms * 1e-3) / 1e12
    traffic = None
    tp = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(tp):
        try:
            traffic = json.load(open(tp)).get("igemm_dram_bytes_per_launch")
        except Exception:
            traffic = None
    roof = {"bound": "tensor", "kernel": "aab::igemm_kernel (tcgen05 implicit GEMM, all launches of one UNet forward)",
            "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf, "traffic": traffic,
            "peak_source": peak_src, "launches": len(prof), "algorithmic_tflop_per_forward": tot_fl / 1e12,
            "igemm_ms_per_forward": tot_ms, "avg_launch_us": tot_ms * 1e3 / max(1, len(prof))}
    ops.KERNEL_PROFILE = []
    fwd()
    torch.cuda.synchronize()
    kp = ops.KERNEL_PROFILE
    ops.KERNEL_PROFILE = None
    other = {}
    for name in sorted({p["name"] for p in kp}):
        sel = [p for p in kp if p["name"] == name]
        ms = sum(p["ev"][0].elapsed_time(p["ev"][1]) for p in sel)
        by = sum(p["bytes"] for p in sel)
        fl = sum(p["flops"] for p in sel)
        ent = {"launches": len(sel), "ms_per_forward": ms, "algorithmic_GB": by / 1e9}
        if name == "flash_attn_d64":
            ent.update(bound="tensor", achieved=fl / (ms * 1e-3) / 1e12, peak=peak_tf, unit="TFLOP/s")
        else:
            ent.update(bound="hbm", achieved=by / (ms * 1e-3) / 1e9, peak=peak_hbm, unit="GB/s")
        ent["frac"] = ent["achieved"] / ent["peak"]
        other[name] = ent
    roof["other_kernels"] = other
    return roof, unet_ms


def run_product(args):
    import torch
    import torch.distributed as dist
    from animate_anything_b200 import _lib
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dtype = torch.bfloat16
    pipe = build_models(dev, dtype)
    pipe.use_cuda_graph = not args.no_graph
    latency = args.mode == "latency" and world > 1
    kw = dict(motion=[4], guidance_scale=GUIDANCE, num_inference_steps=STEPS_DDIM, return_dict=False)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    if latency:
        # BASELINE config 3 ("CFG batch=8 = 4 prompts x cond/uncond, sharded across 8 GPUs"): N=2 -> ONE clip with its CFG
        # halves on two GPUs; N=4 -> 4 prompts, pairs co-located; N=8 -> 4 prompts, one batch element per GPU.
        from animate_anything_b200.parallel import LatencyShardedPipeline
        n_prompts = 1 if world == 2 else 4
        if world not in (2, 4, 8):
            raise SystemExit("--mode latency supports 2, 4 or 8 GPUs")
        host = _stack_inputs(n_prompts, pinned=True)
        devin = {k: v.to(dev) for k, v in host.items()}
        runner = LatencyShardedPipeline(pipe, n_prompts)
        clips_per_step = n_prompts

        def one_clip(inp):
            return runner(inp["prompt_embeds"], inp["negative_prompt_embeds"], inp["latents"], inp["condition_latent"],
                          mask=inp["mask"], **{k: v for k, v in kw.items() if k != "return_dict"})
    else:
        host = synth_inputs(rank)
        devin = {k: v.to(dev) for k, v in host.items()}
        clips_per_step = world
        gather_buf = torch.empty((world, FRAMES, HW, HW, 3), dtype=torch.uint8, device=dev) if world > 1 else None

        def one_clip(inp):
            # N = 1: float video on the device ("pt"); N > 1: uint8 frames from the fused decoder tail, then the one
            # collective of the path: all-gather of the decoded frames (12.6 MB per clip)
            video, lat = pipe(prompt_embeds=inp["prompt_embeds"], negative_prompt_embeds=inp["negative_prompt_embeds"],
                              latents=inp["latents"], condition_latent=inp["condition_latent"], mask=inp["mask"],
                              output_type="pt" if world == 1 else "u8", **kw)
            if world > 1:
                dist.all_gather_into_tensor(gather_buf, video.unsqueeze(0))
            return video, lat

    for _ in range(args.warmup):
        one_clip(devin)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ncu_window = bool(os.environ.get("AAB_BENCH_NCU"))   # `ncu --profile-from-start off`: launch list of the timed region only
    if ncu_window:
        torch.cuda.profiler.start()
    e0.record()
    for _ in range(args.steps):
        video, lat = one_clip(devin)
    e1.record()
    if ncu_window:
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
    barrier()
    if args.dump_outputs and rank == 0:   # here: the calls below reuse the CUDA graph's output buffers
        dump_outputs(args.dump_outputs, {"video": video, "latents": lat})
    t_dev = torch.tensor([e0.elapsed_time(e1) / 1e3], device=dev, dtype=torch.float64)
    launches = _lib.launch_count() - l0
    if pipe.use_cuda_graph:            # python-side calls happen once at capture; every replay re-launches them
        per_step = getattr(pipe, "graph_kernels_per_step", None)
        launches = launches + (per_step or 0) * STEPS_DDIM * args.steps
    finite = bool(torch.isfinite(lat.float()).all().item())

    # ---- e2e: the call a user makes -- pinned HOST inputs copied in every step, the decoded uint8 frames (decode +
    # tensor2vid fused on the device) read back to the host every step
    h2d = sum(v.numel() * v.element_size() for v in host.values())
    d2h = FRAMES * HW * HW * 3 * (clips_per_step if latency else 1)
    barrier()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record()
    for _ in range(args.steps):
        inp = {k: v.to(dev, non_blocking=True) for k, v in host.items()}
        if latency:
            frames, _ = one_clip(inp)
            frames_host = frames.cpu()
            assert frames_host.shape[:2] == (clips_per_step, FRAMES) and frames_host.dtype == torch.uint8
        else:
            frames, _ = pipe(prompt_embeds=inp["prompt_embeds"], negative_prompt_embeds=inp["negative_prompt_embeds"],
                             latents=inp["latents"], condition_latent=inp["condition_latent"], mask=inp["mask"],
                             output_type="np", **kw)
            assert len(frames) == FRAMES and frames[0].dtype.name == "uint8"
    e3.record()
    barrier()
    sampler.stop_flag = True
    t_e2e = torch.tensor([e2.elapsed_time(e3) / 1e3], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t_dev, op=dist.ReduceOp.MAX)
        dist.all_reduce(t_e2e, op=dist.ReduceOp.MAX)
    total_frames = FRAMES * clips_per_step * args.steps
    value = total_frames / t_dev.item()
    e2e_v = total_frames / t_e2e.item()

    lat_info = None
    if latency:
        lat_info = latency_breakdown(pipe, runner, devin, dev, rank, world, lat, video, kw, t_dev.item() / args.steps)

    roof = unet_ms = cpu_base = parity = eager = vae_ms = None
    if rank == 0 and not latency:
        saved_graph = pipe.use_cuda_graph
        pipe.use_cuda_graph = False
        roof, unet_ms = kernel_rooflines(pipe, devin, dev)
        vae_ms = _ev_ms(lambda: pipe.vae.decode_frames_uint8(devin["latents"]), reps=3, warm=1)
        pipe.use_cuda_graph = saved_graph
        if world == 1 and not args.no_parity:
            try:
                parity, ounet, ovae = parity_check(pipe, devin, dev, dict(kw, output_type="pt"))
                eager = torch_eager_leg(ounet, ovae, devin, dev, e2e_v / world)
                del ounet, ovae
            except Exception as ex:      # the oracle is a checker; never let it break the bench line
                parity = {"ok": None, "failed": repr(ex)}
        if world == 1 and not args.no_cpu_baseline:
            try:
                _, fwd, f_sample, desc, threads = _oracle_unet_sample()
                ts = fwd(f_sample, LAT)
                cpu_base = {"value": cpu_frames_per_sec(ts, f_sample), "unit": UNIT, "cores": threads, "kind": "port",
                            "sample": desc + f" ({ts:.1f} s); x(17/T) x 2 (CFG) x 50 steps, extrapolated"}
            except Exception as ex:
                cpu_base = {"value": None, "unit": UNIT, "cores": os.cpu_count(), "kind": "port", "sample": f"failed: {ex}"}
    if rank == 0:
        if latency:
            workload = (f"config3 ({clips_per_step} prompt(s) x cond/uncond, 16x512x512, 50 DDIM steps, CFG 9) on {world} "
                        f"GPUs: " + ("CFG halves of ONE clip on two GPUs (per-step all-gather of the fp32 noise prediction)"
                                     if world == 2 else "pairs co-located, no per-step traffic" if world == 4 else
                                     "one batch element per GPU (pair exchange per step)") +
                        "; VAE decode frame-sharded inside a pair; one NCCL all-gather of uint8 frames")
            par = {2: "cfg2", 4: "prompts4", 8: "prompts4 x cfg2"}[world]
        else:
            workload = ("config2: LatentToVideoPipeline.__call__ 16x512x512, 50 DDIM steps, CFG 9, random-init UNet3D "
                        "(1.41B) + SD VAE, 1 clip per GPU")
            par = f"clips x{world} (prompt-sharded), 1 NCCL all-gather of frames" if world > 1 else "single GPU"
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": t_dev.item() / args.steps * 1e3, "higher_is_better": True,
                "scaling": "strong" if latency else "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                "mode": args.mode if world > 1 else "throughput",
                "config": {"workload": workload,
                           "l2_policy": "working set per UNet forward (2.8 GB weights + activations) >> 126 MB L2",
                           "cuda_graph": not args.no_graph, "finite_output": finite, "parallelism": par,
                           "parity_check": parity},
                "unet_fwd_ms_per_step": unet_ms, "vae_decode_16f_ms": vae_ms, "clocks": sampler.summary(),
                "e2e": {"value": e2e_v, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
                "gpu_launches": launches, "roofline": roof, "cpu_baseline": cpu_base, "torch_eager_gpu": eager}
        if lat_info is not None:
            line["latency"] = lat_info
        print(json.dumps(line), flush=True)
    if world > 1:
        # orderly shutdown: captured graphs hold NCCL kernels of the pair communicators -- drop them before the process
        # group goes away; a watchdog ends the process if the teardown still blocks (the result line is already out)
        import gc
        dist.barrier()
        torch.cuda.synchronize()
        pipe.__dict__.pop("_gstate", None)
        gc.collect()
        torch.cuda.synchronize()
        sys.stdout.flush()
        wd = threading.Timer(20.0, lambda: os._exit(0))
        wd.daemon = True
        wd.start()
        dist.destroy_process_group()
        wd.cancel()


def latency_breakdown(pipe, runner, devin, dev, rank, world, lat_split, frames_split, kw, clip_s):
    """Names the limiter of the split run with numbers (rank 0, CUDA events): the UNet half forward, the per-step
    all-gather of the noise prediction, the fused CFG+scheduler step, the sharded VAE decode, the frame all-gather; and
    checks the split result against the same clip computed on ONE GPU (rank 0 alone), bit for bit."""
    import torch
    import torch.distributed as dist
    from animate_anything_b200 import ops
    info = {"clip_latency_s": clip_s, "clips_in_flight": runner.n_prompts, "ranks_per_prompt": runner.ranks_per_prompt}
    i = runner.prompt
    one = {k: (v if k == "mask" else v[i: i + 1]) for k, v in devin.items()}
    tt = torch.tensor([500.0], device=dev)
    mot = torch.tensor([4.0], device=dev)
    graph = pipe.use_cuda_graph
    if runner.ranks_per_prompt == 2:
        pair = runner.pair
        r = dist.get_rank(pair)
        ehs = (one["negative_prompt_embeds"], one["prompt_embeds"])[r]
        pipe.use_cuda_graph = False

        def half():
            return pipe.unet(one["latents"], tt, ehs, condition_latent=one["condition_latent"], mask=one["mask"],
                             motion=mot, _raw_eps=True)
        info["unet_half_fwd_ms"] = _ev_ms(half, reps=3, warm=2)
        eps_half, _ = half()
        buf = torch.empty((2,) + tuple(eps_half.shape), dtype=eps_half.dtype, device=dev)
        info["eps_allgather_us"] = 1e3 * _ev_ms(lambda: dist.all_gather_into_tensor(buf, eps_half.unsqueeze(0), group=pair),
                                                reps=20, warm=3)
        info["eps_allgather_bytes"] = int(buf.numel() * buf.element_size())
        f = lat_split.shape[2]
        info["vae_decode_half_ms"] = _ev_ms(lambda: pipe.vae.decode_frames_uint8(lat_split[:, :, : f // 2].contiguous()),
                                            reps=2, warm=1)
    fr = torch.empty((world,) + tuple(frames_split.shape[1:]), dtype=torch.uint8, device=dev) \
        if runner.ranks_per_prompt == 1 else torch.empty((world, FRAMES // 2, HW, HW, 3), dtype=torch.uint8, device=dev)
    src = fr[0].clone()
    info["frames_allgather_ms"] = _ev_ms(lambda: dist.all_gather_into_tensor(fr, src.unsqueeze(0)), reps=5, warm=2)
    info["frames_allgather_bytes"] = int(fr.numel())
    # the same clip(s) on ONE GPU: rank 0 alone, the others wait at the barrier
    saved = pipe.cfg_group
    pipe.cfg_group = None
    pipe.use_cuda_graph = graph
    dist.barrier()
    if rank == 0:
        kw1 = {k: v for k, v in kw.items() if k != "return_dict"}

        def single():
            return pipe(prompt_embeds=one["prompt_embeds"], negative_prompt_embeds=one["negative_prompt_embeds"],
                        latents=one["latents"], condition_latent=one["condition_latent"], mask=one["mask"],
                        output_type="u8", return_dict=False, **kw1)
        single()
        ms = _ev_ms(single, reps=1, warm=0)
        f1, l1 = single()
        info["one_gpu_clip_s"] = ms / 1e3
        info["speedup_vs_one_gpu_same_clips"] = (ms / 1e3) * runner.n_prompts / clip_s
        info["latents_bit_identical_to_1gpu"] = bool(torch.equal(l1, lat_split))
        info["frames_bit_identical_to_1gpu"] = bool(torch.equal(f1, frames_split[0]))
    dist.barrier()
    pipe.cfg_group = saved
    return info


def run_svd(args):
    """BASELINE config 4 (opt-in: `--workload svd`; the driver's default line stays config 2): the SVD path of
    train_svd.py:756-777 -- MaskStableVideoDiffusionPipeline.__call__, 25 frames x 576 x 1024, 25 Euler steps, per-frame
    CFG 1 -> 3, full-size random-init UNetSpatioTemporalConditionModel (9 input channels) + AutoencoderKLTemporalDecoder,
    bf16, 1 GPU.  The CLIP vision tower is outside the hot path: a synthetic image embedding is passed in."""
    import torch
    from animate_anything_b200 import _lib
    from animate_anything_b200.autoencoder_kl_temporal_decoder import AutoencoderKLTemporalDecoder
    from animate_anything_b200.pipeline_svd import MaskStableVideoDiffusionPipeline
    from animate_anything_b200.schedulers import EulerDiscreteScheduler
    from animate_anything_b200.unet_spatio_temporal_condition import UNetSpatioTemporalConditionModel
    from oracle.composition import SVD_SCHED
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    dtype = torch.bfloat16
    nf, hh, ww, steps = 25, 576, 1024, 25
    torch.manual_seed(0)
    with torch.device(dev):
        # the released SVD checkpoints' config (heads 5/10/20/20 = head dim 64 everywhere; the class default has a 10 at level 2)
        unet = UNetSpatioTemporalConditionModel(in_channels=9, sample_size=96, num_attention_heads=(5, 10, 20, 20))
        vae = AutoencoderKLTemporalDecoder()
    with torch.no_grad():
        for n, p in unet.named_parameters():
            if p.abs().max() == 0:
                p.normal_(0.0, 0.02)
    pipe = MaskStableVideoDiffusionPipeline(vae=vae.to(dtype).eval(), image_encoder=None, unet=unet.to(dtype).eval(),
                                            scheduler=EulerDiscreteScheduler(**SVD_SCHED))
    g = torch.Generator().manual_seed(7)
    host = {"image": torch.randn(1, 3, hh, ww, generator=g).clamp(-1, 1).pin_memory(),
            "mask": (torch.rand(1, hh // 8, ww // 8, generator=g) > 0.5).float().pin_memory(),
            "latents": torch.randn(1, nf, 4, hh // 8, ww // 8, generator=g).to(dtype).pin_memory(),
            "emb": torch.randn(1, 1, 1024, generator=g).to(dtype).pin_memory()}

    def clip(inp, output_type="pt"):
        return pipe(inp["image"], height=hh, width=ww, num_frames=nf, num_inference_steps=steps, decode_chunk_size=8,
                    latents=inp["latents"], mask=inp["mask"], image_embeddings=inp["emb"], output_type=output_type,
                    return_dict=False)
    devin = {k: v.to(dev) for k, v in host.items()}
    for _ in range(args.warmup):
        clip(devin)
    torch.cuda.synchronize()
    sampler = ClockSampler(0)
    sampler.start()
    l0 = _lib.launch_count()
    last = []

    def timed_clip():
        last[:] = clip(devin)
    t_dev = _ev_ms(timed_clip, reps=args.steps, warm=0) / 1e3
    launches = _lib.launch_count() - l0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"frames": torch.stack(last)})

    def e2e():
        inp = {k: v.to(dev, non_blocking=True) for k, v in host.items()}
        fr = clip(inp)                                   # list of [F, 3, H, W] in [0, 1] on the device
        return (fr[0] * 255).to(torch.uint8).cpu()       # the frames leave the device as uint8
    t_e2e = _ev_ms(e2e, reps=args.steps, warm=0) / 1e3
    sampler.stop_flag = True
    # UNet forward alone (B = 2 CFG halves, 25 frames, 72 x 128 latents)
    from animate_anything_b200 import ops
    x16 = ops.svd_in_assemble(devin["latents"], torch.zeros(1, 4, hh // 8, ww // 8, device=dev, dtype=dtype),
                              devin["mask"].to(dtype).reshape(hh // 8, ww // 8).contiguous(), 1.0, True)
    emb2 = torch.cat([torch.zeros_like(devin["emb"]), devin["emb"]])
    ids = torch.tensor([[6.0, 127.0, 0.02]] * 2, device=dev)
    unet_ms = _ev_ms(lambda: pipe.unet(None, 1.0, emb2, ids, _raw=True, _x16=x16, _shape=(2, nf, 9, hh // 8, ww // 8)),
                     reps=3, warm=1)
    line = {"metric": "denoised_frames_per_sec_25f_576x1024_25euler_svd", "value": nf / t_dev, "unit": UNIT, "n_gpus": 1,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": t_dev * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": "config4: MaskStableVideoDiffusionPipeline.__call__ 25x576x1024, 25 Euler steps, per-frame CFG "
                                   "1->3, random-init UNetSpatioTemporalConditionModel (9-ch) + AutoencoderKLTemporalDecoder, "
                                   "decode_chunk_size 8; image embedding synthetic (CLIP vision tower outside the hot path)",
                       "l2_policy": "working set per UNet forward >> 126 MB L2", "cuda_graph": False},
            "unet_fwd_ms_per_step": unet_ms, "clocks": sampler.summary(),
            "e2e": {"value": nf / t_e2e, "unit": UNIT, "h2d_bytes_per_step": sum(v.numel() * v.element_size() for v in host.values()),
                    "d2h_bytes_per_step": nf * 3 * hh * ww},
            "gpu_launches": launches}
    print(json.dumps(line), flush=True)


def run_vae(args):
    """BASELINE config 5 (opt-in: `--workload vae`): VAE-only throughput sweep.  N frames (64 ... 1024) are split evenly over
    the ranks; every rank decodes its latent frames to uint8 (fused tail) and encodes as many 512x512 images; the decoded
    frames are all-gathered (the path's one collective).  Per N: frames/s (max over ranks) and achieved tensor TFLOP/s
    against the measured peak (2.515 TFLOP per decoded frame, 1.117 per encoded frame: BASELINE.md section 4)."""
    import torch
    import torch.distributed as dist
    from animate_anything_b200.autoencoder_kl import AutoencoderKL
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dtype = torch.bfloat16
    torch.manual_seed(0)
    with torch.device(dev):
        vae = AutoencoderKL()
    vae = vae.to(dtype).eval()
    peak_tf, _, peak_src = _peaks()
    rows = []
    g = torch.Generator().manual_seed(3 + rank)
    for n_total in (64, 128, 256, 512, 1024):
        n = n_total // world
        lat = torch.randn(1, 4, n, LAT, LAT, generator=g).to(dtype).to(dev)
        img = torch.randn(min(n, 64), 3, HW, HW, generator=g).clamp(-1, 1).to(dtype).to(dev)      # encoded in rounds of <= 64
        gather = torch.empty((world, n, HW, HW, 3), dtype=torch.uint8, device=dev) if world > 1 else None
        outs = {}

        def decode():
            fr = vae.decode_frames_uint8(lat)
            if world > 1:
                dist.all_gather_into_tensor(gather, fr.unsqueeze(0))
            outs["frames"] = fr

        def encode():
            done = 0
            while done < n:
                k = min(img.shape[0], n - done)
                outs["latent_parameters"] = vae.encode(img[:k]).latent_dist.parameters
                done += k
        t_dec = torch.tensor([_ev_ms(decode, reps=args.steps, warm=args.warmup)], device=dev, dtype=torch.float64)
        t_enc = torch.tensor([_ev_ms(encode, reps=args.steps, warm=args.warmup)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t_dec, op=dist.ReduceOp.MAX)
            dist.all_reduce(t_enc, op=dist.ReduceOp.MAX)
        d_fps = n_total / (t_dec.item() / 1e3)
        e_fps = n_total / (t_enc.item() / 1e3)
        rows.append({"frames": n_total, "decode_frames_per_s": d_fps, "encode_frames_per_s": e_fps,
                     "decode_tflops_per_gpu": d_fps * 2.515 / world, "encode_tflops_per_gpu": e_fps * 1.117 / world,
                     "decode_frac_of_peak": d_fps * 2.515 / world / peak_tf, "encode_frac_of_peak": e_fps * 1.117 / world / peak_tf})
        del lat, img, gather
        torch.cuda.empty_cache()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, outs)
    if rank == 0:
        last = rows[-1]
        line = {"metric": "vae_decode_frames_per_sec_512x512", "value": last["decode_frames_per_s"], "unit": UNIT,
                "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": 1024 / last["decode_frames_per_s"] * 1e3,
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                "config": {"workload": "config5: AutoencoderKL (SD VAE, random init) decode [N,4,64,64] -> uint8 512x512 frames and "
                                       "encode [N,3,512,512], N = 64..1024 split evenly over the GPUs, one all-gather of decoded frames",
                           "peak_source": peak_src},
                "sweep": rows}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()
        wd = threading.Timer(20.0, lambda: os._exit(0))
        wd.daemon = True
        wd.start()
        dist.destroy_process_group()
        wd.cancel()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-graph", action="store_true", help="disable CUDA-graph replay of the denoising step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the oracle parity check and the torch-eager leg")
    ap.add_argument("--mode", default="throughput", choices=["throughput", "latency"],
                    help="N>1 only. throughput (default, what the driver's scaling run uses): one clip per GPU. latency: "
                         "BASELINE config 3 -- N=2 one clip with its CFG halves on two GPUs; N=4 four prompts, pairs "
                         "co-located; N=8 four prompts, one batch element per GPU")
    ap.add_argument("--workload", default="config2", choices=["config2", "svd", "vae"],
                    help="config2 (default, BASELINE's headline), svd (BASELINE config 4, 1 GPU) or vae (config 5: VAE-only "
                         "sweep, frames split over the GPUs); svd / vae exist for this repo's arm only")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned (rank 0) as DIR/<name>.npy, float32, "
                         "64 MB at most (larger outputs as a fixed seeded sample); inputs and weights are seeded")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs records this repo's arm; the reference arm times a bounded CPU sample only")
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "svd":
        run_svd(args)
    elif args.workload == "vae":
        run_vae(args)
    else:
        run_product(args)


if __name__ == "__main__":
    main()
