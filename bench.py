#!/usr/bin/env python
"""Headline benchmark: frames/sec of MotionClone's guided denoising loop (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            this package, one process per GPU (torchrun for N > 1)
  python bench.py --impl reference --steps K --warmup W     the reference's CPU path (oracle port) on the host cores
  python bench.py ... --dump-outputs DIR                    also write the last timed step's latents to DIR/*.npy

A "step" is one sample: the latent -> latent 50-step DDIM loop (reference sample_video, motionclone_functions.py:164-167)
at BASELINE.json configs[1]: t2v_object, 16 x 512 x 512, random-init SD1.5 + v3_sd15_mm widths, fp16. The shipped YAML
(300 steps / 180 guided / guidance_scale 0.4) is mapped to 50 steps as BASELINE.md §4 states: 30 guided steps,
guidance_scale 0.4, warm_up = cool_up = 10. VAE, CLIP and video I/O are excluded (synthetic latents / embeddings).
One JSON line on stdout (rank 0); everything else goes to stderr.
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

import torch  # noqa: E402

METRIC = "frames/sec at 16x512x512 T2V, 50-step DDIM"
UNIT = "frames/s"
_BASE = dict(cfg_scale=7.5, negative_prompt="", warm_up_steps=10, cool_up_steps=10, motion_guidance_weight=2000,
             motion_guidance_blocks=["up_blocks.1"], add_noise_step=400, inference_steps=50, height=512, width=512,
             new_prompt="synthetic")
# BASELINE.json configs -> 50-step mappings of the shipped YAMLs (BASELINE.md §4: guided fraction and timestep split kept)
CONFIGS = {
    # configs[1] (the headline: BENCH / SCALE stay comparable round over round)
    "object": dict(_BASE, video_length=16, guidance_steps=30, guidance_scale=0.4,
                   workload="t2v_object 16x512x512, 50-step DDIM (30 guided, guidance_scale 0.4), random-init SD1.5 + "
                            "v3_sd15_mm widths, 1 sample per step per GPU"),
    # configs[2]: t2v_camera, one shared reference clip, a different prompt per sample / rank
    "camera": dict(_BASE, video_length=16, guidance_steps=25, guidance_scale=0.3, distinct_prompts=True,
                   workload="t2v_camera 16x512x512, 50-step DDIM (25 guided, guidance_scale 0.3), one shared clip, a distinct "
                            "prompt per sample, random-init SD1.5 + v3_sd15_mm widths, 1 sample per step per GPU"),
    # configs[3]: i2v_rgb + SparseCtrl (latent condition, simplified embedding)
    "rgb": dict(_BASE, video_length=16, guidance_steps=20, guidance_scale=0.3, sparsectrl="latent", image_index=[0],
                controlnet_scale=1.0,
                workload="i2v_rgb + SparseCtrl latent condition 16x512x512, 50-step DDIM (20 guided, guidance_scale 0.3), "
                         "random-init SD1.5 + v3_sd15_mm + SparseCtrl widths, 1 sample per step per GPU"),
    # configs[4]: i2v_sketch + SparseCtrl (image condition, conv embedding), 32 frames (positional-encoding limit)
    "sketch": dict(_BASE, video_length=32, guidance_steps=30, guidance_scale=0.4, sparsectrl="image", image_index=[0],
                   controlnet_scale=1.0,
                   workload="i2v_sketch + SparseCtrl image condition 32x512x512, 50-step DDIM (30 guided, guidance_scale "
                            "0.4), random-init SD1.5 + v3_sd15_mm + SparseCtrl widths, 1 sample per step per GPU"),
}


def workload_of(args):
    c = dict(CONFIGS[args.config])
    workload = c.pop("workload")
    distinct = c.pop("distinct_prompts", False)
    if args.ddim_steps != 50:  # profiling only
        c["guidance_steps"] = int(round(args.ddim_steps * c["guidance_steps"] / 50))
        c["inference_steps"] = args.ddim_steps
    return c, workload, distinct


def config_block(infer, workload, world):
    """Identical for both arms (the driver compares the dicts): what is computed, not how."""
    return {"workload": workload, "ddim_steps": infer["inference_steps"], "guided_steps": infer["guidance_steps"],
            "video_length": infer["video_length"], "replicas": world,
            "l2": "inputs larger than L2 (2.6 GB of weights stream through every UNet forward)"}


def log(*a):
    print(*a, file=sys.stderr, flush=True)


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self._stop_evt = index, [], threading.Event()

    def run(self):
        while not self._stop_evt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i",
                                      str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([c.strip() for c in out.splitlines()[0].split(",")])
            except Exception:
                pass
            self._stop_evt.wait(0.2)

    def finish(self):
        self._stop_evt.set()
        self.join(timeout=6)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        sm = [float(s[0]) for s in self.samples if s[0].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for j, n in enumerate(names) if any(s[3 + j].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": float(self.samples[0][1]),
                "power_w_max": max(float(s[2]) for s in self.samples), "samples": len(self.samples),
                "reasons": reasons}


# ----------------------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the oracle port (oracle/mc_oracle.py) in fp32 on the host cores
# ----------------------------------------------------------------------------------------------------------------
# analytic forward-equivalents (BASELINE.md §3): backward over the grad-carrying 57 % of the UNet costs ~2x its forward
GUIDED_FWD_EQUIV = 2.0 + 2 * 0.57   # uncond forward + cond forward + partial backward
PLAIN_FWD_EQUIV = 2.0               # one b=2 forward


def _physical_cores() -> int:
    """Physical cores of the host (SMT siblings counted once): the thread count the CPU arm uses. Oversubscribing the
    hyper-threads of a shared box made the round-1 probe vary 12x between boxes."""
    try:
        seen = set()
        phys = core = None
        for line in open("/proc/cpuinfo"):
            if line.startswith("physical id"):
                phys = line.split(":")[1].strip()
            elif line.startswith("core id"):
                core = line.split(":")[1].strip()
            elif not line.strip() and phys is not None and core is not None:
                seen.add((phys, core))
                phys = core = None
        if seen:
            return min(len(seen), len(os.sched_getaffinity(0)))
    except Exception:
        pass
    return max(1, len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1))


def _synthetic_representation(infer):
    L, hw = infer["video_length"], (infer["height"] // 32) * (infer["width"] // 32)
    g = torch.Generator().manual_seed(0)  # a synthetic motion representation of the right shape (timing only)
    names = [f"up_blocks.1.motion_modules.{i}.temporal_transformer.transformer_blocks.0.attention_blocks.{j}"
             for i in range(3) for j in range(2)]
    return {n: [torch.rand(hw, 8, L, 1, generator=g), torch.randint(0, L, (hw, 8, L, 1), generator=g).to(torch.uint8)]
            for n in names}


def cpu_reference_steps(budget_s: float, infer: dict):
    """CPU oracle (fp32, one thread per PHYSICAL core) at the bench shapes. Order of work, each stage only if the stages
    so far predict it fits the budget: (1) a b=1 UNet forward at a quarter of the pixels (always; ~1/4.33 of a forward),
    (2) ONE REAL plain DDIM step (b=2 forward + CFG + DDIM), (3) ONE REAL guided step (forward, forward + backward,
    loss, CFG + DDIM). What was not run is extrapolated from what was with the analytic forward-equivalents above, and
    the returned info says which is which and carries every wall time, so box-to-box variance is visible.
    Returns (t_guided, t_plain, info). Only place bench.py executes oracle/ (task spec ④)."""
    from motionclone_b200.synthetic import UNET_SD15_CONFIG, synthetic_inputs, synthetic_state_dict
    from motionclone_b200.unet3d import UNet3DConditionModel
    from oracle import mc_oracle as O

    cores = _physical_cores()
    torch.set_num_threads(cores)
    with torch.device("meta"):
        shapes = {k: v.shape for k, v in UNet3DConditionModel(**UNET_SD15_CONFIG).state_dict().items()}
    t0 = time.time()
    sd = synthetic_state_dict(shapes, 42)
    log(f"[cpu] fp32 weights in {time.time() - t0:.0f}s; {cores} threads (physical cores; {os.cpu_count()} logical)")
    L = infer["video_length"]
    inp = synthetic_inputs(L, infer["height"], infer["width"], 768, 42)
    rep = _synthetic_representation(infer)
    timesteps = O.uneven_timesteps(infer["inference_steps"], infer["guidance_steps"], infer["guidance_scale"])
    acp = O.alphas_cumprod()
    lat, text = inp["noisy_latents"], inp["text_embeddings"]
    start = time.time()
    # (1) probe: all L frames (the threads parallelise over the frame batch as in the full problem), a quarter of the
    # pixels; analytic FLOP ratio full : probe = 17.67 : 4.08 TFLOP (SURVEY.md §6; the N^2 self-attention term makes it
    # 4.33, not 4)
    PROBE_HW, PROBE_SCALE = 256, 17.67 / 4.08
    probe = synthetic_inputs(L, PROBE_HW, PROBE_HW, 768, 42)["noisy_latents"]
    with torch.no_grad():
        t0 = time.time()
        O.unet_forward(sd, UNET_SD15_CONFIG, probe, int(timesteps[0]), text[[0]])
        t_probe = time.time() - t0
    t_fwd = t_probe * PROBE_SCALE
    log(f"[cpu] probe: b=1 UNet forward at {L}x{PROBE_HW}x{PROBE_HW} {t_probe:.1f}s -> {t_fwd:.1f}s per full forward (x{PROBE_SCALE:.2f})")
    info = dict(cores=cores, logical_cpus=os.cpu_count(), probe_wall_s=t_probe, s_per_forward=t_fwd, plain_measured=False,
                guided_measured=False)
    t_plain, t_guided = PLAIN_FWD_EQUIV * t_fwd, GUIDED_FWD_EQUIV * t_fwd
    if (time.time() - start) + 1.15 * t_plain < budget_s:   # (2) one real plain step
        t0 = time.time()
        O.single_step(sd, UNET_SD15_CONFIG, infer, lat, infer["guidance_steps"], timesteps, acp, text, rep)
        t_plain = time.time() - t0
        t_fwd = t_plain / PLAIN_FWD_EQUIV
        t_guided = GUIDED_FWD_EQUIV * t_fwd
        info.update(plain_measured=True, plain_wall_s=t_plain, s_per_forward=t_fwd)
        log(f"[cpu] real plain step {t_plain:.1f}s")
        if (time.time() - start) + 1.15 * t_guided < budget_s:   # (3) one real guided step
            t0 = time.time()
            O.single_step(sd, UNET_SD15_CONFIG, infer, lat, 0, timesteps, acp, text, rep)
            t_guided = time.time() - t0
            info.update(guided_measured=True, guided_wall_s=t_guided)
            log(f"[cpu] real guided step {t_guided:.1f}s")
    parts = [f"probe forward {L}x{PROBE_HW}x{PROBE_HW} {t_probe:.1f} s"]
    parts.append(f"real plain step {t_plain:.1f} s" if info["plain_measured"] else
                 f"plain step extrapolated ({PLAIN_FWD_EQUIV:.2f} forwards x probe x {PROBE_SCALE:.2f})")
    parts.append(f"real guided step {t_guided:.1f} s" if info["guided_measured"] else
                 f"guided step extrapolated ({GUIDED_FWD_EQUIV:.2f} forward-equivalents)")
    info["measured"] = "; ".join(parts)
    return t_guided, t_plain, info


def fps_from_step_times(t_guided, t_plain, infer):
    G, S = infer["guidance_steps"], infer["inference_steps"]
    return infer["video_length"] / (G * t_guided + (S - G) * t_plain)


def cpu_block(tg, tp, info, infer, fps):
    return {"value": fps, "unit": UNIT, "cores": info["cores"], "kind": "port",
            "sample": f"{info['measured']} at {infer['video_length']}x{infer['height']}x{infer['width']} (fp32 CPU oracle, math "
                      f"attention, {info['cores']} threads = physical cores of {info['logical_cpus']} logical), extrapolated to "
                      f"{infer['inference_steps']} steps ({infer['guidance_steps']} guided)",
            "s_per_guided_step": tg, "s_per_plain_step": tp, "s_per_forward": info["s_per_forward"],
            "probe_wall_s": info["probe_wall_s"], "plain_measured": info["plain_measured"],
            "guided_measured": info["guided_measured"]}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    infer, workload, _ = workload_of(args)
    # the arm's bounded sample is the same for every --steps / --warmup, so the whole run fits the time budget
    tg, tp, info = cpu_reference_steps(args.ref_budget, infer)
    fps = fps_from_step_times(tg, tp, infer)
    line = {"impl": "reference", "device": "cpu", "metric": METRIC, "value": fps, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * infer["video_length"] / fps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_block(infer, workload, args.gpus),
            "arm": f"reference CPU path (oracle port, fp32, {info['cores']} host threads), rank 0 only",
            "cpu_baseline": cpu_block(tg, tp, info, infer, fps),
            "e2e": {"value": fps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    _emit(line)


# ----------------------------------------------------------------------------------------------------------------
# same-GPU comparator (BASELINE.md §4 "B-GPU-ref"): the reference's op sequence in fp16 on this B200
# ----------------------------------------------------------------------------------------------------------------
def gpu_reference_steps(infer: dict, dev, reps: int = 2):
    """The oracle port = the reference's own op sequence (per-frame rearranges, separate q/k/v projections, text
    re-projected per frame, baddbmm/softmax/bmm temporal attention, eager GroupNorm / GEGLU / residual adds, full
    probability tensors + topk + gather + mse_loss, autograd through all of it, eager CFG + DDIM) in fp16 on the same
    device, with torch's fused SDPA standing in for xformers at the spatial-attention seam (attention.py:535-542) as it
    would on the reference's GPU configuration. One warm-up + `reps` timed guided and plain steps (CUDA events)."""
    from motionclone_b200.synthetic import UNET_SD15_CONFIG, synthetic_inputs, synthetic_state_dict
    from motionclone_b200.unet3d import UNet3DConditionModel
    from oracle import mc_oracle as O

    with torch.device("meta"):
        shapes = {k: v.shape for k, v in UNet3DConditionModel(**UNET_SD15_CONFIG).state_dict().items()}
    sd = {k: v.to(dev, torch.float16) for k, v in synthetic_state_dict(shapes, 42).items()}
    inp = synthetic_inputs(infer["video_length"], infer["height"], infer["width"], 768, 42)
    rep = {n: [v[0].to(dev, torch.float16), v[1].to(dev)] for n, v in _synthetic_representation(infer).items()}
    timesteps = O.uneven_timesteps(infer["inference_steps"], infer["guidance_steps"], infer["guidance_scale"])
    acp = O.alphas_cumprod()
    lat, text = inp["noisy_latents"].to(dev, torch.float16), inp["text_embeddings"].to(dev, torch.float16)
    prev = O.SPATIAL_ATTENTION
    O.SPATIAL_ATTENTION = "sdpa"
    try:
        def timed(step_index):
            O.single_step(sd, UNET_SD15_CONFIG, infer, lat, step_index, timesteps, acp, text, rep)  # warm-up
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                O.single_step(sd, UNET_SD15_CONFIG, infer, lat, step_index, timesteps, acp, text, rep)
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / reps / 1e3
        t_guided = timed(0)
        t_plain = timed(infer["guidance_steps"])
    finally:
        O.SPATIAL_ATTENTION = prev
    del sd
    torch.cuda.empty_cache()
    return t_guided, t_plain


# ----------------------------------------------------------------------------------------------------------------
# this package's arm
# ----------------------------------------------------------------------------------------------------------------
def _ncu_traffic():
    """Per-launch DRAM traffic of the roofline kernel from the committed ncu capture (profiles/r02_temporal_traffic.json,
    written by scripts/summarize_traffic.py from `ncu --metrics dram__bytes_read.sum,dram__bytes_write.sum`)."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "r02_temporal_traffic.json")))
    except Exception:
        return None


def run_own_arm(args):
    import motionclone_b200 as mc
    from motionclone_b200 import _lib, dist as mcdist, guidance, ops
    from motionclone_b200.synthetic import (SPARSECTRL_IMAGE_KWARGS, SPARSECTRL_LATENT_KWARGS, UNET_SD15_CONFIG,
                                            synthetic_condition, synthetic_inputs, synthetic_normal)
    import torch.distributed as tdist

    t_init = time.time()
    rank, world, local = mcdist.init_from_env()
    assert torch.cuda.is_available(), "bench.py needs CUDA (no CPU fallback); --impl reference is the CPU arm"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    nccl_init_ms = None
    if world > 1:  # NCCL creates its communicators lazily: pay for that here, outside the broadcast's own timing
        tdist.barrier(device_ids=[local])
        torch.cuda.synchronize()
        nccl_init_ms = (time.time() - t_init) * 1e3
    infer, workload, distinct_prompts = workload_of(args)
    L = infer["video_length"]

    cn_kwargs, use_cn = None, False
    inp = synthetic_inputs(L, infer["height"], infer["width"], 768, 42)
    h = lambda t: t.to(dev, torch.float16)  # noqa: E731
    if infer.get("sparsectrl"):
        kind = infer["sparsectrl"]
        use_cn = True
        cn_kwargs = SPARSECTRL_LATENT_KWARGS if kind == "latent" else SPARSECTRL_IMAGE_KWARGS
        cond = synthetic_condition(kind, len(infer["image_index"]), infer["height"], infer["width"], L, 47)
        images = cond["cond_latents"] if kind == "latent" else cond["cond_images"]
        infer["controlnet_images"] = images.permute(1, 0, 2, 3).unsqueeze(0).half()  # [1, c, n_img, h, w]
        if kind == "image":
            infer["video_pixels"] = cond["clip_pixels"]
    t0 = time.time()
    pipe = mc.build_pipeline(UNET_SD15_CONFIG, infer, device=dev, weight_seed=42, controlnet_kwargs=cn_kwargs,
                             use_cuda_graphs=not args.no_cuda_graphs)
    log(f"[rank {rank}] model built in {time.time() - t0:.0f}s")
    # weak scaling: every rank denoises its own samples (seed 1000 + global sample index) of ONE shared reference clip
    pipe.set_prompt_embeds(h(inp["text_embeddings"]))
    rep = None
    if rank == 0:
        pipe.input_config["video_latents"], pipe.input_config["video_noise"] = h(inp["clip_latents"]), h(inp["clip_noise"])
        rep = pipe.obtain_motion_representation(use_controlnet=use_cn) if use_cn else pipe.obtain_motion_representation()
    manifest = mcdist.representation_manifest(list(guidance.guided_modules(pipe)), (infer["height"] // 32) * (infer["width"] // 32),
                                              8, L)
    torch.cuda.synchronize()
    tb = time.time()
    rep = mcdist.broadcast_representation(rep, dev, manifest)  # B1: the only collective of the path
    torch.cuda.synchronize()
    bcast_ms = (time.time() - tb) * 1e3
    pipe.motion_representation_dict, pipe.motion_representation_path = rep, None

    def sample_latents(i):
        return synthetic_inputs(L, infer["height"], infer["width"], 768, 1000 + rank + world * i)["noisy_latents"]

    def sample_text(i):  # configs[2]: a distinct prompt per sample (row 0 = the shared unconditional embedding)
        t = inp["text_embeddings"].clone()
        if distinct_prompts:
            t[1] = synthetic_normal("text", (2, 77, 768), 2000 + rank + world * i)[1]
        return t

    n_total = args.warmup + 2 * args.steps
    host = [sample_latents(i).half().pin_memory() for i in range(n_total)]
    resident = [t.to(dev) for t in host]
    text_host = [sample_text(i).half().pin_memory() for i in range(n_total)]
    text_res = [t.to(dev) for t in text_host]
    rep_buf, _ = mcdist.pack_representation(rep)
    rep_host = rep_buf.cpu().pin_memory()

    def barrier():
        if world > 1:
            tdist.barrier(device_ids=[local])
        torch.cuda.synchronize()

    def timed(fn, n, offset):
        """(ms of the n steps, what the last step returned)"""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n):
            out = fn(offset + i)
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            tdist.all_reduce(ms, op=tdist.ReduceOp.MAX)
        return ms.item(), out

    def step_resident(i):
        pipe.set_prompt_embeds(text_res[i])
        return pipe.sample_video(noisy_latents=resident[i], return_latents=True, add_controlnet=use_cn)

    out_host = torch.empty(1, 4, L, infer["height"] // 8, infer["width"] // 8, dtype=torch.float16).pin_memory()

    def step_e2e(i):  # public API with HOST buffers: H2D of latents, text, motion representation; D2H of the result
        pipe.set_prompt_embeds(text_host[i].to(dev, non_blocking=True))
        pipe.motion_representation_dict = mcdist.unpack_representation(rep_host.to(dev, non_blocking=True), manifest)
        out = pipe.sample_video(noisy_latents=host[i], return_latents=True, add_controlnet=use_cn)
        out_host.copy_(out, non_blocking=True)
        torch.cuda.synchronize()
        return out_host

    for i in range(args.warmup):
        step_resident(i)
    torch.cuda.synchronize()

    clocks = ClockSampler(local)
    clocks.start()
    _lib.reset_launch_count()
    ms, last = timed(step_resident, args.steps, args.warmup)
    outputs = {"latents": last.float().cpu()} if args.dump_outputs else None
    launches = _lib.launch_count()
    ms_e2e, last = timed(step_e2e, args.steps, args.warmup + args.steps)
    if outputs is not None:
        outputs["latents_e2e"] = last.float()
    clk = clocks.finish()
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs, "" if world == 1 else f"_rank{rank}")
    # roofline leg: ONE more sample with a CUDA-event pair around every launch of this package's attention kernels (on the
    # launching stream). Kept out of the timed regions above: ~8 000 event records per sample cost ~3 % of the step.
    ops.TIMER = ops.KernelTimer()
    graphs_on, pipe.use_cuda_graphs = pipe.use_cuda_graphs, False  # every launch through Python, so every one gets its events
    step_resident(args.warmup)
    pipe.use_cuda_graphs = graphs_on
    ksum = ops.TIMER.summary()
    ops.TIMER = None

    frames = L * args.steps * world
    value = frames / (ms / 1e3)
    e2e = frames / (ms_e2e / 1e3)

    if rank != 0:
        return
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    tpeak = float(peaks.get("bf16_tflops_sustained", 1400.0))
    n_l, n_b, n_ms = ksum.get("temporal_attn_fwd", (0, 0, 0.0))
    achieved = (n_b / 1e9) / (n_ms / 1e3) if n_ms > 0 else None
    traffic = _ncu_traffic()
    roof = {"kernel": "temporal_attn_fwd_kernel", "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
            "frac": (achieved / peak) if achieved else None,
            "traffic": traffic["dram_bytes_per_launch"] if traffic else None,
            "traffic_source": traffic["source"] if traffic else "no committed ncu dram capture",
            "peak_source": "MEASURED_PEAKS.json (burst copy)" if peaks else "fallback 6.65 TB/s (B200_PROFILING.md)",
            "launches": n_l, "algorithmic_bytes_per_launch": (n_b / n_l) if n_l else None,
            "avg_launch_us": (1e3 * n_ms / n_l) if n_l else None,
            "l2_policy": "in situ: Q/K/V were just written by the QKV GEMM and can be L2-resident; "
                         "profiles/ holds the cold-L2 per-shape numbers"}
    b_l, b_b, b_ms = ksum.get("temporal_attn_bwd", (0, 0, 0.0))
    if b_ms > 0:
        roof["bwd"] = {"launches": b_l, "achieved": (b_b / 1e9) / (b_ms / 1e3), "frac": (b_b / 1e9) / (b_ms / 1e3) / peak}
    roof["measured_on"] = "one extra sample after the timed regions (event pairs around every launch)"
    # the other hand-written attention kernels, same accounting: HBM-bound cross-attention (bytes), tensor-bound spatial
    # self-attention (flops as launched against the sustained bf16 GEMM peak)
    roof["other_kernels"] = {
        k: {"launches": n_, "achieved": (b_ / 1e9) / (ms_ / 1e3), "frac": (b_ / 1e9) / (ms_ / 1e3) / peak, "unit": "GB/s",
            "avg_launch_us": 1e3 * ms_ / n_}
        for k, (n_, b_, ms_) in ksum.items() if k.startswith("cross_attn") and ms_ > 0}
    roof["other_kernels"].update({
        k: {"launches": n_, "bound": "tensor", "achieved": (f_ / 1e12) / (ms_ / 1e3), "peak": tpeak, "unit": "TFLOP/s",
            "frac": (f_ / 1e12) / (ms_ / 1e3) / tpeak, "avg_launch_us": 1e3 * ms_ / n_,
            "flops": "as launched (4 B N^2 C forward; 14 B N^2 C backward: S and dP are recomputed in both backward kernels)"}
        for k, (n_, f_, ms_) in ksum.items() if k.startswith("spatial_attn") and ms_ > 0})
    gpu_ref = None
    if not args.no_gpu_reference and world == 1 and not use_cn:
        try:
            tg, tp = gpu_reference_steps(infer, dev)
            gpu_ref = {"value": fps_from_step_times(tg, tp, infer), "unit": UNIT, "kind": "port",
                       "what": "reference op sequence (oracle port) in fp16 on the SAME GPU, torch SDPA at the xformers seam",
                       "s_per_guided_step": tg, "s_per_plain_step": tp,
                       "sample": f"1 warm-up + 2 timed guided and plain DDIM steps at {L}x{infer['height']}x{infer['width']}, "
                                 f"extrapolated to {infer['inference_steps']} steps ({infer['guidance_steps']} guided)",
                       "own_over_gpu_reference": value / fps_from_step_times(tg, tp, infer)}
        except Exception as e:  # an out-of-memory comparator must not lose the bench line
            gpu_ref = {"unavailable": f"{type(e).__name__}: {str(e)[:160]}"}
            torch.cuda.empty_cache()
    cpu = None
    if not args.no_cpu_baseline and world == 1:
        tg, tp, info = cpu_reference_steps(args.cpu_budget, infer)
        cpu = cpu_block(tg, tp, info, infer, fps_from_step_times(tg, tp, infer))
    lat_bytes = host[0].numel() * 2
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f16", "data": "synthetic",
            "config": config_block(infer, workload, world),
            "arm": f"replica x{world} (independent samples), one NCCL broadcast of the motion representation; "
                   f"cuda graphs {'on' if pipe.use_cuda_graphs else 'off'}",
            "init": {"nccl_init_ms": nccl_init_ms, "broadcast_ms": bcast_ms, "broadcast_bytes": int(rep_host.numel())},
            "e2e": {"value": e2e, "unit": UNIT,
                    "h2d_bytes_per_step": lat_bytes + text_host[0].numel() * 2 + rep_host.numel(),
                    "d2h_bytes_per_step": lat_bytes, "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": int(launches), "clocks": clk, "roofline": roof, "gpu_reference": gpu_ref, "cpu_baseline": cpu}
    _emit(line)


def dump_outputs(directory: str, outputs: dict, suffix: str = "") -> None:
    """What the timed sample_video calls returned in their last step, as float32 .npy files: `latents` from the
    device-resident loop behind the headline value, `latents_e2e` from the host-buffer loop. The inputs are seeded, so
    two builds run with the same arguments can be compared output for output."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    for name, t in outputs.items():
        np.save(os.path.join(directory, f"{name}{suffix}.npy"), t.to(torch.float32).numpy())
    log(f"[bench] outputs of the last timed step written to {directory}: {', '.join(outputs)}")


_RESULT_FD = None


def _emit(line: dict) -> None:
    data = (json.dumps(line) + "\n").encode()
    if _RESULT_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_RESULT_FD, data)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="object", choices=list(CONFIGS),
                    help="BASELINE.json configs[1..4]; `object` (configs[1]) is the headline the driver runs")
    ap.add_argument("--ddim-steps", type=int, default=50, help="profiling only: anything but 50 is not a bench value")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-reference", action="store_true")
    ap.add_argument("--no-cuda-graphs", action="store_true", help="A/B: launch the no-grad UNet forwards eagerly")
    ap.add_argument("--ref-budget", type=float, default=240.0, help="seconds of CPU work for --impl reference")
    ap.add_argument("--cpu-budget", type=float, default=60.0, help="seconds of CPU work for the cpu_baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the final latents of the last timed step as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours: the reference arm extrapolates from partial steps")
    # The contract is ONE JSON line on stdout. Libraries write there too (NCCL prints its version banner on the first
    # communicator when NCCL_DEBUG=VERSION is set in the environment), so everything but the result goes to stderr: file
    # descriptor 1 is pointed at stderr for the run and the line is written to the saved descriptor at the end.
    global _RESULT_FD
    sys.stdout.flush()
    _RESULT_FD = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_own_arm(args)
    if torch.distributed.is_available() and torch.distributed.is_initialized():
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
