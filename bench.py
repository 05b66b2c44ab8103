#!/usr/bin/env python
"""bench.py — MVOC composition hot path on B200: video frames/s of the 50-step DDIM composition.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl mvoc|reference] [--workload config2]
                    [--dump-outputs DIR]

One "step" = one DDIM composition step (latent fusion + concat, one UNet forward over
[bg, obj_1..obj_n, uncond, cond], CFG + DDIM update) of BASELINE.json configs[1]:
full i2vgen-xl-architecture UNet (random init), 16 frames x 64x64 latents (512x512 px), bg + 2 objects,
boat_surf injection schedule.  The timed region starts at step 0 of the schedule (fusion step, conv
injection on the first 10 % of the steps) and runs K steps; with K = 50 (default) it is the whole run, and a
larger K starts the schedule again from the initial latents.
value = n_frames / (50 * mean step time).

--dump-outputs DIR writes the latents of the timed region's last step as DIR/latents.npy (float32; the inversion
workloads write DIR/latents_video<v>.npy per video); the inputs are seeded, so two builds run with the same
arguments can be compared output for output.

Prints ONE JSON line (see README / DESIGN.md §Measurement for every key).
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

METRIC = "video frames/s, 50-step 16x512^2 bg+2obj composite"
UNIT = "frames/s"
PARITY_BAR = 5e-3      # multi-rank latents vs the single-GPU run after the first steps (relative L2)


def ncu_traffic_per_launch():
    """dram__bytes_read.sum + dram__bytes_write.sum of the l0 attention kernel from the newest committed ncu summary
    (profiles/*ncu_attn_l0*summary.txt); (None, reason) when there is none.  Never a literal."""
    import glob
    import re

    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "*ncu_attn_l0*summary.txt")))
    for path in reversed(files):
        rd = wr = None
        with open(path) as f:
            for ln in f:
                m = re.match(r"\s*dram__bytes_(read|write)\.sum\s+([0-9.]+)\s*(\w+)", ln)
                if m:
                    val = float(m.group(2)) * {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}.get(m.group(3), 1.0)
                    if m.group(1) == "read":
                        rd = val
                    else:
                        wr = val
        if rd is not None and wr is not None:
            return rd + wr, "ncu --set full dram__bytes_read+write per launch, " + os.path.relpath(path, ROOT)
    return None, "no ncu summary under profiles/"


# --------------------------------------------------------------------------- helpers
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._pump, daemon=True)
        self.thread.start()

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
                power.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(names, f[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {
            "sm_mhz": statistics.median(sm) if sm else None,
            "sm_max_mhz": max(mx) if mx else None,
            "power_w_max": max(power) if power else None,
            "samples": len(sm),
            "reasons": sorted(reasons),
        }


def measured_peaks() -> dict:
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        d["_source"] = "measured"
        return d
    # fallback stated in /opt/skills/guides/B200_PROFILING.md
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "_source": "fallback"}


def metric_name(wl) -> str:
    """BASELINE.json's metric for config 2; the same quantity named after the workload for the other configs."""
    if wl.name == "config2":
        return METRIC
    px = f"{wl.n_frames}x{wl.latent_h * 8}x{wl.latent_w * 8}"
    if wl.n_obj == 0:
        return f"video frames/s, {wl.inversion_steps}-step DDIM inversion of {wl.n_videos} x {px} source videos"
    return f"video frames/s, {wl.n_steps}-step {px} bg+{wl.n_obj}obj composite"


def workload_description(wl) -> str:
    if wl.n_obj == 0:
        return (f"{wl.name}: full i2vgen-xl UNet random-init, DDIM inversion ({wl.inversion_steps} steps, cfg 1.0, batch 1) "
                f"of {wl.n_videos} independent source videos of {wl.n_frames} frames x {wl.latent_h}x{wl.latent_w} latents")
    return (f"{wl.name}: full i2vgen-xl UNet random-init, {wl.n_frames} frames x {wl.latent_h}x{wl.latent_w} "
            f"latents, bg+{wl.n_obj} objects, {wl.n_steps}-step DDIM composition, cfg {wl.cfg}, pnp_f_t {wl.pnp_f_t}, "
            f"spatial/temporal attn injection {wl.pnp_spatial_attn_t}/{wl.pnp_temp_attn_t}")


def schedule_passes(steps: int, schedule_len: int) -> list:
    """Step counts of the passes over a schedule of `schedule_len` steps that make `steps` steps in all.  A count
    past the end of the schedule starts it again from the initial latents, so --steps is the number of steps timed
    whatever the length of the schedule."""
    full, rest = divmod(steps, schedule_len)
    return [schedule_len] * full + ([rest] if rest else [])


DUMP_LIMIT_BYTES = 64 * 2 ** 20


def _dump_dtype(t):
    import torch

    return torch.float64 if t.dtype == torch.float64 else torch.float32


def check_dump_size(arrays: dict) -> None:
    """Refuses outputs of more than DUMP_LIMIT_BYTES.  The benchmark also calls it before the warm-up, with tensors
    of the outputs' shapes and dtypes (the initial latents), so that an oversized dump fails before any step runs."""
    total = sum(t.numel() * _dump_dtype(t).itemsize for t in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes of outputs exceed the {DUMP_LIMIT_BYTES}-byte limit")


def dump_outputs(outdir: str, arrays: dict) -> None:
    """--dump-outputs: every tensor as <outdir>/<name>.npy, float64 kept and any other dtype as float32, so that
    two builds of the project can be compared output for output on the same seeded inputs."""
    import numpy as np

    check_dump_size(arrays)
    os.makedirs(outdir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(outdir, name + ".npy"), t.detach().to("cpu", _dump_dtype(t)).numpy())


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


# --------------------------------------------------------------------------- CPU arm (oracle port)
class CpuSampler:
    """Times the fp32 oracle (the reference path restated, oracle/pipeline.py) on the host cores for ONE
    composition step of a bounded sample of the workload: the full UNet and all n_obj+3 branches, but 2 of
    the n_frames frames at a latent size chosen from a GEMM calibration so that a step fits `budget_s`.
    step() -> (frames_per_s_equivalent, seconds)."""

    def __init__(self, wl_name: str, budget_s: float):
        import torch

        from mvoc_b200 import synthetic
        from oracle import pipeline as opipe
        from oracle.scheduler import DDIMScheduler

        self.cores = os.cpu_count() or 1
        torch.set_num_threads(self.cores)
        full = synthetic.WORKLOADS[wl_name]
        a = torch.randn(2048, 2048)
        b = torch.randn(2048, 2048)
        a @ b
        t0 = time.perf_counter()
        for _ in range(3):
            a @ b
        gemm_tfs = 3 * 2 * 2048 ** 3 / (time.perf_counter() - t0) / 1e12
        # ~104 TFLOP per full step at 16 x 64x64 x 5 branches (SURVEY App. C) => per (frame, latent pixel)
        flop_per_frame_pixel = 104.1e12 / (16 * 64 * 64)
        eff = 0.5 * gemm_tfs * 1e12  # convs / attention run below the GEMM rate
        frames, side = 2, 16
        for s in (64, 32, 16):
            if flop_per_frame_pixel * frames * s * s / eff <= budget_s:
                side = s
                break
        self.full = full
        self.wl = synthetic.Workload(
            f"{wl_name}-cpu-sample", full.unet, frames, side, side, full.n_obj, n_steps=full.n_steps, cfg=full.cfg,
            pnp_f_t=full.pnp_f_t, pnp_spatial_attn_t=full.pnp_spatial_attn_t, pnp_temp_attn_t=full.pnp_temp_attn_t,
            fusion_step=full.fusion_step, random_noise_ratio=full.random_noise_ratio)
        sched = DDIMScheduler()
        sched.set_timesteps(self.wl.n_steps)
        self.inputs = synthetic.make_inputs(self.wl, [int(t) for t in sched.timesteps], sched.alphas_cumprod)
        self.unet = opipe.build_unet(self.wl.unet, seed=0)
        self._loop = opipe.composite_loop
        # frames of the 64x64 x 16-frame job per sample step if the per-(frame, latent pixel) cost stayed what it
        # is in the sample (optimistic for the CPU: spatial attention grows quadratically with the latent area)
        self.frame_equiv = frames * (side * side) / float(full.latent_h * full.latent_w)
        self.desc = (f"oracle fp32 (oracle/pipeline.py), 1 composition step, full UNet, {self.wl.n_branches} "
                     f"branches, {frames} of {full.n_frames} frames at {side}x{side} of "
                     f"{full.latent_h}x{full.latent_w} latents; scaled per (frame x latent pixel) and "
                     f"x{full.n_steps} steps (extrapolated, not a full run); host fp32 GEMM {gemm_tfs:.2f} TF/s")

    def step(self):
        t0 = time.perf_counter()
        self._loop(self.unet, self.wl, self.inputs, max_steps=1)
        dt = time.perf_counter() - t0
        return self.frame_equiv / (self.full.n_steps * dt), dt


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path (the oracle port: diffusers and the
    checkpoint are unavailable offline, see DESIGN.md) on all host threads; rank 0 only."""
    rank, world, _ = dist_env()
    if rank != 0:
        return
    n = args.steps + args.warmup
    budget = max(1.0, min(20.0, 150.0 / max(1, n)))
    sampler = CpuSampler(args.workload, budget)
    vals, t_start = [], time.perf_counter()
    for i in range(n):
        fps, dt = sampler.step()
        if i >= args.warmup:
            vals.append((fps, dt))
        if time.perf_counter() - t_start > 240 and vals:  # hard bound on the whole arm
            break
    last = (sampler.cores, sampler.desc)
    fps = statistics.mean(v for v, _ in vals)
    ms = statistics.mean(d for _, d in vals) * 1e3
    line = {
        "impl": "reference", "metric": METRIC, "value": fps, "unit": UNIT, "n_gpus": args.gpus,
        "steps": len(vals), "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_description(sampler.full), "parallelism": f"{last[0]} host threads",
                   "sample_per_step": last[1]},
        "cpu_baseline": {"value": fps, "unit": UNIT, "cores": last[0], "kind": "port", "sample": last[1],
                         "same_config": False,
                         "note": "bounded sample: ms_per_step is the time of the SAMPLE step (2 of the frames), value is "
                                 "scaled to the full workload linearly in frames (spatial attention is per frame, so "
                                 "the latent size of the sample is what matters and it is the full one when it fits)"},
        "e2e": {"value": fps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


# --------------------------------------------------------------------------- GPU arm
def run_mvoc(args):
    import torch

    rank, world, local = dist_env()
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("--gpus N>1 must be launched with torch.distributed.run (one rank per GPU)")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (sm_100a); there is no CPU fallback for the product path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)

    from mvoc_b200 import _cabi, ops, synthetic
    from mvoc_b200.parallel import FrameParallel
    from mvoc_b200.pipeline import Conditioning, I2VGenXLPipeline, LatentBank, init_pnp
    from mvoc_b200.scheduler import DDIMSchedule
    from mvoc_b200.unet3d import build_unet

    lib = _cabi.load()
    _cabi.check(lib.mvoc_device_check(local), "mvoc_device_check")
    wl0 = synthetic.WORKLOADS[args.workload]
    if wl0.n_obj == 0:
        os.environ["MVOC_EXCHANGE"] = "nccl"      # replicas exchange nothing: no peer arena
    elif world > 1 and "MVOC_EXCHANGE_ARENA_MB" not in os.environ:
        # every temporal operator of a forward bump-allocates two buffers of (tensor / P) bytes: ~60 l0-sized ones
        l0 = wl0.n_branches * wl0.n_frames * wl0.latent_h * wl0.latent_w * 320 * 2
        os.environ["MVOC_EXCHANGE_ARENA_MB"] = str(int(min(32768, max(4096, 60 * l0 / world / 2 ** 20))))
    par = FrameParallel.from_env(dev)  # world_size 1 => no-op

    wl = synthetic.WORKLOADS[args.workload]
    if wl.n_obj == 0:
        return run_inversion(args, wl, par, dev, rank, world, local)
    sched = DDIMSchedule(wl.n_steps)
    inputs = synthetic.make_inputs(wl, sched.timesteps, sched.alphas_cumprod)
    if args.dump_outputs:
        check_dump_size({"latents": inputs["init_latents"]})
    torch.backends.cudnn.benchmark = True
    unet = build_unet(wl.unet, seed=0, device=dev)
    pipe = I2VGenXLPipeline(unet, dev, parallel=par, use_cuda_graphs=not args.no_graphs)
    init_pnp(pipe, sched, wl)
    bf = lambda x: x.to(device=dev, dtype=torch.bfloat16)
    cond = Conditioning(bf(inputs["prompt_embeds"]), bf(inputs["image_embeddings"]),
                        bf(inputs["image_latents_first"]), bf(inputs["image_latents"]), inputs["fps"].to(dev))
    banks = [LatentBank(src, dev, pin_host=True) for src in inputs["source_latents"]]
    masks = [(mf.to(dev), mb.to(dev)) for mf, mb in inputs["masks"]]

    def loop(start, steps, host_io=False, lat=None):
        lat = inputs["init_latents"].to(dev).clone() if lat is None else lat
        return pipe.sample_with_pnp_pipeline_with_edit_prompt_extraction_with_attn_injection(
            cond, lat, banks[0], banks[1:], masks, num_inference_steps=wl.n_steps, guidance_scale=wl.cfg,
            ddim_init_latents_t_idx=wl.ddim_init_latents_t_idx, fusion_steps=tuple(wl.fusion_step),
            random_noise_ratio=wl.random_noise_ratio, obj_random_noise_fusion=wl.obj_random_noise_fusion,
            start_step=start, max_steps=steps, host_io=host_io)

    def run(steps, host_io=False):
        lat = None
        for n in schedule_passes(steps, wl.n_steps - wl.ddim_init_latents_t_idx):
            lat = loop(0, n, host_io)
        return lat

    K, W = args.steps, max(args.warmup, 0)
    # warm-up: W steps from the start of the schedule, plus one step of every other hook configuration that
    # occurs in the timed range, so that cuDNN autotuning and CUDA-graph capture happen outside the timing
    if W > 0:
        run(W)
    for i in pipe.step_kinds(sched.timesteps[:K], masks):
        if i >= W:
            loop(i, 1)
    torch.cuda.synchronize()

    def barrier():
        par.barrier()
        torch.cuda.synchronize()

    # ---- timed region 1: inputs resident in HBM ------------------------------------------------
    clocks = ClockSampler(local)
    barrier()
    if rank == 0:
        clocks.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.nvtx.range_push("mvoc_timed_region")   # `ncu --nvtx --nvtx-include "mvoc_timed_region/"`
    ev0.record()
    final = run(K)
    ev1.record()
    barrier()
    torch.cuda.nvtx.range_pop()
    clk = clocks.stop() if rank == 0 else None
    ms_total = par.max_over_ranks(ev0.elapsed_time(ev1))
    ms_step = ms_total / K

    # ---- timed region 2: end to end through the pipeline API with host buffers ------------------
    loop(0, 1, host_io=True)      # untimed: first-use pinned allocations of the host path
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_wall0 = time.perf_counter()
    e0.record()
    final_e2e = run(K, host_io=True)
    e1.record()
    barrier()
    wall_ms = (time.perf_counter() - t_wall0) * 1e3
    e2e_ms_step = par.max_over_ranks(max(e0.elapsed_time(e1), wall_ms)) / K
    E = inputs["init_latents"].numel()
    h2d = (1 + wl.n_obj) * E * 4
    d2h = E * 4
    same = bool(torch.equal(final, final_e2e))

    # ---- per-kernel pass: the same K steps launched eagerly with CUDA events around every C-ABI launch
    # (events cannot be recorded per kernel inside a captured graph; kernel durations are the same) -------
    graphs_on = pipe.use_cuda_graphs
    pipe.use_cuda_graphs = False
    timer = ops.KernelTimer()
    barrier()
    launches0 = ops.launch_count
    ops.set_timer(timer)
    k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    k0.record()
    run(K)
    k1.record()
    barrier()
    ops.set_timer(None)
    pipe.use_cuda_graphs = graphs_on
    launches = ops.launch_count - launches0
    ms_eager_total = k0.elapsed_time(k1)

    # ---- multi-rank parity (every N > 1 line carries it): the first steps of the sharded run against the same
    # steps on ONE GPU (rank 0, no partition).  Only the merge order of the GroupNorm statistics differs.
    parity = None
    if world > 1:
        n_par = min(2, K)
        barrier()
        lat_multi = loop(0, n_par).clone()
        barrier()
        if rank == 0:
            solo = I2VGenXLPipeline(unet, dev, parallel=FrameParallel.single(dev), use_cuda_graphs=False)
            solo.scheduler = pipe.scheduler
            unet.ctx.parallel = None
            lat_solo = inputs["init_latents"].to(dev).clone()
            solo.sample_with_pnp_pipeline_with_edit_prompt_extraction_with_attn_injection(
                cond, lat_solo, banks[0], banks[1:], masks, num_inference_steps=wl.n_steps, guidance_scale=wl.cfg,
                ddim_init_latents_t_idx=wl.ddim_init_latents_t_idx, fusion_steps=tuple(wl.fusion_step),
                random_noise_ratio=wl.random_noise_ratio, obj_random_noise_fusion=wl.obj_random_noise_fusion,
                max_steps=n_par)
            torch.cuda.synchronize()
            rel = float((lat_multi - lat_solo).norm() / lat_solo.norm())
            parity = {"rel_l2_vs_n1": rel, "steps": n_par, "bar": PARITY_BAR, "ok": bool(rel <= PARITY_BAR)}
        barrier()

    if rank != 0:
        _finish(pipe, par)
        return
    peaks = measured_peaks()
    frames_per_s = wl.n_frames / (wl.n_steps * ms_step / 1e3)
    e2e_fps = wl.n_frames / (wl.n_steps * e2e_ms_step / 1e3)

    # ---- roofline of the dominant kernel: l0 spatial self-attention (tcgen05) --------------------
    summ = timer.summary()
    # spatial / cross attention calls: plain ("attn", B, H, Nq, Nk) and injected ("attn_inject", B, H, Nq, Nk, share_p);
    # both carry the REFERENCE's FLOPs (every branch its own softmax), whatever the kernels share
    attn_keys = [k for k in summ if k[0] in ("attn", "attn_inject")]
    attn_ms = sum(summ[k][1] for k in attn_keys)
    attn_flops = sum(summ[k][2] for k in attn_keys)
    tattn_keys = [k for k in summ if k[0] == "attn_temporal"]
    shape = lambda k: tuple(k[1:5])
    by_shape = {}
    for k in attn_keys:
        by_shape.setdefault(shape(k), []).append(k)
    # the dominant shape by algorithmic work, not by measured time: in an eager replay on many GPUs the host cannot
    # keep up with the small low-resolution launches and their event brackets include host gaps
    dom_shape = max(by_shape, key=lambda sh: sum(summ[k][2] for k in by_shape[sh])) if by_shape else None
    roof = None
    if dom_shape is not None:
        ks = by_shape[dom_shape]
        n = sum(summ[k][0] for k in ks)
        ms = sum(summ[k][1] for k in ks)
        work = sum(summ[k][2] for k in ks)
        achieved = work / (ms / 1e3) / 1e12
        peak = peaks["bf16_tflops_sustained"]
        plain = [k for k in ks if k[0] == "attn"]
        inj = [k for k in ks if k[0] == "attn_inject"]
        tfs = lambda kk: (sum(summ[k][2] for k in kk) / (sum(summ[k][1] for k in kk) / 1e3) / 1e12) if kk else None
        traffic, traffic_src = ncu_traffic_per_launch()
        roof = {
            "bound": "tensor",
            "kernel": (f"attn_fwd_kernel: the spatial self-attention layers B={dom_shape[0]} H={dom_shape[1]} "
                       f"Nq={dom_shape[2]} Nk={dom_shape[3]} D=64 (plain layers: one launch; injected layers: "
                       "mvoc_attn_inject_fwd = blend + source branches + one-softmax pair kernel for uncond/cond)"),
            "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
            "flops": "reference count 4*B*H*Nq*Nk*D per layer for all layers (SURVEY 8d: no discount for shared P)",
            "peak_source": peaks["_source"] + " (sustained cuBLAS bf16: kernel timed inside a long step)",
            "launches": n, "avg_launch_ms": ms / n, "share_of_step": ms / ms_total,
            "plain_layers": {"calls": sum(summ[k][0] for k in plain), "tflops": tfs(plain),
                             "frac": (tfs(plain) / peak) if plain else None},
            "injected_layers": {"calls": sum(summ[k][0] for k in inj), "tflops": tfs(inj),
                                "frac": (tfs(inj) / peak) if inj else None},
            "timing": "CUDA events around each C-ABI call while the same K steps are replayed eagerly "
                      "(per-kernel events cannot live inside the captured graphs of the timed region)",
            "traffic": traffic if dom_shape == (80, 5, 4096, 4096) else None,
            "traffic_source": traffic_src if dom_shape == (80, 5, 4096, 4096) else
            "no ncu capture at this shard shape (the committed captures are of the N=1 config-2 shape)",
        }
    gn_keys = [k for k in summ if k[0] == "groupnorm"]
    ex_keys = [k for k in summ if k[0] == "exchange"]
    gemm_keys = [k for k in summ if k[0] == "gemm"]
    gemm_ms = sum(summ[k][1] for k in gemm_keys)
    extra = {
        "gemm_tflops_all": (sum(summ[k][2] for k in gemm_keys) / (gemm_ms / 1e3) / 1e12) if gemm_ms else None,
        "gemm_share_of_step": gemm_ms / ms_total if gemm_keys else None,
        "conv3x3_tflops": (lambda ks: (sum(summ[k][2] for k in ks) / (sum(summ[k][1] for k in ks) / 1e3) / 1e12)
                           if ks else None)([k for k in gemm_keys if k[1] == "conv3x3"]),
        "attn_tflops_all": (attn_flops / (attn_ms / 1e3) / 1e12) if attn_ms else None,
        "attn_share_of_step": attn_ms / ms_total if ms_total else None,
        "temporal_attn_gbs": (sum(summ[k][2] for k in tattn_keys) / (sum(summ[k][1] for k in tattn_keys) / 1e3) / 1e9)
        if tattn_keys else None,
        "groupnorm_gbs": (sum(summ[k][2] for k in gn_keys) / (sum(summ[k][1] for k in gn_keys) / 1e3) / 1e9)
        if gn_keys else None,
        "groupnorm_share_of_step": sum(summ[k][1] for k in gn_keys) / ms_total if gn_keys else None,
        # frame-shard <-> pixel-shard exchange (put kernel + wait) of this rank, per step, in the eager replay
        "exchange_ms_per_step": (sum(summ[k][1] for k in ex_keys) / K) if ex_keys else None,
        "exchange_calls_per_step": (sum(summ[k][0] for k in ex_keys) / K) if ex_keys else None,
    }

    # the kernel the step spends most of its time in since round 2: the tcgen05 GEMM family (same roofline fields)
    roof_dense = None
    if gemm_keys and gemm_ms > 0:
        g_ach = sum(summ[k][2] for k in gemm_keys) / (gemm_ms / 1e3) / 1e12
        roof_dense = {
            "bound": "tensor", "kernel": "gemm_tc_kernel: every 3x3 conv, temporal conv, Linear and GEGLU projection of the step "
                                         "(short-K Linears included, which are epilogue / HBM bound)",
            "achieved": g_ach, "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
            "frac": g_ach / peaks["bf16_tflops_sustained"], "flops": "2*rows*N*K_total per launch",
            "launches": sum(summ[k][0] for k in gemm_keys), "share_of_step": gemm_ms / ms_total,
            "conv3x3_only": {"achieved": extra["conv3x3_tflops"],
                             "frac": (extra["conv3x3_tflops"] / peaks["bf16_tflops_sustained"])
                             if extra["conv3x3_tflops"] else None},
            "traffic": None, "traffic_source": "per-shape ncu captures: profiles/r02_final_ncu_*_summary.txt (DRAM bytes = algorithmic)",
        }

    # where the (eager-replayed) step goes: the twelve heaviest timer keys, work in TFLOP/s or GB/s by kernel family
    tops = sorted(summ.items(), key=lambda kv: -kv[1][1])[:12]
    extra["top"] = [{"key": "/".join(str(x) for x in k), "calls_per_step": n / K, "ms_per_step": ms / K,
                     "rate": (w / (ms / 1e3) / (1e12 if k[0] in ("gemm", "attn", "attn_inject", "attn_pair") else 1e9))
                     if ms else None,
                     "rate_unit": "TFLOP/s" if k[0] in ("gemm", "attn", "attn_inject", "attn_pair") else "GB/s"}
                    for k, (n, ms, w) in tops]

    # ---- CPU baseline beside it (rank 0, N = 1 only) ---------------------------------------------
    cpu = None
    if args.gpus == 1 and not args.no_cpu_baseline:
        try:
            sampler = CpuSampler(args.workload, budget_s=20.0)
            fps, dt = sampler.step()
            cpu = {"value": fps, "unit": UNIT, "cores": sampler.cores, "kind": "port", "sample": sampler.desc,
                   "seconds": dt, "same_config": False}
        except Exception as ex:  # the GPU numbers must still be reported
            cpu = {"value": None, "unit": UNIT, "cores": os.cpu_count(), "kind": "port", "sample": f"failed: {ex}"}

    line = {
        "metric": metric_name(wl), "value": frames_per_s, "unit": UNIT, "n_gpus": args.gpus, "steps": K, "warmup": W,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic",
        "config": {
            "workload": workload_description(wl),
            "parallelism": par.describe(),
            "l2": "activations per step (>= 210 MB per l0 tensor) exceed the 126 MB L2; no explicit flush",
            "timed_steps_start_at": 0,
            "cuda_graphs": bool(pipe.use_cuda_graphs),
            "eager_ms_per_step": ms_eager_total / K,
            # experiment switches (all off for the product numbers; a line with any of them set is an A/B line)
            "switches": {k: os.environ[k] for k in ("MVOC_DENSE", "MVOC_GEMM_VARIANT", "MVOC_EXCHANGE", "MVOC_EXCHANGE_WAIT",
                                                              "MVOC_FP_GATHER_MAX_PIXELS")
                         if os.environ.get(k)},
        },
        "roofline": roof,
        "roofline_dense": roof_dense,
        "cpu_baseline": cpu,
        "e2e": {"value": e2e_fps, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": e2e_ms_step, "matches_device_resident_run": same},
        "gpu_launches": launches,
        "clocks": clk,
        "kernels": extra,
    }
    if parity is not None:
        line["parity"] = parity
    print(json.dumps(line))
    sys.stdout.flush()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"latents": final})   # every rank holds all frames of the latents
    _finish(pipe, par)
    if parity is not None and not parity["ok"]:
        raise SystemExit(f"multi-rank parity failed: rel L2 {parity['rel_l2_vs_n1']:.3e} > {PARITY_BAR}")


def run_inversion(args, wl, par, dev, rank, world, local):
    """BASELINE config 3: group DDIM inversion (pipelines/pipeline_i2vgen_xl.py:1940-2000) of wl.n_videos independent
    source videos, video v on rank v % N — replicas, no data-path collective (inverse.py processes the entries of
    group_config.json one after the other).  One step = one inversion step of EVERY video of the group;
    value = n_videos * n_frames / (inversion_steps * step time)."""
    import torch

    from mvoc_b200 import ops, synthetic
    from mvoc_b200.parallel import FrameParallel
    from mvoc_b200.pipeline import Conditioning, I2VGenXLPipeline
    from mvoc_b200.unet3d import build_unet

    torch.backends.cudnn.benchmark = True
    unet = build_unet(wl.unet, seed=0, device=dev)
    pipe = I2VGenXLPipeline(unet, dev, parallel=FrameParallel.single(dev), use_cuda_graphs=not args.no_graphs)
    mine = [v for v in range(wl.n_videos) if v % world == rank]
    bf = lambda x: x.to(device=dev, dtype=torch.bfloat16)
    vids = []
    for v in mine:
        inv = synthetic.make_inversion_inputs(wl, v)
        pe, ie, il, fps = bf(inv["prompt_embeds"]), bf(inv["image_embeddings"]), bf(inv["image_latents"]), inv["fps"].to(dev)
        vids.append((inv["latents"].to(dev), pe, ie, il, fps, Conditioning(pe, ie, il, il, fps)))
    if args.dump_outputs:
        check_dump_size({f"latents_video{v}": vid[0] for v, vid in zip(mine, vids)})
    K, W = args.steps, max(args.warmup, 0)

    pinned = [torch.empty(v[0].shape, dtype=v[0].dtype).pin_memory() for v in vids]   # once, outside the timing

    def steps(n, host_io=False):
        outs = []
        for (lat, pe, ie, il, fps, cond), host in zip(vids, pinned):
            for m in schedule_passes(n, wl.inversion_steps):
                x = host.copy_(lat.cpu()).to(dev, non_blocking=True) if host_io else lat.clone()
                pipe.invert(x, pe, ie, il, fps, num_inference_steps=wl.inversion_steps, max_steps=m, keep=False,
                            cond=cond, on_step=(lambda t, z: host.copy_(z, non_blocking=False)) if host_io else None)
            outs.append(x)
        return outs

    if W > 0:
        steps(W)
    torch.cuda.synchronize()

    def barrier():
        par_all.barrier()
        torch.cuda.synchronize()

    par_all = par
    clocks = ClockSampler(local)
    barrier()
    if rank == 0:
        clocks.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    outs = steps(K)
    ev1.record()
    barrier()
    clk = clocks.stop() if rank == 0 else None
    # launches of this library per timed region: counted on ONE eager step per video (graph replays do not pass
    # through the Python wrappers), times the K steps
    graphs_on, pipe.use_cuda_graphs = pipe.use_cuda_graphs, False
    l0 = ops.launch_count
    steps(1)
    launches = (ops.launch_count - l0) * K
    pipe.use_cuda_graphs = graphs_on
    ms_step = par_all.max_over_ranks(ev0.elapsed_time(ev1)) / K
    barrier()
    t0 = time.perf_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    steps(K, host_io=True)
    e1.record()
    barrier()
    e2e_ms = par_all.max_over_ranks(max(e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3)) / K
    if rank == 0:
        E = 4 * wl.n_frames * wl.latent_h * wl.latent_w
        fps_val = wl.n_videos * wl.n_frames / (wl.inversion_steps * ms_step / 1e3)
        line = {
            "metric": metric_name(wl), "value": fps_val, "unit": UNIT, "n_gpus": args.gpus, "steps": K, "warmup": W,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic",
            "config": {"workload": workload_description(wl),
                       "parallelism": f"replicas: video v on rank v % {world} (no data-path collective)",
                       "l2": "activations per step exceed the 126 MB L2; no explicit flush",
                       "cuda_graphs": bool(pipe.use_cuda_graphs)},
            "roofline": None, "cpu_baseline": None,
            "e2e": {"value": wl.n_videos * wl.n_frames / (wl.inversion_steps * e2e_ms / 1e3), "unit": UNIT,
                    "h2d_bytes_per_step": 0, "d2h_bytes_per_step": len(mine) * E * 4, "ms_per_step": e2e_ms},
            "gpu_launches": launches, "clocks": clk,
        }
        print(json.dumps(line))
        sys.stdout.flush()
    if args.dump_outputs:      # every rank writes the videos it inverted
        dump_outputs(args.dump_outputs, {f"latents_video{v}": x for v, x in zip(mine, outs)})
    _finish(pipe, par)


def _finish(pipe, par):
    """Orderly teardown: captured CUDA graphs (they hold collective / exchange kernels) go first, then the peer
    arenas and the process group.  A watchdog turns a teardown that blocks (round 1 saw NCCL do that at interpreter
    exit) into a plain exit — the results are already printed."""
    import gc

    import torch

    sys.stdout.flush()
    sys.stderr.flush()
    if par.world > 1:
        dog = threading.Timer(45.0, lambda: os._exit(0))
        dog.daemon = True
        dog.start()
    pipe.drop_graphs()
    gc.collect()
    torch.cuda.synchronize()
    if par.world > 1:
        par.barrier()
        par.shutdown()


def positive_int(text: str) -> int:
    v = int(text)
    if v < 1:
        raise argparse.ArgumentTypeError(f"must be at least 1, not {v}")
    return v


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=positive_int, default=50,
                    help="timed steps; past the end of the schedule it starts again from the initial latents")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="mvoc", choices=["mvoc", "reference"])
    ap.add_argument("--workload", default="config2")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graphs", action="store_true", help="launch every kernel from Python instead of replaying CUDA graphs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the latents they computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs writes what the CUDA path computes; --impl reference times a reduced CPU sample")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_mvoc(args)


if __name__ == "__main__":
    main()
