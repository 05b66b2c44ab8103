"""Reconstruction sampling on one B200: ms per guided step of the plain I2VGenXL loop (I2VGenXLPipeline.sample, UNet at
batch 2 + mvoc_cfg_ddim_step, CUDA graphs on), the VAE decode of its result, and the launch list of one step.

    python tools/recon_bench.py [--steps 12] [--out profiles/r07_recon_bench.jsonl]

Two geometries, those of BASELINE configs 2 and 5: 16 frames of 64x64 latents and 32 frames of 88x160.  Full-width
random-init UNet and decoder (seeded), seeded conditioning.  Prints one JSON line per geometry: the median and spread of
the per-step time over the replayed steps (the first step of a run computes the conditioning caches and captures the
graph and is reported apart), the decode time, and the kernels of one step (eager, under torch.profiler) grouped as
library kernels (namespace mvoc::), cuDNN / cuBLAS kernels (conv_in, conv_out, the stride-2 downsamplers, the
embedding MLPs) and any other torch kernel by name, with each group's device time and share of the step's kernel time
(kernel durations summed; in the eager run, so launch gaps are not counted).  The GPU's name, power limit and SM
clock are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import re
import statistics
import sys
from collections import Counter

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

from tools.vae_decode_bench import gpu_info  # noqa: E402

WORKLOADS = {"config2": (16, 64, 64), "config5": (32, 88, 160)}   # frames, latent h, latent w
VENDOR = re.compile(r"cutlass|cudnn|nvjet|gemm|sm\d+_xmma|conv|nhwc|Kernel2d", re.I)


def build(device):
    from mvoc_b200.unet3d import I2VGenXLUNet, UNetConfig, prepare
    from mvoc_b200.vae import AutoencoderKLDecoder

    torch.manual_seed(0)
    unet = prepare(I2VGenXLUNet(UNetConfig.full()).eval().requires_grad_(False).to(device, torch.bfloat16))
    torch.manual_seed(1)
    vae = prepare(AutoencoderKLDecoder().eval().requires_grad_(False).to(device, torch.bfloat16))
    return unet, vae


def inputs(T, h, w, device):
    from mvoc_b200 import synthetic

    src = synthetic.make_inversion_inputs(synthetic.Workload("recon", "full", T, h, w, 0))
    bf = lambda x: x.to(device, torch.bfloat16)  # noqa: E731
    return (bf(src["prompt_embeds"]), bf(src["negative_prompt_embeds"]), bf(src["image_embeddings"]),
            bf(src["image_latents"]), src["fps"].to(device))


def step_times(pipe, cond, steps, device):
    """Per-step ms of one `sample` run of `steps` guided steps: events recorded in the step callback."""
    ev = [torch.cuda.Event(enable_timing=True)]
    ev[0].record()

    def mark(i, t, lat):
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        ev.append(e)

    g = torch.Generator(device=device).manual_seed(4)
    out = pipe.sample(*cond, num_inference_steps=50, guidance_scale=9.0, generator=g, max_steps=steps, callback=mark)
    torch.cuda.synchronize()
    return [ev[i].elapsed_time(ev[i + 1]) for i in range(len(ev) - 1)], out


def launch_list(unet, cond, device):
    """Kernels of the second step of an eager 3-step run (the first computes the conditioning caches), with their
    device time.  The whole run is profiled and the step is cut out at the DDIM update kernels that end steps 1 and 2,
    so no launch at the window's edge is lost."""
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile

    from mvoc_b200.pipeline import I2VGenXLPipeline

    pipe = I2VGenXLPipeline(unet, device, use_cuda_graphs=False)
    g = torch.Generator(device=device).manual_seed(4)
    pipe.sample(*cond, num_inference_steps=50, guidance_scale=9.0, generator=g, max_steps=2)     # warm-up
    torch.cuda.synchronize()
    g = torch.Generator(device=device).manual_seed(4)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        pipe.sample(*cond, num_inference_steps=50, guidance_scale=9.0, generator=g, max_steps=3)
        torch.cuda.synchronize()
    ev = sorted((e for e in prof.events() if e.device_type == DeviceType.CUDA), key=lambda e: e.time_range.start)
    ends = [i for i, e in enumerate(ev) if "ddim_step_kernel" in e.name]
    assert len(ends) == 3, f"expected 3 DDIM updates in the profile, found {len(ends)}"
    step = ev[ends[0] + 1:ends[1] + 1]
    groups = {"library": Counter(), "cudnn_cublas": Counter(), "other_torch": Counter()}
    us = {k: Counter() for k in groups}
    for e in step:
        n = e.name
        if "mvoc::" in n:
            kind, key = "library", re.sub(r"^void |\(.*$", "", n)[:80]
        elif VENDOR.search(n) and "elementwise" not in n:
            kind, key = "cudnn_cublas", n[:80]
        else:
            kind, key = "other_torch", n[:100]
        groups[kind][key] += 1
        us[kind][key] += e.time_range.elapsed_us()
    total = sum(sum(c.values()) for c in us.values())
    res = {"launches": len(step), "device_ms": round(total / 1e3, 3)}
    for kind in groups:
        res[kind] = sum(groups[kind].values())
        res[f"{kind}_ms"] = round(sum(us[kind].values()) / 1e3, 3)
        res[f"{kind}_share"] = round(sum(us[kind].values()) / total, 4)
    for kind in ("cudnn_cublas", "other_torch"):
        res[f"{kind}_kernels"] = {k: [c, round(us[kind][k], 1)] for k, c in groups[kind].most_common()}
    res["library_kernels"] = dict(groups["library"].most_common())
    return res


def run(name, unet, vae, steps, device):
    from mvoc_b200.pipeline import I2VGenXLPipeline

    T, h, w = WORKLOADS[name]
    cond = inputs(T, h, w, device)
    pipe = I2VGenXLPipeline(unet, device, use_cuda_graphs=True, vae=vae)
    step_times(pipe, cond, 3, device)                                  # warm-up: lazy weight re-layouts, modules
    ms, out = step_times(pipe, cond, steps, device)
    replay = ms[1:]
    res = {"workload": name, "frames": T, "latents": [h, w], "batch": 2, "guidance": 9.0, "steps_timed": len(replay),
           "ms_per_guided_step": round(statistics.median(replay), 2),
           "ms_per_guided_step_min_max": [round(min(replay), 2), round(max(replay), 2)],
           "ms_first_step_with_capture": round(ms[0], 1), "finite": bool(torch.isfinite(out).all())}
    pipe.decode_latents(out)                                           # warm-up
    torch.cuda.synchronize()
    dec = []
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        video = pipe.decode_latents(out)
        e1.record()
        torch.cuda.synchronize()
        dec.append(e0.elapsed_time(e1))
    res["ms_decode"] = round(statistics.median(dec), 2)
    res["decoded_shape"] = list(video.shape)
    del pipe, video
    torch.cuda.empty_cache()
    res["launches_one_step"] = launch_list(unet, cond, device)
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--steps", type=int, default=12)
    ap.add_argument("--workloads", nargs="+", default=list(WORKLOADS), choices=list(WORKLOADS))
    ap.add_argument("--out", type=str, default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("recon_bench: needs a CUDA device (B200); there is no CPU measurement")
    device = torch.device("cuda:0")
    torch.cuda.set_device(device)
    torch.set_grad_enabled(False)
    unet, vae = build(device)
    for name in args.workloads:
        info0 = gpu_info()
        res = run(name, unet, vae, args.steps, device)
        info1 = gpu_info()
        res.update({k: v for k, v in info0.items() if k != "sm_mhz"})
        res["sm_mhz_before_after"] = [info0.get("sm_mhz"), info1.get("sm_mhz")]
        line = json.dumps(res)
        print(line, flush=True)
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "a") as f:
                f.write(line + "\n")


if __name__ == "__main__":
    main()
