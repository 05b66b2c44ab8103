"""VAE encode on one B200: the product encoder (mvoc_b200.vae, this library's kernels) against the same weights run
through torch (oracle.vae_encoder.EncoderKL in bf16, channels_last, cuDNN convs, torch SDPA in the mid block).

    python tools/vae_encode_bench.py [--reps 5] [--out profiles/r04_vae_encode_bench.jsonl]

Two workloads, the encode stage of BASELINE configs 2 and 5: 16 frames of 512x512 and 32 frames of 704x1280, encoded
4 frames at a time (encode_vae_video's default).  Full-width random-init encoder (seeded), seeded frames.  One JSON
line per workload: ms per video and frames/s of both paths (warmed up, then alternated over --reps repetitions;
median and spread), TFLOP/s from the FLOPs the shapes imply, their rel-L2 difference and the peak memory of each
path.  A last line times mvoc_conv3x3_s2_nhwc against cuDNN at the encoder's three downsampler shapes (pads (0, 1),
cuDNN on the F.pad-ed input as the torch path runs it) and the UNet's three (pads (1, 1), config 2's 80 frames).
Every line carries the GPU's name, power limit and SM clock read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import types

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for p in (ROOT, HERE):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402
import torch.nn as nn  # noqa: E402
import torch.nn.functional as F  # noqa: E402

from vae_decode_bench import _sdpa_mid_attention, gpu_info, timed  # noqa: E402

WORKLOADS = {"config2": (16, 512, 512), "config5": (32, 704, 1280)}   # frames, height, width
CHUNK = 4
S2_SHAPES = {   # N, H, W, C, pads
    "encoder_down0": (CHUNK, 512, 512, 128, (0, 1)), "encoder_down1": (CHUNK, 256, 256, 256, (0, 1)),
    "encoder_down2": (CHUNK, 128, 128, 512, (0, 1)),
    "unet_down0": (80, 64, 64, 320, (1, 1)), "unet_down1": (80, 32, 32, 640, (1, 1)),
    "unet_down2": (80, 16, 16, 1280, (1, 1)),
}


def build(device):
    from mvoc_b200.unet3d import prepare
    from mvoc_b200.vae import AutoencoderKLEncoder
    from oracle import vae_encoder as oenc
    from tests.test_vae_encode_cpu import diffusers_encoder_state_dict

    oracle = oenc.build_encoder(narrow=False, seed=0)
    product = AutoencoderKLEncoder().eval().requires_grad_(False)
    product.load_state_dict(diffusers_encoder_state_dict(oracle.state_dict()), strict=True)
    product = prepare(product.to(device, torch.bfloat16))
    ref = oracle.to(device, torch.bfloat16).to(memory_format=torch.channels_last)
    ref.mid_attn.forward = types.MethodType(_sdpa_mid_attention, ref.mid_attn)
    return product, ref


def encoder_flops(ref, frames, H, W, device) -> float:
    """FLOPs of one pass over `frames` frames of H x W: 2 x MACs of every conv and Linear (forward hooks on one
    frame) plus 4 N^2 C for the two products of the mid-block attention over its N tokens."""
    total = [0.0]

    def hook(m, inp, out):
        k = m.kernel_size[0] * m.kernel_size[1] if isinstance(m, nn.Conv2d) else 1
        total[0] += 2.0 * out.numel() * (m.in_channels if isinstance(m, nn.Conv2d) else m.in_features) * k

    hs = [m.register_forward_hook(hook) for m in ref.modules() if isinstance(m, (nn.Conv2d, nn.Linear))]
    with torch.no_grad():
        moments = ref(torch.zeros(1, 3, H, W, device=device, dtype=torch.bfloat16).contiguous(
            memory_format=torch.channels_last))
    for h in hs:
        h.remove()
    n = moments.shape[2] * moments.shape[3]
    return frames * (total[0] + 4.0 * n * n * ref.mid_attn.to_q.in_features)


def run_workload(name, product, ref, reps, device):
    from mvoc_b200.pipeline import I2VGenXLPipeline

    T, H, W = WORKLOADS[name]
    torch.manual_seed(0)
    frames = torch.rand(T, 3, H, W, device=device) * 2 - 1
    pipe = I2VGenXLPipeline(None, device, vae_encoder=product)
    torch_enc = lambda x: ref(x.to(torch.bfloat16).contiguous(memory_format=torch.channels_last)).float()  # noqa

    def moments(enc):
        return torch.cat([enc(frames[i:i + CHUNK]) for i in range(0, T, CHUNK)])

    paths = {"product": lambda: moments(product), "torch": lambda: moments(torch_enc)}
    peak, outs = {}, {}
    for label, f in paths.items():                # warm-up, and the peak memory of one encode
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        outs[label] = f()
        torch.cuda.synchronize()
        peak[label] = round((torch.cuda.max_memory_allocated() - base) / 2 ** 20, 1)
        f()
    rel = float((outs["product"] - outs["torch"]).norm() / outs["torch"].norm())
    del outs
    ms = {"product": [], "torch": []}
    for _ in range(reps):                          # alternate the two paths
        for label, f in paths.items():
            ms[label].append(timed(f)[0])
    flops = encoder_flops(ref, T, H, W, device)
    res = {"workload": name, "frames": T, "px": [H, W], "chunk": CHUNK, "reps": reps,
           "tflop_per_video": round(flops / 1e12, 3)}
    for label in ("product", "torch"):
        med = statistics.median(ms[label])
        res[f"{label}_ms_per_video"] = round(med, 2)
        res[f"{label}_ms_min_max"] = [round(min(ms[label]), 2), round(max(ms[label]), 2)]
        res[f"{label}_frames_per_s"] = round(T / med * 1e3, 2)
        res[f"{label}_tflops"] = round(flops / med / 1e9, 1)
        res[f"{label}_peak_mib"] = peak[label]
    res["speedup_product_vs_torch"] = round(res["torch_ms_per_video"] / res["product_ms_per_video"], 3)
    res["rel_l2_moments_product_vs_torch"] = rel
    # the full path of encode_vae_video (chunks, posterior sample, scaling) once, for its overhead over the moments
    gen = torch.Generator(device=device)
    pipe.encode_vae_video(frames, gen.manual_seed(0))
    res["encode_vae_video_ms"] = round(statistics.median(
        [timed(lambda: pipe.encode_vae_video(frames, gen.manual_seed(0)))[0] for _ in range(3)]), 2)
    return res


def s2_vs_cudnn(device, reps=20):
    from mvoc_b200 import ops

    out = {"workload": "conv3x3_s2_vs_cudnn", "reps": reps}
    for name, (N, H, W, C, pad) in S2_SHAPES.items():
        torch.manual_seed(1)
        x = torch.randn(N, H, W, C, device=device, dtype=torch.bfloat16)
        w = (torch.randn(C, C, 3, 3, device=device) * (9 * C) ** -0.5).to(torch.bfloat16)
        b = torch.randn(C, device=device, dtype=torch.bfloat16)
        wt = ops.conv_taps(w)
        wcl = w.contiguous(memory_format=torch.channels_last)
        xn = x.permute(0, 3, 1, 2)                  # channels_last NCHW view
        if pad == (0, 1):
            cudnn = lambda: F.conv2d(F.pad(xn, (0, 1, 0, 1)), wcl, b, stride=2)  # noqa: E731
        else:
            cudnn = lambda: F.conv2d(xn, wcl, b, stride=2, padding=1)  # noqa: E731
        mine = lambda: ops.conv3x3_s2(x, wt, b, pad=pad)  # noqa: E731
        for f in (mine, cudnn, mine, cudnn):
            f()
        torch.cuda.synchronize()
        t_m, t_c = [], []
        for _ in range(3):                          # alternated
            t_m.append(timed(mine, reps)[0])
            t_c.append(timed(cudnn, reps)[0])
        y_m, y_c = mine().float(), cudnn().permute(0, 2, 3, 1).float()
        Ho, Wo = y_m.shape[1], y_m.shape[2]
        flop = 2.0 * N * Ho * Wo * C * 9 * C
        out[name] = {"shape": [N, H, W, C, C], "pads": list(pad), "mvoc_ms": round(statistics.median(t_m), 4),
                     "cudnn_ms": round(statistics.median(t_c), 4),
                     "mvoc_tflops": round(flop / statistics.median(t_m) / 1e9, 1),
                     "cudnn_tflops": round(flop / statistics.median(t_c) / 1e9, 1),
                     "mvoc_ms_min_max": [round(min(t_m), 4), round(max(t_m), 4)],
                     "cudnn_ms_min_max": [round(min(t_c), 4), round(max(t_c), 4)],
                     "rel_l2_mvoc_vs_cudnn": float((y_m - y_c).norm() / y_c.norm())}
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--workloads", nargs="+", default=list(WORKLOADS), choices=list(WORKLOADS))
    ap.add_argument("--out", type=str, default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("vae_encode_bench: needs a CUDA device (B200); there is no CPU measurement")
    device = torch.device("cuda:0")
    torch.cuda.set_device(device)
    torch.set_grad_enabled(False)
    product, ref = build(device)
    jobs = [lambda n=n: run_workload(n, product, ref, args.reps, device) for n in args.workloads]
    jobs.append(lambda: s2_vs_cudnn(device))
    for job in jobs:
        info0 = gpu_info()
        res = job()
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
