"""VAE decode on one B200: the product decoder (mvoc_b200.vae, this library's kernels) against the same weights run
through torch (oracle.vae.DecoderKL in bf16, channels_last, cuDNN convs, torch SDPA in the mid block).

    python tools/vae_decode_bench.py [--reps 5] [--out results/vae_decode_bench.jsonl]

Two workloads, the decode stage of BASELINE configs 2 and 5: 16 frames of 64x64 latents (-> 512x512) and 32 frames of
88x160 latents (-> 704x1280).  Full-width random-init decoder (seeded), seeded latents.  Prints one JSON line per
workload: ms per video and frames/s of both paths (warmed up, then alternated over --reps repetitions; median and
spread), their rel-L2 difference, the peak memory of each path, the time per decode_chunk_size in {4, 16}, a
per-stage split, the mid-block attention kernel against torch SDPA at the same shape (with the SDPA kernels torch
actually ran) and the GPU's name, power limit and SM clock read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

WORKLOADS = {"config2": (16, 64, 64), "config5": (32, 88, 160)}   # frames, latent h, latent w


def gpu_info() -> dict:
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        line = subprocess.run(["nvidia-smi", "--id=0", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                              capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, plim, sm, smmax = [x.strip() for x in line.split(",")]
        return {"gpu": name, "power_limit_w": float(plim), "sm_mhz": float(sm), "sm_max_mhz": float(smmax)}
    except Exception as e:  # noqa: BLE001 - the numbers are reported without it, and say so
        return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi_error": str(e)}


def _sdpa_mid_attention(self, x):
    """oracle.vae._MidAttention with its softmax(QK^T)V replaced by F.scaled_dot_product_attention."""
    b, c, h, w = x.shape
    t = self.group_norm(x).view(b, c, h * w).transpose(1, 2)
    q, k, v = self.to_q(t), self.to_k(t), self.to_v(t)
    a = F.scaled_dot_product_attention(q[:, None], k[:, None], v[:, None])[:, 0]
    return x + self.to_out[0](a).transpose(1, 2).reshape(b, c, h, w)


def build(device):
    from mvoc_b200.unet3d import prepare
    from mvoc_b200.vae import AutoencoderKLDecoder
    from oracle import vae as ovae
    from tests.test_vae_cpu import diffusers_state_dict

    oracle = ovae.build_decoder(narrow=False, seed=0)
    product = AutoencoderKLDecoder().eval().requires_grad_(False)
    product.load_state_dict(diffusers_state_dict(oracle.state_dict()), strict=True)
    product = prepare(product.to(device, torch.bfloat16))
    ref = oracle.to(device, torch.bfloat16).to(memory_format=torch.channels_last)
    ref.mid_attn.forward = types.MethodType(_sdpa_mid_attention, ref.mid_attn)
    return product, ref


def timed(fn, reps=1):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps, out


def stage_split(product, ref, z):
    """ms per stage for one chunk of frames z [n, 4, h, w] (already scaled), both paths."""
    from mvoc_b200.unet3d import conv_nhwc

    d = product.decoder
    x = z.to(torch.bfloat16).permute(0, 2, 3, 1).contiguous()
    p_st = [("conv_in", lambda x: conv_nhwc(conv_nhwc(x, product.post_quant_conv), d.conv_in)),
            ("mid_block", d.mid_block)] + [(f"up_block{i}", b) for i, b in enumerate(d.up_blocks)] + \
           [("norm_out+conv_out", lambda x: conv_nhwc(d.conv_norm_out(x, silu=True), d.conv_out))]
    t_st = [("conv_in", lambda x: ref.conv_in(ref.post_quant_conv(x))),
            ("mid_block", lambda x: ref.mid_resnet2(ref.mid_attn(ref.mid_resnet1(x))))] + \
           [(f"up_block{i}", b) for i, b in enumerate(ref.up_blocks)] + \
           [("norm_out+conv_out", lambda x: ref.conv_out(F.silu(ref.conv_norm_out(x))))]
    out = {}
    for label, stages, x0 in (("product", p_st, x), ("torch", t_st, z.to(torch.bfloat16).contiguous(
            memory_format=torch.channels_last))):
        with torch.no_grad():
            for _ in range(2):                        # warm-up pass, then the timed pass
                xs, ms = x0, {}
                for name, f in stages:
                    ms[name], xs = timed(lambda: f(xs))
        out[label] = {k: round(v, 3) for k, v in ms.items()}
    return out


def attention_vs_sdpa(n_frames, h, w, device, reps=20):
    from mvoc_b200 import ops

    N = h * w
    torch.manual_seed(1)
    qkv = torch.randn(n_frames, N, 1536, device=device, dtype=torch.bfloat16)
    q, k, v = qkv[..., :512], qkv[..., 512:1024], qkv[..., 1024:]
    flop = 4.0 * n_frames * N * N * 512
    res = {"shape": [n_frames, N, 512]}
    sdpa = lambda: F.scaled_dot_product_attention(q[:, None], k[:, None], v[:, None])  # noqa: E731
    mine = lambda: ops.attention_d512(q, k, v)  # noqa: E731
    for f in (mine, sdpa, mine, sdpa):            # warm-up
        f()
    torch.cuda.synchronize()
    ms_m, ms_s = [], []
    for _ in range(3):
        ms_m.append(timed(mine, reps)[0])
        ms_s.append(timed(sdpa, reps)[0])
    o_m, o_s = mine().float(), sdpa()[:, 0].float()
    res.update(mvoc_ms=round(min(ms_m), 4), mvoc_tflops=round(flop / min(ms_m) / 1e9, 1),
               sdpa_ms=round(min(ms_s), 4), sdpa_tflops=round(flop / min(ms_s) / 1e9, 1),
               rel_l2_mvoc_vs_sdpa=float((o_m - o_s).norm() / o_s.norm()))
    # which kernels torch's default SDPA dispatch ran at D = 512 (a separate, profiled call)
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        sdpa()
        torch.cuda.synchronize()
    res["sdpa_cuda_kernels"] = sorted({e.name[:120] for e in prof.events() if e.device_type == DeviceType.CUDA})[:8]
    backends = {}
    from torch.nn.attention import SDPBackend, sdpa_kernel

    for be in (SDPBackend.FLASH_ATTENTION, SDPBackend.EFFICIENT_ATTENTION, SDPBackend.CUDNN_ATTENTION, SDPBackend.MATH):
        try:
            with sdpa_kernel(be):
                sdpa()
            torch.cuda.synchronize()
            backends[be.name] = "supported"
        except RuntimeError as e:
            backends[be.name] = "unsupported: " + str(e).splitlines()[0][:100]
    res["sdpa_backends_at_d512"] = backends
    return res


def run_workload(name, product, ref, reps, device):
    from mvoc_b200.pipeline import I2VGenXLPipeline
    from oracle import vae as ovae

    T, h, w = WORKLOADS[name]
    torch.manual_seed(0)
    latents = torch.randn(1, 4, T, h, w, device=device)
    pipe = I2VGenXLPipeline(None, device, vae=product)
    torch_dec = lambda z: ref(z.to(torch.bfloat16).contiguous(memory_format=torch.channels_last)).float()  # noqa
    paths = {"product": lambda c=4: pipe.decode_latents(latents, c),
             "torch": lambda c=4: ovae.decode_latents(torch_dec, latents, c)}
    peak = {}
    outs = {}
    for label, f in paths.items():                # warm-up, and the peak memory of one decode
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        outs[label] = f()
        torch.cuda.synchronize()
        peak[label] = round((torch.cuda.max_memory_allocated() - base) / 2 ** 20, 1)
        f()
    rel = float((outs["product"] - outs["torch"]).norm() / outs["torch"].norm())
    psnr = ovae.psnr(outs["product"], outs["torch"])
    del outs
    ms = {"product": [], "torch": []}
    for _ in range(reps):                          # alternate the two paths
        for label, f in paths.items():
            ms[label].append(timed(f)[0])
    chunk = {}
    for c in (4, 16):
        for label, f in paths.items():
            f(c)
            t = [timed(lambda: f(c))[0] for _ in range(2)]
            chunk[f"{label}_chunk{c}_ms"] = round(min(t), 2)
    res = {"workload": name, "frames": T, "latents": [h, w], "out_px": [8 * h, 8 * w], "reps": reps}
    for label in ("product", "torch"):
        med = statistics.median(ms[label])
        res[f"{label}_ms_per_video"] = round(med, 2)
        res[f"{label}_ms_min_max"] = [round(min(ms[label]), 2), round(max(ms[label]), 2)]
        res[f"{label}_frames_per_s"] = round(T / med * 1e3, 2)
        res[f"{label}_peak_mib"] = peak[label]
    res["speedup_product_vs_torch"] = round(res["torch_ms_per_video"] / res["product_ms_per_video"], 3)
    res["rel_l2_product_vs_torch"] = rel
    res["psnr_product_vs_torch_db"] = round(psnr, 2)
    res["chunk_ms_per_video"] = chunk
    z = (1 / 0.18215) * latents[0, :, :4].permute(1, 0, 2, 3)
    res["stage_ms_chunk4"] = stage_split(product, ref, z)
    res["attention"] = attention_vs_sdpa(4, h, w, device)
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--workloads", nargs="+", default=list(WORKLOADS), choices=list(WORKLOADS))
    ap.add_argument("--out", type=str, default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("vae_decode_bench: needs a CUDA device (B200); there is no CPU measurement")
    device = torch.device("cuda:0")
    torch.cuda.set_device(device)
    torch.set_grad_enabled(False)
    product, ref = build(device)
    for name in args.workloads:
        info0 = gpu_info()
        res = run_workload(name, product, ref, args.reps, device)
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
