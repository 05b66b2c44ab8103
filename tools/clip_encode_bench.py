"""CLIP image tower on one B200: the product encoder (mvoc_b200.clip, this library's kernels) against the same weights
run through torch (F.linear on cuBLAS, F.scaled_dot_product_attention, F.layer_norm, F.gelu; bf16).

    python tools/clip_encode_bench.py [--reps 20] [--out profiles/r05_clip_encode_bench.jsonl]

Three batches: 1 (the inversion's first frame), n+2 = 4 (one embedding per branch of a two-object composition) and 64
(T x (n_obj+2) images of config 2, what the reference encodes).  Full-width random-init weights (seeded), seeded
inputs.  One JSON line per batch: ms per call of both paths (warmed up, then alternated over --reps windows; median
and spread), TFLOP/s from the FLOPs the shapes imply, and their rel-L2 difference.  A last line times
mvoc_attn_d80_fwd against SDPA at 16 heads x 257 tokens.  Every line carries the GPU's name, power limit and SM clock
read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for p in (ROOT, HERE):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

from vae_decode_bench import gpu_info, timed  # noqa: E402

BATCHES = {"inversion": 1, "composition_branches": 4, "config2_reference_calls": 64}


def torch_forward(enc, x):
    """The same tower on torch kernels."""
    vm, cfg = enc.vision_model, enc.cfg
    n, p, d, h = x.shape[0], cfg.patch_size, cfg.hidden_size, cfg.num_attention_heads
    e = F.conv2d(x.to(enc.dtype), vm.embeddings.patch_embedding.weight, stride=p).flatten(2).transpose(1, 2)
    t = torch.cat([vm.embeddings.class_embedding.expand(n, 1, -1), e], 1) + vm.embeddings.position_embedding.weight
    t = F.layer_norm(t, (d,), vm.pre_layrnorm.weight, vm.pre_layrnorm.bias, 1e-5)
    for L in vm.encoder.layers:
        a = F.layer_norm(t, (d,), L.layer_norm1.weight, L.layer_norm1.bias, 1e-5)
        sa = L.self_attn
        q, k, v = (F.linear(a, m.weight, m.bias).view(n, -1, h, d // h).transpose(1, 2)
                   for m in (sa.q_proj, sa.k_proj, sa.v_proj))
        o = F.scaled_dot_product_attention(q, k, v).transpose(1, 2).reshape(n, -1, d)
        t = t + F.linear(o, sa.out_proj.weight, sa.out_proj.bias)
        m = F.layer_norm(t, (d,), L.layer_norm2.weight, L.layer_norm2.bias, 1e-5)
        t = t + F.linear(F.gelu(F.linear(m, L.mlp.fc1.weight, L.mlp.fc1.bias)), L.mlp.fc2.weight, L.mlp.fc2.bias)
    pooled = F.layer_norm(t[:, 0], (d,), vm.post_layernorm.weight, vm.post_layernorm.bias, 1e-5)
    return F.linear(pooled, enc.visual_projection.weight)


def tower_flops(cfg, n) -> float:
    """2 x MACs of the Linears (patch GEMM at K = 588) + 4 B H N^2 D of the attention."""
    d, f, tok = cfg.hidden_size, cfg.intermediate_size, cfg.num_patches + 1
    per_layer = 2 * tok * (4 * d * d + 2 * d * f) + 4 * tok * tok * d
    return n * (cfg.num_hidden_layers * per_layer + 2 * cfg.num_patches * d * 3 * cfg.patch_size ** 2
                + 2 * d * cfg.projection_dim)


def alternate(fns, reps):
    """Median and spread (min, max) of ms per call of each fn, windows of 5 calls alternated over `reps` rounds."""
    times = [[] for _ in fns]
    for _ in range(reps):
        for i, fn in enumerate(fns):
            times[i].append(timed(fn, 5)[0])
    return [(statistics.median(t), min(t), max(t)) for t in times]


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", type=str, default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("clip_encode_bench: no CUDA device (this tool measures on the GPU only)")
    from mvoc_b200 import ops
    from mvoc_b200.clip import CLIPVisionEncoder
    from mvoc_b200.unet3d import prepare

    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    torch.manual_seed(0)
    enc = CLIPVisionEncoder()
    for prm in enc.parameters():
        torch.nn.init.normal_(prm, std=0.02)
    enc = prepare(enc.eval().requires_grad_(False).to(dev, torch.bfloat16))
    info = gpu_info()
    lines = []
    with torch.no_grad():
        for name, n in BATCHES.items():
            x = torch.randn(n, 3, 224, 224, device=dev, generator=torch.Generator(dev).manual_seed(n))
            for _ in range(3):
                a, b = enc(x), torch_forward(enc, x)
            torch.cuda.synchronize()
            (pm, plo, phi), (tm, tlo, thi) = alternate([lambda: enc(x), lambda: torch_forward(enc, x)], args.reps)
            fl = tower_flops(enc.cfg, n)
            lines.append(dict(workload=name, batch=n, product_ms=round(pm, 4), product_ms_range=[round(plo, 4), round(phi, 4)],
                              torch_ms=round(tm, 4), torch_ms_range=[round(tlo, 4), round(thi, 4)],
                              speedup=round(tm / pm, 3), product_tflops=round(fl / pm / 1e9, 1),
                              torch_tflops=round(fl / tm / 1e9, 1), gflop=round(fl / 1e9, 2),
                              rel_l2_vs_torch=float((a.float() - b.float()).norm() / b.float().norm()), **info))
            print(json.dumps(lines[-1]), flush=True)
        # the attention alone at the tower's shape: 16 heads x 257 tokens, q / k / v slices of a fused projection
        for n in (1, 64):
            qkv = torch.randn(n, 257, 3 * 1280, device=dev, dtype=torch.bfloat16)
            q, k, v = qkv[..., :1280], qkv[..., 1280:2560], qkv[..., 2560:]
            sp = lambda t: t.view(n, 257, 16, 80).transpose(1, 2)
            fk = lambda: ops.attention_d80(q, k, v, 16)
            ft = lambda: F.scaled_dot_product_attention(sp(q), sp(k), sp(v))
            for _ in range(3):
                fk(), ft()
            torch.cuda.synchronize()
            (km, klo, khi), (sm, slo, shi) = alternate([fk, ft], args.reps)
            fl = 4.0 * n * 16 * 257 * 257 * 80
            lines.append(dict(workload=f"attn_d80_b{n}_h16_n257", kernel_us=round(km * 1e3, 2),
                              kernel_us_range=[round(klo * 1e3, 2), round(khi * 1e3, 2)], sdpa_us=round(sm * 1e3, 2),
                              sdpa_us_range=[round(slo * 1e3, 2), round(shi * 1e3, 2)],
                              kernel_tflops=round(fl / km / 1e9, 1), sdpa_tflops=round(fl / sm / 1e9, 1), **info))
            print(json.dumps(lines[-1]), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.writelines(json.dumps(l) + "\n" for l in lines)


if __name__ == "__main__":
    main()
