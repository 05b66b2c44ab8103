"""CLIP text tower on one B200: the product encoder (mvoc_b200.clip_text, this library's kernels) against the same
weights run through torch (F.linear on cuBLAS, F.scaled_dot_product_attention with is_causal, F.layer_norm, F.gelu;
bf16).

    python tools/clip_text_encode_bench.py [--reps 20] [--out profiles/r06_clip_text_encode_bench.jsonl]

Three batches of 77-token prompts: 1 (the inversion's prompt), 5 (the n+3 branches of a two-object composition) and 64.
Full-width random-init weights (seeded), seeded token ids.  One JSON line per batch: ms per call of both paths (warmed
up, then alternated over --reps windows; median and spread), TFLOP/s from the FLOPs the shapes imply, and their rel-L2
difference.  Then the causal attention alone (mvoc_attn_causal_fwd against SDPA with is_causal) at the tower's 16 heads
x 77 tokens and at 4096 tokens, where skipping the key blocks above the diagonal halves the work.  Every line carries
the GPU's name, power limit and SM clock read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for p in (ROOT, HERE):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

from clip_encode_bench import alternate  # noqa: E402
from vae_decode_bench import gpu_info  # noqa: E402

BATCHES = {"inversion": 1, "composition_branches_2obj": 5, "batch64": 64}
ATTN_SHAPES = [(1, 77), (5, 77), (64, 77), (1, 4096), (4, 4096)]   # (batch, tokens) at 16 heads of 64


def torch_forward(enc, ids):
    """The same tower on torch kernels."""
    tm, cfg = enc.text_model, enc.cfg
    n, d, h = ids.shape[0], cfg.hidden_size, cfg.num_attention_heads
    t = tm.embeddings.token_embedding.weight[ids] + tm.embeddings.position_embedding.weight[:ids.shape[1]]
    for L in tm.encoder.layers:
        a = F.layer_norm(t, (d,), L.layer_norm1.weight, L.layer_norm1.bias, 1e-5)
        sa = L.self_attn
        q, k, v = (F.linear(a, m.weight, m.bias).view(n, -1, h, d // h).transpose(1, 2)
                   for m in (sa.q_proj, sa.k_proj, sa.v_proj))
        o = F.scaled_dot_product_attention(q, k, v, is_causal=True).transpose(1, 2).reshape(n, -1, d)
        t = t + F.linear(o, sa.out_proj.weight, sa.out_proj.bias)
        m = F.layer_norm(t, (d,), L.layer_norm2.weight, L.layer_norm2.bias, 1e-5)
        t = t + F.linear(F.gelu(F.linear(m, L.mlp.fc1.weight, L.mlp.fc1.bias)), L.mlp.fc2.weight, L.mlp.fc2.bias)
    return F.layer_norm(t, (d,), tm.final_layer_norm.weight, tm.final_layer_norm.bias, 1e-5)


def causal_attention_flops(b, h, n, hd=64) -> float:
    """2 B H N (N + 1) hd: the causal half of Q K^T and P V (row r has r + 1 keys)."""
    return 2.0 * b * h * n * (n + 1) * hd


def tower_flops(cfg, n, tokens=77) -> float:
    """2 x MACs of the Linears (44.6 GFLOP per prompt at full width) + the causal attention."""
    d, f = cfg.hidden_size, cfg.intermediate_size
    per_layer = 2 * tokens * (4 * d * d + 2 * d * f) + causal_attention_flops(1, cfg.num_attention_heads, tokens,
                                                                                d // cfg.num_attention_heads)
    return n * cfg.num_hidden_layers * per_layer


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", type=str, default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("clip_text_encode_bench: no CUDA device (this tool measures on the GPU only)")
    from mvoc_b200 import ops
    from mvoc_b200.clip_text import CLIPTextEncoder

    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    torch.manual_seed(0)
    enc = CLIPTextEncoder()
    for prm in enc.parameters():
        torch.nn.init.normal_(prm, std=0.02)
    enc = enc.eval().requires_grad_(False).to(dev, torch.bfloat16)
    info = gpu_info()
    lines = []
    with torch.no_grad():
        for name, n in BATCHES.items():
            ids = torch.randint(0, enc.cfg.vocab_size, (n, 77), device=dev,
                                generator=torch.Generator(dev).manual_seed(n))
            for _ in range(3):
                a, b = enc(ids), torch_forward(enc, ids)
            torch.cuda.synchronize()
            (pm, plo, phi), (tm, tlo, thi) = alternate([lambda: enc(ids), lambda: torch_forward(enc, ids)], args.reps)
            fl = tower_flops(enc.cfg, n)
            lines.append(dict(workload=name, batch=n, product_ms=round(pm, 4), product_ms_range=[round(plo, 4), round(phi, 4)],
                              torch_ms=round(tm, 4), torch_ms_range=[round(tlo, 4), round(thi, 4)],
                              speedup=round(tm / pm, 3), product_tflops=round(fl / pm / 1e9, 1),
                              torch_tflops=round(fl / tm / 1e9, 1), gflop=round(fl / 1e9, 2),
                              rel_l2_vs_torch=float((a.float() - b.float()).norm() / b.float().norm()), **info))
            print(json.dumps(lines[-1]), flush=True)
        for n, N in ATTN_SHAPES:
            qkv = torch.randn(n, N, 3 * 1024, device=dev, dtype=torch.bfloat16)
            q, k, v = qkv[..., :1024], qkv[..., 1024:2048], qkv[..., 2048:]
            sp = lambda t: t.view(n, N, 16, 64).transpose(1, 2)
            fk = lambda: ops.attention_causal(q, k, v, 16)
            ft = lambda: F.scaled_dot_product_attention(sp(q), sp(k), sp(v), is_causal=True)
            for _ in range(3):
                a, b = fk(), ft()
            torch.cuda.synchronize()
            (km, klo, khi), (sm, slo, shi) = alternate([fk, ft], args.reps)
            fl = causal_attention_flops(n, 16, N)
            lines.append(dict(workload=f"attn_causal_b{n}_h16_n{N}", kernel_us=round(km * 1e3, 2),
                              kernel_us_range=[round(klo * 1e3, 2), round(khi * 1e3, 2)], sdpa_us=round(sm * 1e3, 2),
                              sdpa_us_range=[round(slo * 1e3, 2), round(shi * 1e3, 2)],
                              kernel_tflops=round(fl / km / 1e9, 1), sdpa_tflops=round(fl / sm / 1e9, 1),
                              rel_l2_vs_sdpa=float((a.float() - b.transpose(1, 2).reshape(a.shape).float()).norm()
                                                   / b.float().norm()), **info))
            print(json.dumps(lines[-1]), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.writelines(json.dumps(l) + "\n" for l in lines)


if __name__ == "__main__":
    main()
