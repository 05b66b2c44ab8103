"""CLIP text tower on the GPU: both causal attention kernels element by element against float64 (the bound and input
kinds of test_attention_matrix_gpu.py with the reference restricted to keys <= the query), the full-width encoder
against transformers' CLIPTextModel in fp32 on the same random weights, chunk invariance of encode_prompt, and the
scripts' prompt embeddings.

The causal kernel is the plain head_dim-64 kernel of attn_tc.cu at the default exp2 split (0xA8) with a per-CTA key
block count of min(ceil(N / 128), m + 1) for query tile m and a diagonal select.  Its arithmetic on every key it uses
is the dense kernel's, so the dense bound applies row by row over the keys 0..r.  Without a GPU, a float32 emulation of
the causal kernel stays inside that bound on every input kind, and an off-by-one diagonal (the key r itself masked,
or the key r + 1 let in) breaks it (a key let in moves a retrieval row by nothing visible; uniform and random rows
see it).  Retrieval inputs here choose, for row r, the key r, r - 1, 0 or a random key <= r, so the diagonal and its
neighbours are hit in every query tile."""
import copy
import json
import math
import os

import pytest
import torch
import torch.nn.functional as F

from tests.test_attention_matrix_gpu import (ACC, DTYPES, HD, KINDS, LAYOUTS, RESCALE_LOG2, SCORE_FP32, SIGMA, UNIT,
                                             check_attention, ex2_poly32, exp2_bound, f32, fma32, groups, make_inputs,
                                             out_maker, qkv_operands, run_twice, same_bits)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FULL = dict(vocab_size=49408, hidden_size=1024, intermediate_size=4096, num_hidden_layers=23, num_attention_heads=16,
            max_position_embeddings=77)
CAUSAL_MASK = 0xA8                        # the exp2 split of the causal kernels
CAUSAL_NS = [1, 2, 63, 64, 65, 77, 127, 128, 129, 255, 256, 257, 1000]
CAUSAL_BH = {1: (3, 16), 2: (2, 3), 63: (2, 2), 64: (1, 3), 65: (2, 2), 77: (2, 16), 127: (1, 3), 128: (2, 2),
             129: (3, 1), 255: (1, 2), 256: (2, 1), 257: (1, 3), 1000: (1, 2)}


def rel_l2(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-300))


# ------------------------------------------------------------------ inputs, reference and bound
def causal_inputs(kind, B, H, N, seed):
    """float32 q, k, v [B, N, H*64] of one input kind.  Retrieval: row r's query is 4 k_sigma(r) with sigma(r) = r,
    r - 1, 0 or a random key <= r, cycling with (batch, head, row)."""
    if kind != "retrieval":
        return make_inputs(kind, B, H, N, N, HD, B, "cpu", seed)
    gen = torch.Generator().manual_seed(seed)
    k = torch.randint(0, 2, (B, H, N, HD), generator=gen).float() * 2 - 1
    rows = torch.arange(N)
    which = (torch.arange(B * H).view(B, H, 1) + rows) % 4
    rnd = (torch.rand(B, H, N, generator=gen) * (rows + 1)).long().clamp(max=N - 1)
    sel = torch.where(which == 0, rows, torch.where(which == 1, (rows - 1).clamp_min(0),
                                                    torch.where(which == 2, torch.zeros_like(rows), rnd)))
    q = 4 * torch.gather(k, 2, sel.unsqueeze(-1).expand(-1, -1, -1, HD))
    v = torch.randn(B, H, N, HD, generator=gen)
    to = lambda t: t.permute(0, 2, 1, 3).reshape(B, N, H * HD)
    return to(q), to(k), to(v)


def causal_reference(q, k, v, scale, dtype, E):
    """The bound of test_attention_matrix_gpu.reference over the keys 0..r of row r: q, k, v [G, N, D] (16-bit) ->
    float64 ref, bound and the largest softmax weight of every row."""
    G, N, _ = q.shape
    qd, kd, vd = q.double(), k.double(), v.double()
    ka, va = kd.abs().transpose(1, 2), vd.abs()
    u = UNIT[dtype]
    ref = torch.empty(G, N, vd.shape[2], dtype=torch.float64, device=q.device)
    bound, top = torch.empty_like(ref), torch.empty(G, N, dtype=torch.float64, device=q.device)
    keys = torch.arange(N, device=q.device)
    step = max(1, 2 ** 26 // (G * N))
    for i in range(0, N, step):
        qc = qd[:, i:i + step]
        allowed = keys[None, :] <= torch.arange(i, i + qc.shape[1], device=q.device)[:, None]
        s = (scale * (qc @ kd.transpose(1, 2))).masked_fill(~allowed, -math.inf)
        e = torch.exp(s - s.amax(-1, keepdim=True))
        den = e.sum(-1, keepdim=True)
        pi = e / den
        r, A = pi @ vd, pi @ va
        qk = (qc.abs() @ ka).masked_fill(~allowed, 0.0)
        delta = ACC * scale * qk.amax(-1, keepdim=True) + SCORE_FP32 * s.abs().masked_fill(~allowed, 0.0).amax(
            -1, keepdim=True)
        v1 = allowed.double() @ va
        ref[:, i:i + step] = r
        bound[:, i:i + step] = u * r.abs() + (u + E + ACC + 2 * delta) * A + SIGMA[dtype] * v1 / den
        top[:, i:i + step] = pi.amax(-1)
    return ref, bound, top


# ------------------------------------------------------------------ the CPU emulation of the causal kernel
DIAG_SHIFT = {None: 0, "diag_excluded": -1, "diag_plus_one": 1}


def emulate_causal(q, k, v, scale, dtype, mask=CAUSAL_MASK, mutant=None):
    """The causal kernel's arithmetic in fp32 on [G, N, 64] groups: query tile m runs key blocks 0..m (128 keys each,
    TMA zero fill past N), keys past the row and past N score -inf, then test_attention_matrix_gpu's emulation of the
    dense kernel (lagging maximum, exp2 split, l from the unrounded p, P rounded).  Mutants move the diagonal by one:
    diag_excluded masks the key r itself, diag_plus_one lets the key r + 1 in."""
    BN = 128
    G, N, _ = q.shape
    sl2 = torch.tensor(f32(scale), dtype=torch.float32) * torch.tensor(1.4426950408889634, dtype=torch.float32)
    emu = torch.tensor([(mask >> ((c // 2) % 8)) & 1 for c in range(BN)], dtype=torch.bool)
    out = torch.empty(G, N, v.shape[2], dtype=dtype)
    for m in range(-(-N // BN)):
        r0, r1 = m * BN, min(N, (m + 1) * BN)
        nk = min(N, (m + 1) * BN)
        kp = F.pad(k[:, :nk].double(), (0, 0, 0, (m + 1) * BN - nk))
        vp = F.pad(v[:, :nk].float(), (0, 0, 0, (m + 1) * BN - nk))
        s_all = (q[:, r0:r1].double() @ kp.transpose(1, 2)).float()
        lim = torch.arange(r0, r1)[:, None] + DIAG_SHIFT[mutant]
        m_used = l = O = None
        for j in range(m + 1):
            col = j * BN + torch.arange(BN)[None, :]
            s = s_all[..., j * BN:(j + 1) * BN].masked_fill((col > lim) | (col >= N), -math.inf)
            mx = s.amax(-1)
            if j == 0:
                m_used, l, O = mx, torch.zeros(G, r1 - r0), torch.zeros(G, r1 - r0, v.shape[2])
            else:
                m_new = torch.maximum(m_used, mx)
                need = (m_new - m_used) * sl2 > RESCALE_LOG2
                f = torch.where(need, torch.exp2((m_used - m_new) * sl2), torch.ones(()))
                l, O = l * f, O * f[..., None]
                m_used = torch.where(need, m_new, m_used)
            x = fma32(s, sl2, (-m_used * sl2)[..., None])
            p = torch.where(emu, ex2_poly32(x), torch.exp2(x))
            l = l + p.sum(-1)
            O = O + (p.to(dtype).double() @ vp[:, j * BN:(j + 1) * BN].double()).float()
        out[:, r0:r1] = (O * (1.0 / l)[..., None]).to(dtype)
    return out


EMU_SHAPE = (1, 2, 300)     # B, H, N: three query tiles and key blocks, the last ragged


def emulation_case(kind, dtype, mutant=None):
    B, H, N = EMU_SHAPE
    q, k, v = (groups(t.to(dtype), H, HD) for t in causal_inputs(kind, B, H, N, seed=13))
    out = emulate_causal(q, k, v, HD ** -0.5, dtype, mutant=mutant)
    ref, bound, top = causal_reference(q, k, v, f32(HD ** -0.5), dtype, exp2_bound(CAUSAL_MASK))
    if kind == "retrieval":
        assert float(top.min()) >= 0.99
    ratio = ((out.double() - ref).abs() / bound.clamp_min(torch.finfo(torch.float64).tiny)).nan_to_num(math.inf)
    return float(ratio.max())


@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("kind", KINDS)
def test_causal_emulation_inside_the_bound(kind, dt):
    r = emulation_case(kind, DTYPES[dt])
    print(f"causal emulation {kind} {dt}: max err/bound {r:.4f}")
    assert r <= 1.0


@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("mutant,kind", [("diag_excluded", "retrieval"), ("diag_excluded", "uniform"),
                                         ("diag_plus_one", "uniform"), ("diag_plus_one", "random")])
def test_off_by_one_diagonal_breaks_the_bound(mutant, kind, dt):
    r = emulation_case(kind, DTYPES[dt], mutant)
    print(f"mutant {mutant} on {kind} {dt}: max err/bound {r:.1f}")
    assert r > 4.0, f"the bound does not see the {mutant} mutant (max err/bound {r:.3f})"


# ------------------------------------------------------------------ both causal kernels against float64
@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("N", CAUSAL_NS)
@pytest.mark.parametrize("dt", list(DTYPES))
def test_attention_causal_vs_float64(cuda_device, dt, N, layout, kind):
    from mvoc_b200 import ops

    dtype, dev = DTYPES[dt], cuda_device
    B, H = CAUSAL_BH[N]
    scale = HD ** -0.5
    desc = f"ops.attention_causal {dt} mask {CAUSAL_MASK:#04x} causal, 128-key blocks, B={B} H={H} N={N} {layout} {kind}"
    q, k, v = qkv_operands(*causal_inputs(kind, B, H, N, seed=N + H + 7), dtype, dev, layout)
    make_out = out_maker((B, N, H * HD), dtype, dev, layout)
    out = run_twice(desc, lambda o: ops.attention_causal(q.t, k.t, v.t, H, scale, o), make_out,
                    {"q": q, "k": k, "v": v})
    ref, bound, top = causal_reference(groups(q.t, H, HD), groups(k.t, H, HD), groups(v.t, H, HD), f32(scale), dtype,
                                       exp2_bound(CAUSAL_MASK))
    if kind == "retrieval":
        assert float(top.min()) >= 0.99, f"{desc}: retrieval input puts only {float(top.min()):.3f} on its key"
    r = check_attention(desc, groups(out, H, HD), ref, bound, H, -(-N // 128))
    print(f"[attention matrix] {desc}: max err/bound {r:.4f}")
    b = B - 1
    alone = ops.attention_causal(q.t[b:b + 1], k.t[b:b + 1], v.t[b:b + 1], H, scale)
    torch.cuda.synchronize()
    assert same_bits(alone, out[b:b + 1]), f"{desc}: batch {b} alone differs from batch {b} of the full call"
    if N > 128:
        # the first query tile never reads a key block above the diagonal: NaN keys and values there change no bit
        kk, vv = k.t.clone(), v.t.clone()
        kk[:, 128:], vv[:, 128:] = math.nan, math.nan
        o2 = ops.attention_causal(q.t, kk, vv, H, scale)
        torch.cuda.synchronize()
        assert same_bits(o2[:, :128], out[:, :128]), f"{desc}: the first query tile read keys past its diagonal"


@pytest.mark.gpu
def test_attention_causal_rejects_bad_operands(cuda_device):
    from mvoc_b200 import _cabi, ops

    z = lambda *s, dt=torch.bfloat16: torch.zeros(*s, dtype=dt, device=cuda_device)
    x = z(2, 77, 128)
    with pytest.raises(ValueError, match="attention_causal"):
        ops.attention_causal(x, z(2, 76, 128), z(2, 76, 128), 2)
    with pytest.raises(ValueError, match="attention_causal"):
        ops.attention_causal(x, x, x, 2, out=z(2, 77, 128, dt=torch.float16))
    with pytest.raises(ValueError, match="attention_causal"):
        ops.attention_causal(x, x, x, 2, out=z(2, 76, 128))
    with pytest.raises(ValueError):
        ops.attention_causal(z(2, 77, 160), z(2, 77, 160), z(2, 77, 160), 2)
    with pytest.raises(_cabi.MvocError, match="mvoc_attn_causal_fwd"):
        ops.attention_causal(x.float(), x.float(), x.float(), 2)


# ------------------------------------------------------------------ the full-width encoder
@pytest.fixture(scope="module")
def full_models(cuda_device):
    """(transformers fp32 model, product encoder in bf16) on the same random-init weights."""
    transformers = pytest.importorskip("transformers")
    from mvoc_b200.clip_text import CLIPTextEncoder

    torch.manual_seed(0)
    cfg = transformers.CLIPTextConfig(hidden_act="gelu", layer_norm_eps=1e-5, **FULL)
    cfg._attn_implementation = "sdpa"
    with torch.device(cuda_device):
        ref = transformers.CLIPTextModel(cfg).eval().requires_grad_(False)
    ours = CLIPTextEncoder().eval().requires_grad_(False)
    ours.load_state_dict({k: v.cpu() for k, v in ref.state_dict().items()}, strict=True)
    return ref, ours.to(cuda_device, torch.bfloat16)


def prompt_ids(n, seed):
    """[n, 77] ids shaped like tokenized prompts: BOS, 0-75 word tokens, EOS, then pad ("!", id 0)."""
    g = torch.Generator().manual_seed(seed)
    ids = torch.zeros(n, 77, dtype=torch.int64)
    for i in range(n):
        w = int(torch.randint(0, 76, (1,), generator=g))
        ids[i, 0] = 49406
        ids[i, 1:w + 1] = torch.randint(1, 49406, (w,), generator=g)
        ids[i, w + 1] = 49407
    return ids


# The product's last_hidden_state against transformers fp32 must stay within 1.5x the error of the same transformers
# model run in bf16 (cuBLAS + SDPA) on the same ids, measured in the same test; and cosine >= 0.999 per prompt.
ENVELOPE, MIN_COS = 1.5, 0.999


@pytest.mark.gpu
@pytest.mark.parametrize("batch", [1, 5, 64])
def test_encoder_full_width_vs_transformers(cuda_device, full_models, batch):
    ref, ours = full_models
    ids = prompt_ids(batch, batch).to(cuda_device)
    tf32 = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
    try:
        with torch.no_grad():
            want = ref(input_ids=ids).last_hidden_state
            ref16 = copy.deepcopy(ref).to(torch.bfloat16)
            env = ref16(input_ids=ids).last_hidden_state
            del ref16
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = tf32
    got = ours(ids)
    torch.cuda.synchronize()
    assert got.shape == want.shape == (batch, 77, 1024) and got.dtype == torch.bfloat16
    err, env_err = rel_l2(got, want), rel_l2(env, want)
    cos = F.cosine_similarity(got.double().flatten(1), want.double().flatten(1), dim=-1)
    print(f"[clip text tower, batch {batch}] rel L2 {err:.4e} (torch bf16 envelope {env_err:.4e}), "
          f"min cosine {float(cos.min()):.6f}")
    assert err <= ENVELOPE * env_err, f"rel L2 {err:.3e} > {ENVELOPE} x envelope {env_err:.3e}"
    assert float(cos.min()) >= MIN_COS


PROMPTS = ["", "a boat and a surfer on the sea", "blurry", "it's a photo of 1 dog running!",
           " ".join(["surfer"] * 90), "café naïve, boats"] * 3


@pytest.mark.gpu
def test_encode_prompt_is_bit_invariant_to_chunk_size(cuda_device, full_models, tmp_path):
    from mvoc_b200.clip_text import CLIPTokenizer
    from mvoc_b200.pipeline import I2VGenXLPipeline
    from tests.test_clip_text_cpu import write_tokenizer_dir

    _, ours = full_models
    write_tokenizer_dir(str(tmp_path), "!")
    pipe = I2VGenXLPipeline(None, cuda_device, text_encoder=ours, tokenizer=CLIPTokenizer.from_dir(str(tmp_path)))
    outs = [pipe.encode_prompt(PROMPTS, encode_chunk_size=c) for c in (64, 16, 5, 1)]
    singly = torch.cat([pipe.encode_prompt(p) for p in PROMPTS])
    torch.cuda.synchronize()
    assert outs[0].shape == (len(PROMPTS), 77, 1024)
    for o in outs[1:] + [singly]:
        assert torch.equal(o, outs[0])


# ------------------------------------------------------------------ the scripts
@pytest.mark.gpu
def test_scripts_prompt_embeds_equal_encode_prompt(cuda_device, full_models, tmp_path, monkeypatch):
    """inverse.py and composite.py with --synthetic --text_encoder_state_dict FILE --tokenizer_dir DIR: what reaches the
    step loops is encode_prompt of the config's prompts (inverse: inverse_config.prompt; composite:
    [ddim_inv_prompt x (n+1), negative_prompt, prompt])."""
    from mvoc_b200 import composite, inverse
    from mvoc_b200.pipeline import I2VGenXLPipeline
    from tests.test_clip_text_cpu import write_tokenizer_dir

    ref, _ = full_models
    enc_path, tok_dir = str(tmp_path / "text_encoder.pt"), str(tmp_path / "tokenizer")
    torch.save({k: v.to("cpu", torch.bfloat16) for k, v in ref.state_dict().items()}, enc_path)
    write_tokenizer_dir(tok_dir, "!")
    T, w_px, h_px = 2, 128, 64

    seen = {}

    def record(self, latents, prompt_embeds, image_embeddings, image_latents, fps, **kw):
        seen.update(pipe=self, prompt_embeds=prompt_embeds.clone())
        return {}

    monkeypatch.setattr(I2VGenXLPipeline, "invert", record)
    data = tmp_path / "inv"
    data.mkdir()
    cfg = data / "group.json"
    cfg.write_text(json.dumps([{"active": True, "force_recompute_latents": True, "video_name": "clip",
                                "data_dir": str(data), "image_size": [w_px, h_px], "n_frames": T,
                                "inverse_config": {"prompt": "a boat and a surfer on the sea"}}]))
    template = os.path.join(ROOT, "configs", "group_inversion", "template.yaml")
    assert inverse.main(template, str(cfg), synthetic_inputs=True, text_encoder_state_dict=enc_path,
                        tokenizer_dir=tok_dir) == 1
    want = seen["pipe"].encode_prompt(["a boat and a surfer on the sea"])
    assert seen["prompt_embeds"].shape == (1, 77, 1024)
    assert torch.equal(seen["prompt_embeds"], want)

    got = {}

    def run_entry(pipe, config, device, conditioning=None, allow_synthetic=False):
        got.update(pipe=pipe, cond=conditioning)
        return torch.zeros(1, 4, T, h_px // 8, w_px // 8, device=device)

    monkeypatch.setattr(composite, "run_entry", run_entry)
    data = tmp_path / "comp"
    data.mkdir()
    cfg = data / "group.json"
    cfg.write_text(json.dumps([{"active": True, "video_name": "clip", "edited_video_name": "clip_edit",
                                "data_dir": str(data), "image_size": [w_px, h_px], "n_frames": T,
                                "obj_mask_path": ["m0", "m1"], "obj_ddim_latents_path": ["l0", "l1"],
                                "prompt": "a boat and a surfer on the sea", "negative_prompt": "blurry",
                                "ddim_inv_prompt": "", "output_dir": str(data / "out")}]))
    template = os.path.join(ROOT, "configs", "group_composite", "template.yaml")
    assert composite.main(template, str(cfg), synthetic_inputs=True, text_encoder_state_dict=enc_path,
                          tokenizer_dir=tok_dir, max_entries=1) == 1
    emb = got["cond"]["prompt_embeds"]
    want = got["pipe"].encode_prompt(["", "blurry", "a boat and a surfer on the sea"])
    assert emb.shape == (5, 77, 1024)
    for i, j in ((0, 0), (1, 0), (2, 0), (3, 1), (4, 2)):
        assert torch.equal(emb[i], want[j])
