"""CLIP image tower on the GPU: mvoc_attn_d80_fwd's error codes, every compiled mvoc_linear_gelu kernel element by
element against float64, the full-width encoder against transformers' CLIPVisionModelWithProjection in
fp32 on the same random weights, chunk invariance, and the scripts' embeddings."""
import json
import os

import pytest
import torch
import torch.nn.functional as F

from tests.test_gemm_matrix_gpu import (ACC, DTYPES, ERF_ERR, GELU_SLOPE, LINEAR_N, UNIT, Guarded, Kernel, check_bound,
                                        device_sms, linear_dims, linear_terms, operand, run_twice, tensor)

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FULL = dict(hidden_size=1280, intermediate_size=5120, num_hidden_layers=32, num_attention_heads=16, patch_size=14,
            image_size=224, projection_dim=1024)


def rel_l2(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-300))


# ------------------------------------------------------------------ mvoc_attn_d80_fwd
# (element by element against float64 attention: tests/test_attention_matrix_gpu.py)
def test_attention_d80_error_codes(cuda_device):
    from mvoc_b200 import _cabi, ops

    x = torch.zeros(1, 4, 160, device=cuda_device, dtype=torch.bfloat16)
    with pytest.raises(ValueError, match="attention_d80"):
        ops.attention_d80(x, x, x, 3)
    with pytest.raises(_cabi.MvocError, match="mvoc_attn_d80_fwd"):
        ops.attention_d80(x.float(), x.float(), x.float(), 2)


# ------------------------------------------------------------------ mvoc_linear_gelu: every compiled kernel
GELU_CASES = [(bn, pair, dt, shape) for bn in (256, 192, 160, 128, 64) for pair in (False, True) for dt in DTYPES
              for shape in ("long", "m1", "m129")]


def gelu_reference(x, w, b, dtype):
    """gelu(x w^T + b) in float64 and its bound: the accumulation allowance goes through gelu (slope <= 1.13) and the
    epilogue's erf approximation adds ERF_ERR relative to the pre-activation."""
    z, mag = linear_terms(x, w, b)
    ref = F.gelu(z)
    return ref, UNIT[dtype] * ref.abs() + GELU_SLOPE * ACC * mag + ERF_ERR * z.abs()


@pytest.mark.parametrize("case", GELU_CASES, ids=lambda c: f"bn{c[0]}-{'pair' if c[1] else 'one_cta'}-{c[2]}-{c[3]}")
def test_linear_gelu_every_kernel_vs_float64(cuda_device, case):
    from mvoc_b200 import ops

    bn, pair, dt, shape = case
    sms = device_sms(cuda_device)
    M, K, N, extras = linear_dims("linear", bn, shape, sms)
    dtype, dev = DTYPES[dt], cuda_device
    torch.manual_seed(M + K + N + bn + 1)
    variant = bn << 8 | int(pair)
    kernel = Kernel("mvoc_linear_gelu", dtype, (M, 1, 1), N, variant, sms)
    assert (kernel.bn, kernel.pair, kernel.tail) == (bn, pair, N % bn), f"the plan does not launch {kernel}"
    w = operand((N, K), dtype, dev, K ** -0.5)
    b = operand((N,), dtype, dev) if extras else None
    x = operand((M, K), dtype, dev, ld=K + 64)
    make_out = lambda: Guarded((M, N), dtype, dev, ld=N + 96)
    out = run_twice(kernel, lambda o: ops.linear_gelu(x.t, w.t, tensor(b), out=o, variant=variant), make_out,
                    {"x": x, "w": w, "bias": b})
    ref, bound = gelu_reference(x.t, w.t, tensor(b), dtype)
    ratio, acc = check_bound(kernel, out.view(1, 1, M, N), ref.view(1, 1, M, N), bound.view(1, 1, M, N))
    print(f"max err/bound {ratio:.4f} accumulation share {acc:.4f}")


def test_linear_gelu_matches_linear_then_gelu_kernel_bits(cuda_device):
    """The GELU epilogue computes the Linear's accumulator exactly as mvoc_linear does: gelu of the fp32 accumulator
    differs from gelu of the rounded Linear output only by that rounding."""
    from mvoc_b200 import ops

    torch.manual_seed(3)
    x = torch.randn(257 * 4, 1280, device=cuda_device).to(torch.bfloat16)
    w = (torch.randn(5120, 1280, device=cuda_device) * 1280 ** -0.5).to(torch.bfloat16)
    b = torch.randn(5120, device=cuda_device).to(torch.bfloat16)
    fused = ops.linear_gelu(x, w, b)
    two = F.gelu(ops.linear(x, w, b).float())
    assert rel_l2(fused, two) <= 2.0 ** -8


# ------------------------------------------------------------------ the full-width encoder
@pytest.fixture(scope="module")
def full_models(cuda_device):
    """(transformers fp32 model, product encoder in bf16) on the same random-init weights."""
    transformers = pytest.importorskip("transformers")
    from mvoc_b200.clip import CLIPVisionEncoder
    from mvoc_b200.unet3d import prepare

    torch.manual_seed(0)
    cfg = transformers.CLIPVisionConfig(hidden_act="gelu", layer_norm_eps=1e-5, **FULL)
    cfg._attn_implementation = "sdpa"
    with torch.device(cuda_device):
        ref = transformers.CLIPVisionModelWithProjection(cfg).eval().requires_grad_(False)
    ours = CLIPVisionEncoder().eval().requires_grad_(False)
    ours.load_state_dict({k: v.cpu() for k, v in ref.state_dict().items()}, strict=True)
    return ref, prepare(ours.to(cuda_device, torch.bfloat16))


@pytest.fixture()
def no_tf32():
    saved = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
    yield
    torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = saved


# Bars for image_embeds of the bf16 product against transformers fp32 (32 layers of bf16 activations): relative L2
# <= 2e-2 and cosine >= 0.999 per image.
ENC_REL_L2, ENC_COS = 2e-2, 0.999


@pytest.mark.parametrize("batch", [1, 64])
def test_encoder_full_width_vs_transformers(cuda_device, full_models, no_tf32, batch):
    ref, ours = full_models
    torch.manual_seed(batch)
    x = torch.randn(batch, 3, 224, 224, device=cuda_device)
    with torch.no_grad():
        want = ref(pixel_values=x).image_embeds
    got = ours(x)
    torch.cuda.synchronize()
    assert got.shape == want.shape == (batch, 1024) and got.dtype == torch.bfloat16
    err = rel_l2(got, want)
    cos = F.cosine_similarity(got.double(), want.double(), dim=-1)
    print(f"[clip image tower, batch {batch}] rel L2 {err:.4e}, min cosine {float(cos.min()):.6f}")
    assert err <= ENC_REL_L2 and float(cos.min()) >= ENC_COS


def test_encode_image_is_bit_invariant_to_chunk_size(cuda_device, full_models):
    from mvoc_b200.pipeline import I2VGenXLPipeline

    _, ours = full_models
    pipe = I2VGenXLPipeline(None, cuda_device, image_encoder=ours)
    torch.manual_seed(9)
    x = torch.randn(64, 3, 224, 224, device=cuda_device)
    outs = [pipe.encode_image(x, encode_chunk_size=c) for c in (64, 16, 5, 1)]
    torch.cuda.synchronize()
    assert outs[0].shape == (64, 1, 1024)
    for o in outs[1:]:
        assert torch.equal(o, outs[0])


# ------------------------------------------------------------------ the scripts
def _write_encoder(full_models, path):
    ref, _ = full_models
    torch.save({k: v.to("cpu", torch.bfloat16) for k, v in ref.state_dict().items()}, path)


def test_scripts_embeddings_equal_encode_image(cuda_device, full_models, tmp_path, monkeypatch):
    """inverse.py and composite.py with --synthetic --image_encoder_state_dict FILE: what reaches the step loops is
    encode_image of the entry's frames (inverse: the first frame; composite: [bg, objs, zeros, main] repeated over T)."""
    from PIL import Image

    from mvoc_b200 import composite, inverse
    from mvoc_b200.clip import clip_image_input
    from mvoc_b200.pipeline import I2VGenXLPipeline

    enc_path = str(tmp_path / "image_encoder.pt")
    _write_encoder(full_models, enc_path)
    T, w_px, h_px = 2, 128, 64
    g = torch.Generator().manual_seed(2)
    rnd = lambda: Image.fromarray(torch.randint(0, 256, (h_px, w_px, 3), generator=g, dtype=torch.uint8).numpy())

    # inversion: frames on disk, the first one is encoded
    seen = {}

    def record(self, latents, prompt_embeds, image_embeddings, image_latents, fps, **kw):
        seen.update(pipe=self, image_embeddings=image_embeddings.clone())
        return {}

    monkeypatch.setattr(I2VGenXLPipeline, "invert", record)
    data = tmp_path / "inv"
    frame_dir = data / "demo" / "clip"
    frame_dir.mkdir(parents=True)
    frames = [rnd() for _ in range(T)]
    for i, im in enumerate(frames):
        im.save(frame_dir / f"{i:03d}.png")
    cfg = data / "group.json"
    cfg.write_text(json.dumps([{"active": True, "force_recompute_latents": True, "video_name": "clip",
                                "data_dir": str(data), "image_size": [w_px, h_px], "n_frames": T}]))
    template = os.path.join(ROOT, "configs", "group_inversion", "template.yaml")
    assert inverse.main(template, str(cfg), synthetic_inputs=True, image_encoder_state_dict=enc_path) == 1
    pipe = seen["pipe"]
    want = pipe.encode_image(clip_image_input(frames[0], w_px))
    assert seen["image_embeddings"].shape == (1, 1, 1024)
    assert torch.equal(seen["image_embeddings"], want)

    # composition: control frames of two objects, the background as a directory
    got = {}

    def run_entry(pipe, config, device, conditioning=None, allow_synthetic=False):
        got.update(pipe=pipe, cond=conditioning, config=config)
        return torch.zeros(1, 4, T, h_px // 8, w_px // 8, device=device)

    monkeypatch.setattr(composite, "run_entry", run_entry)
    data = tmp_path / "comp"
    (data / "bg").mkdir(parents=True)
    imgs = [rnd() for _ in range(4)]
    imgs[0].save(data / "bg" / "000.png")
    for j in range(2):
        imgs[1 + j].save(data / f"obj{j}.png")
    imgs[3].save(data / "main.png")
    cfg = data / "group.json"
    cfg.write_text(json.dumps([{"active": True, "video_name": "clip", "edited_video_name": "clip_edit",
                                "data_dir": str(data), "image_size": [w_px, h_px], "n_frames": T,
                                "obj_mask_path": ["m0", "m1"], "obj_ddim_latents_path": ["l0", "l1"],
                                "edited_contorl_frame_path_background": "bg",
                                "edited_contorl_frame_path": ["obj0.png", "obj1.png"],
                                "edited_contorl_frame_path_main": "main.png", "output_dir": str(data / "out")}]))
    template = os.path.join(ROOT, "configs", "group_composite", "template.yaml")
    assert composite.main(template, str(cfg), synthetic_inputs=True, image_encoder_state_dict=enc_path,
                          max_entries=1) == 1
    emb = got["cond"]["image_embeddings"]
    assert emb.shape == (5, T, 1024)
    want = got["pipe"].encode_image(clip_image_input(imgs, w_px))[:, 0]        # bg, obj0, obj1, main
    for i, j in ((0, 0), (1, 1), (2, 2), (4, 3)):
        assert torch.equal(emb[i], want[j].expand(T, -1))
    assert not emb[3].any()
