"""AutoencoderKL encoder on the GPU: the stride-2 convolution kernel against fp32 torch (edges checked on their own),
the whole encoder against the fp32 oracle inside the torch-bf16 envelope, chunked encoding and the inversion
script's --vae_state_dict path."""
import json
import os

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GEMM_BAR = 5e-3


def rel_l2(a, b):
    a, b = a.float().cpu(), b.float().cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-20))


@pytest.fixture()
def no_tf32():
    saved = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
    yield
    torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = saved


# ------------------------------------------------------------------ mvoc_conv3x3_s2_nhwc
S2_SHAPES = [
    # N, H, W, Cin, Cout: the encoder's three downsamplers (+ config 5's first level), an odd shape, and the UNet's
    # three downsamplers at config 2 (the first two need tail column tiles)
    (2, 512, 512, 128, 128), (2, 256, 256, 256, 256), (2, 128, 128, 512, 512), (1, 704, 1280, 128, 128),
    (3, 45, 77, 64, 192),
    (5, 64, 64, 320, 320), (5, 32, 32, 640, 640), (5, 16, 16, 1280, 1280),
]
VARIANTS = {"single_cta": 0, "pair": 1, "narrow64": 64 << 8}


@pytest.mark.parametrize("variant", list(VARIANTS))
@pytest.mark.parametrize("shape", S2_SHAPES, ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("pad", [(0, 1), (1, 1)], ids=["pad01", "pad11"])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
def test_conv3x3_s2_vs_fp32(cuda_device, no_tf32, dtype, pad, shape, variant):
    from mvoc_b200 import ops

    N, H, W, ci, co = shape
    torch.manual_seed(H + W + ci)
    x = torch.randn(N, H, W, ci, device=cuda_device).to(dtype)
    w = (torch.randn(co, ci, 3, 3, device=cuda_device) * (9 * ci) ** -0.5).to(dtype)
    b = torch.randn(co, device=cuda_device).to(dtype)
    out = ops.conv3x3_s2(x, ops.conv_taps(w), b, pad=pad, variant=VARIANTS[variant])
    ref = F.conv2d(F.pad(x.permute(0, 3, 1, 2).float(), (pad[0], pad[1], pad[0], pad[1])), w.float(), b.float(),
                   stride=2).permute(0, 2, 3, 1)
    torch.cuda.synchronize()
    Ho, Wo = ((n + pad[0] + pad[1] - 3) // 2 + 1 for n in (H, W))
    assert out.shape == ref.shape == (N, Ho, Wo, co) and out.dtype == dtype
    err = rel_l2(out, ref)
    assert err <= GEMM_BAR, f"rel L2 {err:.3e}"
    # padding errors sit on the first / last output row and column, where the whole-tensor error would hide them
    for name, sl in (("top", (slice(None), 0)), ("bottom", (slice(None), -1)),
                     ("left", (slice(None), slice(None), 0)), ("right", (slice(None), slice(None), -1))):
        e = rel_l2(out[sl], ref[sl])
        assert e <= GEMM_BAR, f"{name} edge rel L2 {e:.3e}"


def test_conv3x3_s2_error_codes(cuda_device):
    from mvoc_b200 import _cabi, ops

    x = torch.zeros(1, 8, 8, 64, device=cuda_device, dtype=torch.bfloat16)
    wt = torch.zeros(9, 64, 64, device=cuda_device, dtype=torch.bfloat16)
    with pytest.raises(ValueError, match="pad"):
        ops.conv3x3_s2(x, wt, pad=(2, 0))
    with pytest.raises(ValueError, match="w_taps"):
        ops.conv3x3_s2(x, wt[:, :, :32].contiguous())
    with pytest.raises(_cabi.MvocError, match="mvoc_conv3x3_s2_nhwc"):
        ops.conv3x3_s2(torch.zeros(1, 8, 8, 96, device=cuda_device, dtype=torch.bfloat16),
                       torch.zeros(9, 64, 96, device=cuda_device, dtype=torch.bfloat16))


# ------------------------------------------------------------------ whole encoder
@pytest.fixture(scope="module")
def full_encoders(cuda_device):
    """(fp32 oracle on the GPU, product encoder in bf16) with the same random-init weights."""
    from mvoc_b200.unet3d import prepare
    from mvoc_b200.vae import AutoencoderKLEncoder
    from oracle import vae_encoder as oenc
    from tests.test_vae_encode_cpu import diffusers_encoder_state_dict

    oracle = oenc.build_encoder(narrow=False, seed=0)
    product = AutoencoderKLEncoder().eval().requires_grad_(False)
    product.load_state_dict(diffusers_encoder_state_dict(oracle.state_dict()), strict=True)
    product = prepare(product.to(cuda_device, torch.bfloat16))
    return oracle.to(cuda_device), product


def test_encoder_full_width_vs_oracle(cuda_device, full_encoders, no_tf32):
    """Full-width encoder, 2 frames of 192 x 320 (960 attention tokens): bf16 product moments against the fp32
    oracle, inside 1.5x the error of the oracle's own module tree run in bf16 on torch kernels."""
    import copy

    oracle, product = full_encoders
    torch.manual_seed(5)
    images = torch.rand(2, 3, 192, 320, device=cuda_device) * 2 - 1
    with torch.no_grad():
        ref = oracle(images)
        ov16 = copy.deepcopy(oracle).to(torch.bfloat16).to(memory_format=torch.channels_last)
        env = ov16(images.to(torch.bfloat16).contiguous(memory_format=torch.channels_last)).float()
    del ov16
    env_err = rel_l2(env, ref)
    out = product(images)
    torch.cuda.synchronize()
    assert out.shape == ref.shape == (2, 8, 24, 40) and out.dtype == torch.float32
    err = rel_l2(out, ref)
    print(f"[vae encoder 2x192x320] rel L2 {err:.4e} (torch bf16 envelope {env_err:.4e})")
    assert err <= 1.5 * env_err, f"rel L2 {err:.3e} > 1.5 x envelope {env_err:.3e}"


def test_encode_chunk_size_does_not_change_latents(cuda_device, full_encoders):
    from mvoc_b200.pipeline import I2VGenXLPipeline

    _, product = full_encoders
    pipe = I2VGenXLPipeline(None, cuda_device, vae_encoder=product)
    torch.manual_seed(6)
    frames = torch.rand(5, 3, 128, 192, device=cuda_device) * 2 - 1
    outs = [pipe.encode_vae_video(frames, torch.Generator().manual_seed(3), encode_chunk_size=c) for c in (1, 2, 5)]
    torch.cuda.synchronize()
    assert outs[0].shape == (1, 4, 5, 16, 24)
    assert rel_l2(outs[0], outs[2]) <= 1e-3 and rel_l2(outs[1], outs[2]) <= 1e-3


# ------------------------------------------------------------------ the script
def _write_vae(path):
    from oracle import vae_encoder as oenc
    from tests.test_vae_encode_cpu import diffusers_encoder_state_dict

    torch.save(diffusers_encoder_state_dict(oenc.build_encoder(narrow=False, seed=1).state_dict()), path)


def test_inverse_script_encodes_frames(cuda_device, tmp_path, monkeypatch):
    """--synthetic --vae_state_dict FILE writes the expected ddim_latents_{t}.pt files; with frames on disk the
    latents handed to invert are encode_vae_video of those frames under the entry's seed; without the flag invert
    receives the synthetic inputs it received before the flag existed."""
    from PIL import Image

    from mvoc_b200 import inverse, synthetic
    from mvoc_b200.pipeline import I2VGenXLPipeline, ddim_latents_filename
    from mvoc_b200.scheduler import DDIMSchedule
    from mvoc_b200.vae import load_frames

    vae_path = str(tmp_path / "vae.pt")
    _write_vae(vae_path)
    T, w_px, h_px = 2, 128, 64
    template = os.path.join(ROOT, "configs", "group_inversion", "template.yaml")

    def entry(run):
        data = tmp_path / run
        data.mkdir()
        cfg = data / "group.json"
        cfg.write_text(json.dumps([{"active": True, "force_recompute_latents": True, "video_name": "clip",
                                    "data_dir": str(data), "image_size": [w_px, h_px], "n_frames": T}]))
        return data, str(cfg)

    # 1. synthetic frames, real inversion of two steps
    data, cfg = entry("synthetic")
    torch.manual_seed(0)
    assert inverse.main(template, cfg, synthetic_inputs=True, vae_state_dict=vae_path, max_steps=2) == 1
    out_dir = data / "inversions" / "i2vgen-xl" / "clip" / "ddim_latents"
    want = sorted(ddim_latents_filename(t) for t in DDIMSchedule(500, inverse=True).timesteps[:2])
    assert sorted(os.listdir(out_dir)) == want
    for n in want:
        x = torch.load(out_dir / n)
        assert x.shape == (1, 4, T, h_px // 8, w_px // 8) and x.dtype == torch.float16 and torch.isfinite(x).all()

    # 2. frames on disk: what invert receives
    seen = {}

    def record(self, latents, prompt_embeds, image_embeddings, image_latents, fps, **kw):
        seen.update(pipe=self, latents=latents.clone(), image_latents=image_latents.clone())
        return {}

    monkeypatch.setattr(I2VGenXLPipeline, "invert", record)
    data, cfg = entry("frames")
    frame_dir = data / "demo" / "clip"
    frame_dir.mkdir(parents=True)
    g = torch.Generator().manual_seed(2)
    for i in range(T + 1):
        a = torch.randint(0, 256, (h_px, w_px, 3), generator=g, dtype=torch.uint8).numpy()
        Image.fromarray(a).save(frame_dir / f"{i:03d}.png")
    assert inverse.main(template, cfg, synthetic_inputs=True, vae_state_dict=vae_path) == 1
    frames = load_frames(str(frame_dir), T, (w_px, h_px)).to(cuda_device)
    gen = torch.Generator().manual_seed(8888)                                 # the template's seed
    want_lat = seen["pipe"].encode_vae_video(frames, gen)
    want_il = seen["pipe"].prepare_image_latents(frames[:1], T, gen)
    assert torch.equal(seen["latents"], want_lat)
    assert torch.equal(seen["image_latents"], want_il.to(seen["image_latents"].dtype))

    # 3. without the flag: the synthetic inputs, unchanged
    seen.clear()
    data, cfg = entry("plain")
    assert inverse.main(template, cfg, synthetic_inputs=True) == 1
    src = synthetic.make_inversion_inputs(
        synthetic.Workload("clip", "full", T, h_px // 8, w_px // 8, 0, inversion_steps=500), 0)
    assert seen["pipe"].vae_encoder is None
    assert torch.equal(seen["latents"].cpu(), src["latents"].float())
    assert torch.equal(seen["image_latents"].cpu(), src["image_latents"].to(seen["image_latents"].dtype))
