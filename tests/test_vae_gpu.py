"""AutoencoderKL decoder on the GPU: the head_dim-512 attention kernel, GroupNorm at the decoder's shapes, the
whole decoder against the fp32 oracle inside the torch-bf16 envelope, chunked decoding and the script's frame
output."""
import json
import os

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def rel_l2(a, b):
    a, b = a.float().cpu(), b.float().cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-20))


def _attn_ref(q, k, v, scale):
    """fp32 attention, one batch at a time (the score matrix of N = 14080 is 0.8 GB)."""
    return torch.stack([torch.softmax((qb.float() @ kb.float().t()) * scale, dim=-1) @ vb.float()
                        for qb, kb, vb in zip(q, k, v)])


# ------------------------------------------------------------------ mvoc_attn_d512_fwd
@pytest.mark.parametrize("N", [1, 100, 1024, 2880, 4096, 14080])
@pytest.mark.parametrize("B", [1, 3])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
def test_attention_d512_fused_qkv_vs_fp32(cuda_device, dtype, B, N):
    """q, k, v are the column slices of one fused [B*N, 1536] projection output, as the decoder calls it."""
    from mvoc_b200 import ops

    torch.manual_seed(N + B)
    qkv = torch.randn(B, N, 3 * 512, device=cuda_device).to(dtype)
    q, k, v = qkv[..., :512], qkv[..., 512:1024], qkv[..., 1024:]
    out = ops.attention_d512(q, k, v)
    torch.cuda.synchronize()
    ref = _attn_ref(q, k, v, 512 ** -0.5)
    err = rel_l2(out, ref)
    assert out.shape == (B, N, 512) and out.dtype == dtype
    assert err <= 1e-2, f"rel L2 {err:.3e}"


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
def test_attention_d512_contiguous_peaked_and_strided_out(cuda_device, dtype):
    """Separate contiguous q / k / v, logits large enough that the running maximum is rescaled, and an output
    written into a column slice of a wider buffer."""
    from mvoc_b200 import ops

    torch.manual_seed(7)
    B, N = 2, 2500
    q = (6.0 * torch.randn(B, N, 512, device=cuda_device)).to(dtype)
    k = torch.randn(B, N, 512, device=cuda_device).to(dtype)
    v = torch.randn(B, N, 512, device=cuda_device).to(dtype)
    wide = torch.zeros(B, N, 1024, device=cuda_device, dtype=dtype)
    out = ops.attention_d512(q, k, v, out=wide[..., 256:768])
    torch.cuda.synchronize()
    assert rel_l2(out, _attn_ref(q, k, v, 512 ** -0.5)) <= 1e-2
    assert not wide[..., :256].any() and not wide[..., 768:].any()


def test_attention_d512_error_codes(cuda_device):
    from mvoc_b200 import _cabi, ops

    lib = _cabi.load()
    B, N = 1, 256
    buf = torch.zeros(B * N * 1536 + 64, device=cuda_device, dtype=torch.bfloat16)
    o = torch.empty(B * N * 1536, device=cuda_device, dtype=torch.bfloat16)
    p = buf.data_ptr()
    st = [N * 1536, 1536] * 4

    def call(ptr=p, D=512, strides=st):
        return lib.mvoc_attn_d512_fwd(ptr, ptr + 1024, ptr + 2048, o.data_ptr(), B, N, D, *strides, 1.0,
                                      _cabi.MVOC_BF16, None)

    assert call() == 0
    torch.cuda.synchronize()
    assert call(D=256) == -2 and "512" in lib.mvoc_last_error().decode()
    assert call(D=64) == -2
    assert call(ptr=p + 2) == -1 and "aligned" in lib.mvoc_last_error().decode()
    assert call(strides=[N * 1536, 1540] + st[2:]) == -2
    assert call(strides=st[:6] + [N * 1536 + 4, 1536]) == -2
    with pytest.raises(ValueError):
        ops.attention_d512(*(torch.zeros(1, 8, 256, device=cuda_device, dtype=torch.bfloat16),) * 3)
    with pytest.raises(RuntimeError):
        ops.attention_d512(*(torch.zeros(1, 8, 512, dtype=torch.bfloat16),) * 3)


# ------------------------------------------------------------------ GroupNorm at the decoder's shapes
GN_DECODER_CASES = [
    # N, C, H, W, silu: 4 channels per group at C = 128 (G = 32), up to the 704 x 1280 level of config 5
    (4, 512, 64, 64, False),     # mid-block attention norm
    (2, 512, 88, 160, True),
    (2, 256, 352, 640, True),
    (1, 128, 704, 1280, True),
    (3, 128, 512, 512, True),
    (2, 256, 40, 72, True),
]


@pytest.mark.parametrize("N,C,H,W,silu", GN_DECODER_CASES)
def test_groupnorm_nhwc_decoder_shapes(cuda_device, N, C, H, W, silu):
    from mvoc_b200 import ops

    torch.manual_seed(C + H)
    x = (torch.randn(N, H, W, C, device=cuda_device) * 2.0 + 0.7).bfloat16()
    wgt = (1.0 + 0.2 * torch.randn(C, device=cuda_device)).bfloat16()
    bias = (0.1 * torch.randn(C, device=cuda_device)).bfloat16()
    out = ops.groupnorm_nhwc(x, wgt, bias, 32, 1e-6, silu)
    ref = F.group_norm(x.permute(0, 3, 1, 2).float(), 32, wgt.float(), bias.float(), 1e-6)
    ref = F.silu(ref) if silu else ref
    torch.cuda.synchronize()
    err = float((out.permute(0, 3, 1, 2).float() - ref).norm() / ref.norm())
    assert err <= 3e-3, f"rel L2 {err:.3e}"


# ------------------------------------------------------------------ whole decoder
@pytest.fixture(scope="module")
def full_decoders(cuda_device):
    """(fp32 oracle on the GPU, product decoder in bf16) with the same random-init weights."""
    from mvoc_b200.vae import AutoencoderKLDecoder
    from mvoc_b200.unet3d import prepare
    from oracle import vae as ovae
    from tests.test_vae_cpu import diffusers_state_dict

    oracle = ovae.build_decoder(narrow=False, seed=0)
    product = AutoencoderKLDecoder().eval().requires_grad_(False)
    product.load_state_dict(diffusers_state_dict(oracle.state_dict()), strict=True)
    product = prepare(product.to(cuda_device, torch.bfloat16))
    return oracle.to(cuda_device), product


def test_decoder_full_width_vs_oracle(cuda_device, full_decoders):
    """Full-width decoder, 2 frames of 24 x 40 latents (960 attention tokens: ragged and non-square): bf16 product
    against the fp32 oracle, inside 1.5x the error of the oracle's own module tree run in bf16 on torch kernels."""
    import copy

    from mvoc_b200.pipeline import I2VGenXLPipeline
    from oracle import vae as ovae

    oracle, product = full_decoders
    torch.manual_seed(5)
    latents = torch.randn(1, 4, 2, 24, 40, device=cuda_device)
    tf32 = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
    try:
        ref = ovae.decode_latents(oracle, latents)
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = tf32
    ov16 = copy.deepcopy(oracle).to(torch.bfloat16).to(memory_format=torch.channels_last)
    with torch.no_grad():
        env = ovae.decode_latents(lambda z: ov16(z.to(torch.bfloat16)).float(), latents)
    del ov16
    env_err = rel_l2(env, ref)
    out = I2VGenXLPipeline(None, cuda_device, vae=product).decode_latents(latents)
    torch.cuda.synchronize()
    assert out.shape == ref.shape == (1, 3, 2, 192, 320)
    err = rel_l2(out, ref)
    db, db_env = ovae.psnr(out, ref), ovae.psnr(env, ref)
    print(f"[vae decoder 2x24x40] rel L2 {err:.4e} (torch bf16 envelope {env_err:.4e}); "
          f"PSNR {db:.2f} dB (envelope {db_env:.2f} dB)")
    assert err <= 1.5 * env_err, f"rel L2 {err:.3e} > 1.5 x envelope {env_err:.3e}"


def test_decode_chunk_size_does_not_change_frames(cuda_device, full_decoders):
    from mvoc_b200.pipeline import I2VGenXLPipeline

    _, product = full_decoders
    pipe = I2VGenXLPipeline(None, cuda_device, vae=product)
    torch.manual_seed(6)
    latents = torch.randn(1, 4, 5, 16, 24, device=cuda_device)
    outs = [pipe.decode_latents(latents, decode_chunk_size=c) for c in (1, 2, 5)]
    torch.cuda.synchronize()
    assert rel_l2(outs[0], outs[2]) <= 1e-3 and rel_l2(outs[1], outs[2]) <= 1e-3


# ------------------------------------------------------------------ the script
def test_composite_script_writes_frames(cuda_device, tmp_path):
    """`--synthetic --vae_state_dict FILE --max_entries 1` writes T PNGs of 8h x 8w; the latents file is
    byte-identical to that of a run without the flag."""
    from PIL import Image

    from mvoc_b200 import composite
    from oracle import vae as ovae
    from tests.test_vae_cpu import diffusers_state_dict

    vae_path = str(tmp_path / "vae.pt")
    torch.save(diffusers_state_dict(ovae.build_decoder(narrow=False, seed=1).state_dict()), vae_path)
    T, h, w = 2, 8, 16
    entry = {"active": True, "video_name": "tiny", "edited_video_name": "tiny edit", "image_size": [8 * w, 8 * h],
             "n_frames": T, "n_steps": 2, "ddim_init_latents_t_idx": 0, "fusion_step": [0, 1],
             "obj_mask_path": ["demo/tiny/obj1_mask"], "obj_ddim_latents_path": ["inversions/obj1/ddim_latents"],
             "bg_ddim_latents_path": "inversions/tiny/ddim_latents"}
    template = os.path.join(ROOT, "configs", "group_composite", "template.yaml")
    files = {}
    for run, vae in (("plain", None), ("vae", vae_path)):
        data = tmp_path / run
        data.mkdir()
        cfg = data / "group.json"
        cfg.write_text(json.dumps([dict(entry, data_dir=str(data))]))
        torch.manual_seed(0)         # the UNet is random-initialised from the global generator
        assert composite.main(template, str(cfg), synthetic_inputs=True, vae_state_dict=vae, max_entries=1) == 1
        out_dir = data / "Results" / "MVOC-B200" / "i2vgen-xl" / "tiny" / "tiny edit"
        files[run] = (out_dir / "composite_latents.synthetic.pt").read_bytes()
        frames_dir = out_dir / "composite_frames.synthetic"
        if vae is None:
            assert not frames_dir.exists()
            continue
        names = sorted(os.listdir(frames_dir))
        assert names == [f"{i:03d}.png" for i in range(T)]
        for n in names:
            img = Image.open(frames_dir / n)
            assert img.mode == "RGB" and img.size == (8 * w, 8 * h)
    assert files["plain"] == files["vae"]
