"""AutoencoderKL decoder without a GPU: the diffusers key layout, the state-dict loader, the host layer against the
oracle (fp32, kernel wrappers replaced by torch emulations of their C-ABI contracts) and the frame export mapping."""
import copy
import os

import numpy as np
import pytest
import torch

TOL = 1e-5


def rel_l2(a, b):
    return float((a.float() - b.float()).norm() / b.float().norm())


def diffusers_state_dict(oracle_sd: dict) -> dict:
    """oracle.vae.DecoderKL's state dict under the names diffusers 0.27.2's AutoencoderKL writes."""
    out = {}
    for k, v in oracle_sd.items():
        if k.startswith("post_quant_conv."):
            nk = k
        elif k.startswith("mid_resnet1."):
            nk = "decoder.mid_block.resnets.0." + k[len("mid_resnet1."):]
        elif k.startswith("mid_resnet2."):
            nk = "decoder.mid_block.resnets.1." + k[len("mid_resnet2."):]
        elif k.startswith("mid_attn."):
            nk = "decoder.mid_block.attentions.0." + k[len("mid_attn."):]
        elif ".upsample." in k:
            nk = "decoder." + k.replace(".upsample.", ".upsamplers.0.conv.")
        else:
            nk = "decoder." + k
        out[nk] = v
    return out


def diffusers_decoder_keys(block_out_channels=(128, 256, 512, 512)):
    """The decoder-side keys of diffusers 0.27.2's AutoencoderKL.state_dict(), written out from its module tree."""
    wb = (".weight", ".bias")
    keys = ["post_quant_conv" + s for s in wb] + ["decoder.conv_in" + s for s in wb]

    def resnet(prefix, cin, cout):
        parts = ["norm1", "conv1", "norm2", "conv2"] + (["conv_shortcut"] if cin != cout else [])
        return [f"{prefix}.{p}{s}" for p in parts for s in wb]

    top = block_out_channels[-1]
    for i in range(2):
        keys += resnet(f"decoder.mid_block.resnets.{i}", top, top)
    keys += [f"decoder.mid_block.attentions.0.{p}{s}" for p in ("group_norm", "to_q", "to_k", "to_v", "to_out.0")
             for s in wb]
    rev = list(block_out_channels)[::-1]
    for i, cout in enumerate(rev):
        cin = rev[max(i - 1, 0)]
        for j in range(3):
            keys += resnet(f"decoder.up_blocks.{i}.resnets.{j}", cin if j == 0 else cout, cout)
        if i < len(rev) - 1:
            keys += [f"decoder.up_blocks.{i}.upsamplers.0.conv{s}" for s in wb]
    keys += ["decoder.conv_norm_out" + s for s in wb] + ["decoder.conv_out" + s for s in wb]
    return keys


def test_full_width_decoder_matches_diffusers_layout():
    from mvoc_b200.vae import AutoencoderKLDecoder
    from oracle import vae as ovae

    with torch.device("meta"):
        m = AutoencoderKLDecoder()
        o = ovae.DecoderKL()
    n_product = sum(p.numel() for p in m.parameters())
    assert n_product == sum(p.numel() for p in o.parameters()) == 49_490_179 + 4 * 4 + 4
    assert sorted(m.state_dict().keys()) == sorted(diffusers_decoder_keys())
    want = {k: tuple(v.shape) for k, v in diffusers_state_dict(o.state_dict()).items()}
    assert {k: tuple(v.shape) for k, v in m.state_dict().items()} == want


def _autoencoder_sd(seed=0):
    """A full-width random-init AutoencoderKL state dict: the decoder side plus encoder-side entries to ignore."""
    from oracle import vae as ovae

    sd = diffusers_state_dict(ovae.build_decoder(narrow=False, seed=seed).state_dict())
    sd["encoder.conv_in.weight"] = torch.randn(128, 3, 3, 3)
    sd["encoder.conv_in.bias"] = torch.randn(128)
    sd["quant_conv.weight"] = torch.randn(8, 8, 1, 1)
    sd["quant_conv.bias"] = torch.randn(8)
    return sd


@pytest.mark.parametrize("fmt", ["safetensors", "torch"])
def test_load_vae_decoder_round_trip(tmp_path, fmt):
    from safetensors.torch import save_file

    from mvoc_b200.vae import load_vae_decoder

    sd = _autoencoder_sd()
    path = str(tmp_path / ("vae.safetensors" if fmt == "safetensors" else "vae.pt"))
    if fmt == "safetensors":
        save_file({k: v.contiguous() for k, v in sd.items()}, path)
    else:
        torch.save(sd, path)
    m = load_vae_decoder(path, "cpu", dtype=torch.float32)
    got = m.state_dict()
    assert sorted(got) == sorted(k for k in sd if not k.startswith(("encoder.", "quant_conv.")))
    for k, v in got.items():
        assert v.dtype == torch.float32 and torch.equal(v, sd[k]), k
    assert not any(p.requires_grad for p in m.parameters())
    assert load_vae_decoder(path, "cpu").dtype == torch.bfloat16


def test_load_vae_decoder_names_the_bad_key(tmp_path):
    from mvoc_b200.vae import load_vae_decoder

    base = _autoencoder_sd()
    cases = []
    missing = dict(base)
    del missing["decoder.mid_block.attentions.0.to_k.bias"]
    cases.append((missing, KeyError, "decoder.mid_block.attentions.0.to_k.bias"))
    extra = dict(base)
    extra["decoder.mid_block.attentions.0.query.weight"] = torch.zeros(512, 512)   # pre-0.14 name: not mapped
    cases.append((extra, KeyError, "decoder.mid_block.attentions.0.query.weight"))
    shape = dict(base)
    shape["decoder.up_blocks.3.resnets.0.conv_shortcut.weight"] = torch.zeros(128, 256, 3, 3)
    cases.append((shape, ValueError, "decoder.up_blocks.3.resnets.0.conv_shortcut.weight"))
    for i, (sd, exc, key) in enumerate(cases):
        path = str(tmp_path / f"bad{i}.pt")
        torch.save(sd, path)
        with pytest.raises(exc, match=key.replace(".", r"\.")):
            load_vae_decoder(path, "cpu", dtype=torch.float32)
    with pytest.raises(FileNotFoundError):
        load_vae_decoder(str(tmp_path / "absent.safetensors"), "cpu")


# ------------------------------------------------------------------ host layer against the oracle
def attention_d512(q, k, v, scale=None, out=None):
    """Contract of mvoc_attn_d512_fwd: q, k, v [B, N, 512], contiguous last dim, 8-element-aligned strides."""
    for t in (q, k, v):
        assert t.dim() == 3 and t.shape == q.shape and t.shape[-1] == 512 and t.stride(-1) == 1
        assert all(s % 8 == 0 for s in t.stride()[:-1]), t.stride()
    scale = 512 ** -0.5 if scale is None else scale
    o = torch.softmax(q @ k.transpose(1, 2) * scale, dim=-1) @ v
    if out is not None:
        out.copy_(o)
        return out
    return o


@pytest.fixture()
def emulated_vae_ops():
    from mvoc_b200 import ops
    from tests import cpu_ops_emulation as emu

    saved = emu.install()
    saved_attn = ops.attention_d512
    ops.attention_d512 = attention_d512
    yield emu
    ops.attention_d512 = saved_attn
    emu.uninstall(saved)


def test_host_decoder_vs_oracle(emulated_vae_ops):
    """The product decoder's host layer (channels-last wiring, fused QKV with biases, residuals and shortcuts in the
    GEMM epilogues, decode_latents' chunking) in fp32 against oracle/vae.py.  Narrow lower levels keep it quick;
    the mid block stays 512 wide because the attention kernel is for D = 512 only."""
    from mvoc_b200.pipeline import I2VGenXLPipeline
    from mvoc_b200.vae import AutoencoderKLDecoder
    from oracle import vae as ovae

    widths = (32, 64, 128, 512)
    torch.manual_seed(3)
    oracle = ovae.DecoderKL(widths, groups=8).eval().requires_grad_(False)
    product = AutoencoderKLDecoder(widths, groups=8).eval().requires_grad_(False)
    product.load_state_dict(diffusers_state_dict(oracle.state_dict()), strict=True)
    torch.manual_seed(4)
    latents = torch.randn(1, 4, 3, 6, 10)
    ref = ovae.decode_latents(copy.deepcopy(oracle), latents, decode_chunk_size=2)
    pipe = I2VGenXLPipeline(None, "cpu", vae=product)
    out = pipe.decode_latents(latents, decode_chunk_size=2)
    assert out.shape == ref.shape == (1, 3, 3, 48, 80) and out.dtype == torch.float32
    assert rel_l2(out, ref) <= TOL, f"{rel_l2(out, ref):.3e}"
    for key in ("linear", "linear_res", "conv", "conv_res", "conv_shortcut"):
        assert emulated_vae_ops.calls[key] > 0, key


def test_decode_latents_needs_a_decoder():
    from mvoc_b200.pipeline import I2VGenXLPipeline

    with pytest.raises(RuntimeError, match="VAE"):
        I2VGenXLPipeline(None, "cpu").decode_latents(torch.zeros(1, 4, 1, 2, 2))


# ------------------------------------------------------------------ frame export
def test_frames_to_uint8_mapping():
    from mvoc_b200.vae import frames_to_uint8

    vals = [-1.0, 1.0, -3.0, 5.0, 0.0, 0.5, -0.5, 2 * 100.5 / 255 - 1, float("-inf")]
    want = [0, 255, 0, 255, 128, 191, 64, 100, 0]
    # 0 -> 127.5 and 100.5 / 255 * 255: halves go to the even neighbour, like numpy's round in the reference
    video = torch.tensor(vals).view(1, 1, 1, -1).expand(3, 2, 1, len(vals))
    got = frames_to_uint8(video)
    assert got.dtype == torch.uint8 and tuple(got.shape) == (2, 1, len(vals), 3)
    x = torch.tensor(vals, dtype=torch.float32)
    numpy_ref = ((x / 2 + 0.5).clamp(0, 1).numpy() * 255).round().astype("uint8")
    assert got[0, 0, :, 0].tolist() == numpy_ref.tolist() == want


def test_save_frames_writes_rgb_pngs(tmp_path):
    from PIL import Image

    from mvoc_b200.vae import frames_to_uint8, save_frames

    torch.manual_seed(0)
    video = torch.rand(3, 4, 6, 10) * 2.4 - 1.2
    paths = save_frames(video, str(tmp_path / "frames"))
    assert [os.path.basename(p) for p in paths] == ["000.png", "001.png", "002.png", "003.png"]
    u8 = frames_to_uint8(video)
    for i, p in enumerate(paths):
        img = Image.open(p)
        assert img.mode == "RGB" and img.size == (10, 6)
        assert torch.equal(torch.from_numpy(np.array(img)), u8[i])
