"""AutoencoderKL encoder without a GPU: the diffusers key layout, both loaders on one AutoencoderKL file, the host
layer against the oracle (fp32, kernel wrappers replaced by torch emulations of their C-ABI contracts), the
posterior, prepare_image_latents against the reference's own output, and the argument checks of the stride-2
convolution entry."""
import copy
import os

import pytest
import torch
import torch.nn.functional as F

from tests.test_vae_cpu import attention_d512, diffusers_state_dict, rel_l2

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOL = 1e-5


def diffusers_encoder_state_dict(oracle_sd: dict) -> dict:
    """oracle.vae_encoder.EncoderKL's state dict under the names diffusers 0.27.2's AutoencoderKL writes."""
    out = {}
    for k, v in oracle_sd.items():
        if k.startswith("quant_conv."):
            nk = k
        elif k.startswith("mid_resnet1."):
            nk = "encoder.mid_block.resnets.0." + k[len("mid_resnet1."):]
        elif k.startswith("mid_resnet2."):
            nk = "encoder.mid_block.resnets.1." + k[len("mid_resnet2."):]
        elif k.startswith("mid_attn."):
            nk = "encoder.mid_block.attentions.0." + k[len("mid_attn."):]
        elif ".downsample." in k:
            nk = "encoder." + k.replace(".downsample.", ".downsamplers.0.")
        else:
            nk = "encoder." + k
        out[nk] = v
    return out


def diffusers_encoder_keys(block_out_channels=(128, 256, 512, 512)):
    """The encoder-side keys of diffusers 0.27.2's AutoencoderKL.state_dict(), written out from its module tree."""
    wb = (".weight", ".bias")
    keys = ["encoder.conv_in" + s for s in wb]

    def resnet(prefix, cin, cout):
        parts = ["norm1", "conv1", "norm2", "conv2"] + (["conv_shortcut"] if cin != cout else [])
        return [f"{prefix}.{p}{s}" for p in parts for s in wb]

    c = list(block_out_channels)
    for i, cout in enumerate(c):
        cin = c[max(i - 1, 0)]
        for j in range(2):
            keys += resnet(f"encoder.down_blocks.{i}.resnets.{j}", cin if j == 0 else cout, cout)
        if i < len(c) - 1:
            keys += [f"encoder.down_blocks.{i}.downsamplers.0.conv{s}" for s in wb]
    for i in range(2):
        keys += resnet(f"encoder.mid_block.resnets.{i}", c[-1], c[-1])
    keys += [f"encoder.mid_block.attentions.0.{p}{s}" for p in ("group_norm", "to_q", "to_k", "to_v", "to_out.0")
             for s in wb]
    keys += ["encoder.conv_norm_out" + s for s in wb] + ["encoder.conv_out" + s for s in wb]
    keys += ["quant_conv" + s for s in wb]
    return keys


def test_full_width_encoder_matches_diffusers_layout():
    from mvoc_b200.vae import AutoencoderKLDecoder, AutoencoderKLEncoder
    from oracle import vae_encoder as oenc

    with torch.device("meta"):
        m = AutoencoderKLEncoder()
        o = oenc.EncoderKL()
        d = AutoencoderKLDecoder()
    n = sum(p.numel() for p in m.parameters())
    assert n == sum(p.numel() for p in o.parameters()) == 34_163_664
    assert n + sum(p.numel() for p in d.parameters()) == 83_653_863          # the published AutoencoderKL total
    assert sorted(m.state_dict().keys()) == sorted(diffusers_encoder_keys())
    want = {k: tuple(v.shape) for k, v in diffusers_encoder_state_dict(o.state_dict()).items()}
    assert {k: tuple(v.shape) for k, v in m.state_dict().items()} == want


def _autoencoder_sd(seed=0):
    """A full-width random-init AutoencoderKL state dict: encoder and decoder sides."""
    from oracle import vae as ovae
    from oracle import vae_encoder as oenc

    sd = diffusers_state_dict(ovae.build_decoder(narrow=False, seed=seed).state_dict())
    sd.update(diffusers_encoder_state_dict(oenc.build_encoder(narrow=False, seed=seed + 1).state_dict()))
    return sd


@pytest.fixture(scope="module")
def autoencoder_files(tmp_path_factory):
    from safetensors.torch import save_file

    sd = _autoencoder_sd()
    d = tmp_path_factory.mktemp("vae")
    paths = {"safetensors": str(d / "vae.safetensors"), "torch": str(d / "vae.pt")}
    save_file({k: v.contiguous() for k, v in sd.items()}, paths["safetensors"])
    torch.save(sd, paths["torch"])
    return sd, paths


@pytest.mark.parametrize("fmt", ["safetensors", "torch"])
def test_both_loaders_read_one_autoencoder_file(autoencoder_files, fmt):
    from mvoc_b200.vae import load_vae_decoder, load_vae_encoder

    sd, paths = autoencoder_files
    enc = load_vae_encoder(paths[fmt], "cpu", dtype=torch.float32)
    dec = load_vae_decoder(paths[fmt], "cpu", dtype=torch.float32)
    for m, prefixes in ((enc, ("encoder.", "quant_conv.")), (dec, ("decoder.", "post_quant_conv."))):
        got = m.state_dict()
        assert sorted(got) == sorted(k for k in sd if k.startswith(prefixes))
        for k, v in got.items():
            assert v.dtype == torch.float32 and torch.equal(v, sd[k]), k
        assert not any(p.requires_grad for p in m.parameters())
    assert load_vae_encoder(paths[fmt], "cpu").dtype == torch.bfloat16


def test_load_vae_encoder_names_the_bad_key(autoencoder_files, tmp_path):
    from mvoc_b200.vae import load_vae_encoder

    base = autoencoder_files[0]
    cases = []
    missing = dict(base)
    del missing["encoder.down_blocks.1.downsamplers.0.conv.bias"]
    cases.append((missing, KeyError, "encoder.down_blocks.1.downsamplers.0.conv.bias"))
    extra = dict(base)
    extra["encoder.down_blocks.3.downsamplers.0.conv.weight"] = torch.zeros(512, 512, 3, 3)   # the last block has none
    cases.append((extra, KeyError, "encoder.down_blocks.3.downsamplers.0.conv.weight"))
    shape = dict(base)
    shape["quant_conv.weight"] = torch.zeros(4, 8, 1, 1)
    cases.append((shape, ValueError, "quant_conv.weight"))
    for i, (sd, exc, key) in enumerate(cases):
        path = str(tmp_path / f"bad{i}.pt")
        torch.save(sd, path)
        with pytest.raises(exc, match=key.replace(".", r"\.")):
            load_vae_encoder(path, "cpu", dtype=torch.float32)
    with pytest.raises(FileNotFoundError):
        load_vae_encoder(str(tmp_path / "absent.safetensors"), "cpu")


# ------------------------------------------------------------------ host layer against the oracle
def conv3x3_s2(x, w_taps, bias=None, pad=(0, 1), out=None, variant=None):
    """Contract of mvoc_conv3x3_s2_nhwc: contiguous channels-last x, w_taps [9, Cout, Cin], 64-aligned channels,
    pads (zeros before, zeros after) each 0 or 1."""
    co, ci = w_taps.shape[1], w_taps.shape[2]
    assert co % 64 == 0 and ci % 64 == 0 and x.dim() == 4 and x.is_contiguous() and w_taps.is_contiguous()
    assert tuple(pad) in ((0, 1), (1, 1), (0, 0), (1, 0))
    w = w_taps.view(3, 3, co, ci).permute(2, 3, 0, 1)
    xp = F.pad(x.permute(0, 3, 1, 2), (pad[0], pad[1], pad[0], pad[1]))
    conv3x3_s2.calls += 1
    return F.conv2d(xp, w, bias, stride=2).permute(0, 2, 3, 1).contiguous()


@pytest.fixture()
def emulated_encoder_ops():
    from mvoc_b200 import ops
    from tests import cpu_ops_emulation as emu

    saved = emu.install()
    saved_ops = (ops.attention_d512, getattr(ops, "conv3x3_s2"))
    ops.attention_d512, ops.conv3x3_s2 = attention_d512, conv3x3_s2
    conv3x3_s2.calls = 0
    yield emu
    ops.attention_d512, ops.conv3x3_s2 = saved_ops
    emu.uninstall(saved)


def _narrow_pair(seed=3):
    """(oracle, product) encoders with the same weights: narrow lower levels, a 512-wide mid block (the attention
    kernel is for D = 512 only)."""
    from mvoc_b200.vae import AutoencoderKLEncoder
    from oracle import vae_encoder as oenc

    widths = (64, 128, 192, 512)
    torch.manual_seed(seed)
    oracle = oenc.EncoderKL(widths, groups=8).eval().requires_grad_(False)
    product = AutoencoderKLEncoder(widths, groups=8).eval().requires_grad_(False)
    product.load_state_dict(diffusers_encoder_state_dict(oracle.state_dict()), strict=True)
    return oracle, product


def test_host_encoder_vs_oracle(emulated_encoder_ops):
    """The product encoder's host layer (channels-last wiring, stride-2 downsamplers with the pad on the right and
    bottom, shortcuts and residuals in the GEMM epilogues, the fused QKV mid block) in fp32 against the oracle, at
    40 x 72 px: every level below the first has an odd extent (5 x 9 at the bottom)."""
    oracle, product = _narrow_pair()
    torch.manual_seed(4)
    images = torch.rand(2, 3, 40, 72) * 2 - 1
    ref = copy.deepcopy(oracle)(images)
    out = product(images)
    assert out.shape == ref.shape == (2, 8, 5, 9) and out.dtype == torch.float32
    assert rel_l2(out, ref) <= TOL, f"{rel_l2(out, ref):.3e}"
    assert conv3x3_s2.calls == 3
    for key in ("linear", "linear_res", "conv", "conv_res", "conv_shortcut"):
        assert emulated_encoder_ops.calls[key] > 0, key


def test_downsampler_without_kernels_is_pad_then_conv():
    """The cuDNN branch (MVOC_DENSE=lib, or channels the kernel cannot take): F.pad (0, 1, 0, 1) + stride-2 conv."""
    from mvoc_b200.vae import Downsample2D

    torch.manual_seed(0)
    m = Downsample2D(8)
    x = torch.randn(2, 7, 10, 8)
    ref = F.conv2d(F.pad(x.permute(0, 3, 1, 2), (0, 1, 0, 1)), m.conv.weight, m.conv.bias, stride=2)
    assert torch.allclose(m(x), ref.permute(0, 2, 3, 1), atol=1e-6) and m(x).shape == (2, 3, 5, 8)


# ------------------------------------------------------------------ posterior
def test_posterior_clamps_logvar():
    from mvoc_b200.vae import DiagonalGaussian

    mean = torch.randn(1, 4, 2, 3)
    logvar = torch.tensor([-50.0, -30.0, 0.0, 20.0, 40.0, 1.5]).view(1, 1, 2, 3).expand(1, 4, 2, 3)
    post = DiagonalGaussian(torch.cat([mean, logvar], dim=1))
    want = logvar.clamp(-30, 20)
    assert torch.equal(post.logvar, want) and torch.equal(post.mode(), mean)
    assert torch.allclose(post.std, torch.exp(0.5 * want))
    eps = torch.randn(1, 4, 2, 3)
    assert torch.equal(post.sample(eps), mean + torch.exp(0.5 * want) * eps)


def test_sample_does_not_depend_on_the_chunk_size():
    """The posterior noise is one draw for all frames: chunk sizes 1, 2 and T give bit-identical latents.  The
    encoder is a per-frame stand-in (a CPU convolution's rounding may depend on the batch it runs in)."""
    from mvoc_b200.pipeline import I2VGenXLPipeline
    from mvoc_b200.vae import SCALING_FACTOR, DiagonalGaussian

    def product(x):
        p = F.avg_pool2d(x.float(), 8)
        return torch.cat([p, p.flip(1), -p[:, :2]], dim=1)      # 8 channels: mean and logvar of 4

    pipe = I2VGenXLPipeline(None, "cpu", vae_encoder=product)
    torch.manual_seed(6)
    frames = torch.rand(3, 3, 16, 24) * 2 - 1
    outs = [pipe.encode_vae_video(frames, torch.Generator().manual_seed(11), encode_chunk_size=c) for c in (1, 2, 3)]
    assert outs[0].shape == (1, 4, 3, 2, 3) and outs[0].dtype == torch.float32
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[0], outs[2])
    post = DiagonalGaussian(product(frames))
    eps = torch.randn((3, 4, 2, 3), generator=torch.Generator().manual_seed(11))
    assert torch.equal(outs[2][0].permute(1, 0, 2, 3), post.sample(eps) * SCALING_FACTOR)


def test_encoding_needs_an_encoder():
    from mvoc_b200.pipeline import I2VGenXLPipeline

    with pytest.raises(RuntimeError, match="VAE encoder"):
        I2VGenXLPipeline(None, "cpu").encode_vae_video(torch.zeros(1, 3, 8, 8))


# ------------------------------------------------------------------ pinned against the reference
def test_prepare_image_latents_matches_reference_golden():
    """The first frame of the golden inversion fixture through center_crop_wide -> pil_to_model_input ->
    prepare_image_latents, with the golden generator's VAE double in place of the encoder, equals the image latents
    the reference's own prepare_image_latents produced (tests/golden/inversion_loop_tiny4.pt)."""
    from mvoc_b200.pipeline import I2VGenXLPipeline
    from mvoc_b200.vae import SCALING_FACTOR, center_crop_wide, pil_to_model_input
    from tests.golden import spec

    fx = spec.inversion_fixture()
    golden = torch.load(os.path.join(ROOT, "tests", "golden", "inversion_loop_tiny4.pt"))["seam"]["image_latents"]
    pil = spec.loop_images(fx)["main"][0]
    image = pil_to_model_input(center_crop_wide(pil, (fx["W"] * 8, fx["H"] * 8)))

    def vae_double(images, generator=None, encode_chunk_size=4):
        # make_golden_loops.FakeVAE: average pooling, the channel mean as the fourth channel, x3; the double's
        # latent_dist.sample() returns that tensor, which the reference then scales
        p = F.avg_pool2d(images.float(), 8)
        return torch.cat([p, p.mean(1, keepdim=True)], dim=1) * 3.0 * SCALING_FACTOR

    pipe = I2VGenXLPipeline(None, "cpu")
    pipe._vae_latents = vae_double
    got = pipe.prepare_image_latents(image, fx["T"], torch.Generator().manual_seed(0))
    assert got.shape == golden.shape == (1, 4, fx["T"], fx["H"], fx["W"])
    assert float((got - golden.float()).abs().max()) <= 1e-6


def test_center_crop_wide_covers_then_crops():
    from PIL import Image

    from mvoc_b200.vae import center_crop_wide, pil_to_model_input

    img = Image.new("RGB", (300, 100), (255, 0, 0))
    out = center_crop_wide(img, (128, 64))
    assert out.size == (128, 64)
    x = pil_to_model_input([out, out])
    assert x.shape == (2, 3, 64, 128) and x.dtype == torch.float32
    assert torch.equal(x[:, 0], torch.ones(2, 64, 128)) and torch.equal(x[:, 1], -torch.ones(2, 64, 128))


def test_load_frames_sorted_and_counted(tmp_path):
    from PIL import Image

    from mvoc_b200.vae import load_frames

    for i, name in enumerate(["b.png", "a.jpg", "c.png", "notes.txt"]):
        if name.endswith("txt"):
            (tmp_path / name).write_text("x")
        else:
            Image.new("RGB", (32, 16), (10 * i, 0, 0)).save(tmp_path / name)
    x = load_frames(str(tmp_path), 2, (32, 16))
    assert x.shape == (2, 3, 16, 32)
    assert x[0, 0, 0, 0] == pytest.approx(10 / 127.5 - 1, abs=0.02) and x[1, 0, 0, 0] == pytest.approx(-1.0)
    with pytest.raises(FileNotFoundError, match=r"3 frames.*4 are needed"):
        load_frames(str(tmp_path), 4, (32, 16))


# ------------------------------------------------------------------ C-ABI argument checks
def test_conv3x3_s2_entry_rejects_bad_arguments():
    """Checked before any CUDA call (this machine may have no GPU): codes and the named entry point."""
    from mvoc_b200 import _cabi

    lib = _cabi.load()

    def call(x=16, w=16, bias=None, out=16, N=1, H=8, W=8, ci=64, co=64, pb=0, pe=1, dtype=0):
        rc = lib.mvoc_conv3x3_s2_nhwc(x, w, bias, out, N, H, W, ci, co, pb, pe, dtype, 0, None)
        return rc, lib.mvoc_last_error().decode()

    for kw, code, text in [(dict(ci=48), -2, "K=48"), (dict(co=96), -2, "N=96"), (dict(pb=2), -1, "pad_begin=2"),
                           (dict(pe=-1), -1, "pad_end=-1"), (dict(H=2, pb=0, pe=0), -1, "empty output"),
                           (dict(W=1, pb=0, pe=1), -1, "empty output"), (dict(x=None), -1, "non-null"),
                           (dict(w=24), -1, "aligned"), (dict(out=None), -1, "non-null"),
                           (dict(bias=8), -1, "aligned"), (dict(N=0), -1, "empty problem"), (dict(dtype=2), -2, "dtype")]:
        rc, msg = call(**kw)
        assert rc == code and "mvoc_conv3x3_s2_nhwc" in msg and text in msg, (kw, rc, msg)


def test_conv3x3_s2_wrapper_checks_shapes():
    from mvoc_b200 import ops

    x = torch.zeros(1, 8, 8, 64)
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.conv3x3_s2(x, torch.zeros(9, 64, 64))


# ------------------------------------------------------------------ the script
def test_inverse_without_frames_names_the_directory(tmp_path, monkeypatch):
    """--vae_state_dict without --synthetic: a missing <video_dir>/<video_name>/ is an error that names it."""
    import json

    from mvoc_b200 import inverse, unet3d, vae

    monkeypatch.setattr(unet3d.UNetConfig, "full", staticmethod(unet3d.UNetConfig.tiny4))
    unet = unet3d.I2VGenXLUNet(unet3d.UNetConfig.tiny4())
    unet_path = str(tmp_path / "unet.pt")
    torch.save(unet.state_dict(), unet_path)
    monkeypatch.setattr(vae, "load_vae_encoder", lambda path, device: _narrow_pair()[1])
    inputs = str(tmp_path / "inputs.pt")
    torch.save({"prompt_embeds": torch.zeros(1, 77, 1024), "image_embeddings": torch.zeros(1, 1, 1024)}, inputs)
    cfg = tmp_path / "group.json"
    cfg.write_text(json.dumps([{"active": True, "video_name": "clip", "data_dir": str(tmp_path),
                                "force_recompute_latents": True, "n_frames": 2, "image_size": [64, 32]}]))
    template = os.path.join(ROOT, "configs", "group_inversion", "template.yaml")
    with pytest.raises(FileNotFoundError, match=str(tmp_path / "demo" / "clip")):
        inverse.main(template, str(cfg), unet_state_dict=unet_path, inputs=inputs, device="cpu",
                     vae_state_dict="unused.safetensors")
