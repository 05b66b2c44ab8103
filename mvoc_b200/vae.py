"""AutoencoderKL, product side: frames -> latents (encoder) and latents -> frames (decoder) on the library's
kernels (bf16 on one B200).

The module trees and parameter names are those of diffusers 0.27.2's ``AutoencoderKL`` (the stabilityai/sd-vae
architecture i2vgen-xl ships), so one checkpoint's state dict feeds both loaders unchanged: ``quant_conv.*`` and
``encoder.{conv_in, down_blocks, mid_block, conv_norm_out, conv_out}.*`` for the encoder, ``post_quant_conv.*`` and
``decoder.{conv_in, mid_block, up_blocks, conv_norm_out, conv_out}.*`` for the decoder.  The reference runs the
decoder from ``decode_latents`` (pipelines/pipeline_i2vgen_xl.py:771-791) and the encoder from
``encode_vae_video`` (:893-920) and ``prepare_image_latents`` (:860-890).

Activations are channels-last ``[n, H, W, C]`` from conv_in to conv_out.  The resnets, GroupNorms and
upsamplers are the UNet's (``unet3d.ResnetBlock2D`` without a time embedding, ``GroupNormAct``, ``Upsample2D``):
3x3 convs on the tcgen05 implicit GEMM with the 1x1 shortcut and the residual in its epilogue, GroupNorm(+SiLU)
with statistics per frame.  The mid-block attention is one head of width 512: GroupNorm, one fused QKV GEMM with
the three biases, ``mvoc_attn_d512_fwd``, then ``to_out[0]`` with bias and the block's residual in the epilogue.
conv_in (4 input channels), conv_out (3 output channels) and the 1x1 post_quant_conv run on cuDNN through torch,
the same choice the UNet makes for its 4- and 8-channel convs.  The encoder is built from the same blocks; its three
stride-2 downsamplers run on ``mvoc_conv3x3_s2_nhwc``, and its conv_in (3 input channels), conv_out (8 output
channels) and 1x1 quant_conv on cuDNN.
"""
from __future__ import annotations

import os
from typing import Sequence

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import ops, unet3d
from .unet3d import GroupNormAct, ResnetBlock2D, Upsample2D, conv_nhwc, dense_linear, derived, prepare

SCALING_FACTOR = 0.18215   # AutoencoderKL.config.scaling_factor of the sd-vae checkpoints


class VAEAttention(nn.Module):
    """diffusers Attention as the VAE mid block builds it: one head over all C channels, GroupNorm on the input,
    biases on every projection, residual_connection=True, rescale_output_factor 1."""

    def __init__(self, channels: int, groups: int, eps: float = 1e-6):
        super().__init__()
        self.group_norm = GroupNormAct(groups, channels, eps=eps, affine=True)
        self.to_q = nn.Linear(channels, channels)
        self.to_k = nn.Linear(channels, channels)
        self.to_v = nn.Linear(channels, channels)
        self.to_out = nn.ModuleList([nn.Linear(channels, channels), nn.Dropout(0.0)])

    def forward(self, x):
        n, h, w, c = x.shape
        t = self.group_norm(x).view(n, h * w, c)
        ws = (self.to_q.weight, self.to_k.weight, self.to_v.weight)
        bs = (self.to_q.bias, self.to_k.bias, self.to_v.bias)
        w_qkv = derived(self, "w_qkv", ws, lambda: torch.cat(ws, dim=0).contiguous())
        b_qkv = derived(self, "b_qkv", bs, lambda: torch.cat(bs, dim=0).contiguous())
        qkv = dense_linear(t, w_qkv, b_qkv)
        a = ops.attention_d512(qkv[..., :c], qkv[..., c:2 * c], qkv[..., 2 * c:], scale=c ** -0.5)
        out = self.to_out[0]
        return dense_linear(a, out.weight, out.bias, x.view(n, h * w, c)).view(n, h, w, c)


class UNetMidBlock2D(nn.Module):
    def __init__(self, channels: int, groups: int, eps: float = 1e-6):
        super().__init__()
        self.attentions = nn.ModuleList([VAEAttention(channels, groups, eps)])
        self.resnets = nn.ModuleList([ResnetBlock2D(channels, channels, None, groups, eps) for _ in range(2)])

    def forward(self, x):
        x = self.resnets[0](x, None)
        return self.resnets[1](self.attentions[0](x), None)


class UpDecoderBlock2D(nn.Module):
    def __init__(self, in_channels: int, out_channels: int, groups: int, add_upsample: bool, eps: float = 1e-6,
                 num_layers: int = 3):
        super().__init__()
        self.resnets = nn.ModuleList([ResnetBlock2D(in_channels if i == 0 else out_channels, out_channels, None,
                                                    groups, eps) for i in range(num_layers)])
        self.upsamplers = nn.ModuleList([Upsample2D(out_channels)]) if add_upsample else None

    def forward(self, x):
        for r in self.resnets:
            x = r(x, None)
        if self.upsamplers is not None:
            x = self.upsamplers[0](x)
        return x


class Decoder(nn.Module):
    def __init__(self, block_out_channels: Sequence[int], groups: int, eps: float = 1e-6):
        super().__init__()
        c = list(block_out_channels)
        self.conv_in = nn.Conv2d(4, c[-1], 3, padding=1)
        self.mid_block = UNetMidBlock2D(c[-1], groups, eps)
        rev = c[::-1]
        self.up_blocks = nn.ModuleList([UpDecoderBlock2D(rev[max(i - 1, 0)], rev[i], groups, i < len(rev) - 1, eps)
                                        for i in range(len(rev))])
        self.conv_norm_out = GroupNormAct(groups, c[0], eps=eps, affine=True)
        self.conv_act = nn.SiLU()
        self.conv_out = nn.Conv2d(c[0], 3, 3, padding=1)

    def forward(self, x):
        """x [n, h, w, 4] channels-last -> [n, 8h, 8w, 3] channels-last."""
        x = self.mid_block(conv_nhwc(x, self.conv_in))
        for blk in self.up_blocks:
            x = blk(x)
        return conv_nhwc(self.conv_norm_out(x, silu=True), self.conv_out)


class AutoencoderKLDecoder(nn.Module):
    """post_quant_conv + decoder of AutoencoderKL; forward(z [n, 4, h, w]) -> images [n, 3, 8h, 8w] fp32."""

    def __init__(self, block_out_channels: Sequence[int] = (128, 256, 512, 512), groups: int = 32):
        super().__init__()
        self.post_quant_conv = nn.Conv2d(4, 4, 1)
        self.decoder = Decoder(block_out_channels, groups)

    @property
    def dtype(self):
        return self.decoder.conv_in.weight.dtype

    def forward(self, z):
        x = z.to(self.dtype).permute(0, 2, 3, 1).contiguous()
        y = self.decoder(conv_nhwc(x, self.post_quant_conv))
        return y.permute(0, 3, 1, 2).float()


# ------------------------------------------------------------------ encoder
class Downsample2D(nn.Module):
    """diffusers Downsample2D as the VAE encoder builds it (padding=0): F.pad (0, 1, 0, 1), then a 3x3 stride-2 conv
    without padding.  mvoc_conv3x3_s2_nhwc with pads (0, 1) where the GEMM kernels apply (unet3d._tc_ok); otherwise,
    MVOC_DENSE=lib included, the same two steps on cuDNN."""

    def __init__(self, channels: int):
        super().__init__()
        self.conv = nn.Conv2d(channels, channels, 3, stride=2, padding=0)

    def forward(self, x):
        conv = self.conv
        if unet3d._tc_ok(x, conv.in_channels, conv.out_channels):
            wt = derived(conv, "w_taps", (conv.weight,), lambda: ops.conv_taps(conv.weight))
            return ops.conv3x3_s2(x if x.is_contiguous() else x.contiguous(), wt, conv.bias, pad=(0, 1))
        y = F.conv2d(F.pad(x.permute(0, 3, 1, 2), (0, 1, 0, 1)), conv.weight, conv.bias, stride=2)
        return y.permute(0, 2, 3, 1).contiguous()


class DownEncoderBlock2D(nn.Module):
    def __init__(self, in_channels: int, out_channels: int, groups: int, add_downsample: bool, eps: float = 1e-6,
                 num_layers: int = 2):
        super().__init__()
        self.resnets = nn.ModuleList([ResnetBlock2D(in_channels if i == 0 else out_channels, out_channels, None,
                                                    groups, eps) for i in range(num_layers)])
        self.downsamplers = nn.ModuleList([Downsample2D(out_channels)]) if add_downsample else None

    def forward(self, x):
        for r in self.resnets:
            x = r(x, None)
        if self.downsamplers is not None:
            x = self.downsamplers[0](x)
        return x


class Encoder(nn.Module):
    def __init__(self, block_out_channels: Sequence[int], groups: int, eps: float = 1e-6):
        super().__init__()
        c = list(block_out_channels)
        self.conv_in = nn.Conv2d(3, c[0], 3, padding=1)
        self.down_blocks = nn.ModuleList([DownEncoderBlock2D(c[max(i - 1, 0)], c[i], groups, i < len(c) - 1, eps)
                                          for i in range(len(c))])
        self.mid_block = UNetMidBlock2D(c[-1], groups, eps)
        self.conv_norm_out = GroupNormAct(groups, c[-1], eps=eps, affine=True)
        self.conv_act = nn.SiLU()
        self.conv_out = nn.Conv2d(c[-1], 8, 3, padding=1)    # double_z: mean and logvar of 4 latent channels

    def forward(self, x):
        """x [n, H, W, 3] channels-last -> moments [n, H/8, W/8, 8] channels-last."""
        x = conv_nhwc(x, self.conv_in)
        for blk in self.down_blocks:
            x = blk(x)
        return conv_nhwc(self.conv_norm_out(self.mid_block(x), silu=True), self.conv_out)


class AutoencoderKLEncoder(nn.Module):
    """encoder + quant_conv of AutoencoderKL; forward(images [n, 3, H, W] in [-1, 1]) -> moments [n, 8, H/8, W/8]
    fp32 (mean and logvar of the latent posterior, see DiagonalGaussian)."""

    def __init__(self, block_out_channels: Sequence[int] = (128, 256, 512, 512), groups: int = 32):
        super().__init__()
        self.encoder = Encoder(block_out_channels, groups)
        self.quant_conv = nn.Conv2d(8, 8, 1)

    @property
    def dtype(self):
        return self.encoder.conv_in.weight.dtype

    def forward(self, images):
        x = images.to(self.dtype).permute(0, 2, 3, 1).contiguous()
        y = conv_nhwc(self.encoder(x), self.quant_conv)
        return y.permute(0, 3, 1, 2).float()


class DiagonalGaussian:
    """diffusers DiagonalGaussianDistribution of the encoder's moments [n, 8, h, w]: mean and logvar are the two
    channel halves, logvar clamped to [-30, 20], std = exp(logvar / 2).  The noise of `sample` is passed in, so a
    caller can draw it once for frames it encodes in several chunks."""

    def __init__(self, moments: torch.Tensor):
        self.mean, logvar = moments.float().chunk(2, dim=1)
        self.logvar = logvar.clamp(-30.0, 20.0)
        self.std = torch.exp(0.5 * self.logvar)

    def sample(self, noise: torch.Tensor) -> torch.Tensor:
        return self.mean + self.std * noise

    def mode(self) -> torch.Tensor:
        return self.mean


# ------------------------------------------------------------------ loaders
def _read_state_dict(path: str) -> dict:
    if path.endswith(".safetensors"):
        from safetensors.torch import load_file

        return load_file(path, device="cpu")
    return torch.load(path, map_location="cpu", weights_only=True)


def _load_part(path: str, model_cls, part: str, ignore: tuple, device, dtype, kind: str = "VAE"):
    """One side of a diffusers AutoencoderKL state dict (or another `kind` of checkpoint) into `model_cls()`: keys
    under `ignore` (the other side) are skipped; a missing or unexpected key, or a tensor of the wrong shape, raises an
    error that names it."""
    if not os.path.exists(path):
        raise FileNotFoundError(f"{kind} state dict {path!r} not found")
    sd = _read_state_dict(path)
    with torch.device("meta"):
        model = model_cls()
    want = model.state_dict()
    keep = {}
    for k, v in sd.items():
        if k.startswith(ignore):
            continue
        if k not in want:
            raise KeyError(f"{path}: unexpected {part} key {k!r}")
        if tuple(v.shape) != tuple(want[k].shape):
            raise ValueError(f"{path}: {k!r} has shape {tuple(v.shape)}, the {part} needs {tuple(want[k].shape)}")
        keep[k] = v
    missing = [k for k in want if k not in keep]
    if missing:
        raise KeyError(f"{path}: missing {part} key {missing[0]!r} ({len(missing)} missing)")
    model.load_state_dict(keep, strict=True, assign=True)
    model = model.to(device=device, dtype=dtype).eval().requires_grad_(False)
    return prepare(model)


def load_vae_decoder(path: str, device, dtype=torch.bfloat16) -> AutoencoderKLDecoder:
    """AutoencoderKL decoder from a diffusers ``AutoencoderKL`` state dict (``.safetensors`` or a torch file).
    ``decoder.*`` and ``post_quant_conv.*`` are loaded, ``encoder.*`` and ``quant_conv.*`` ignored; a missing or
    unexpected decoder key, or a tensor of the wrong shape, raises an error that names it.  Only the key names of
    diffusers >= 0.14 are accepted (``to_q`` / ``to_k`` / ``to_v`` / ``to_out.0``)."""
    return _load_part(path, AutoencoderKLDecoder, "decoder", ("encoder.", "quant_conv."), device, dtype)


def load_vae_encoder(path: str, device, dtype=torch.bfloat16) -> AutoencoderKLEncoder:
    """AutoencoderKL encoder from the same state dict as load_vae_decoder: ``encoder.*`` and ``quant_conv.*`` are
    loaded, ``decoder.*`` and ``post_quant_conv.*`` ignored, with the same key and shape checks."""
    return _load_part(path, AutoencoderKLEncoder, "encoder", ("decoder.", "post_quant_conv."), device, dtype)


# ------------------------------------------------------------------ frames in
def center_crop_wide(image, resolution):
    """The reference's _center_crop_wide (pipelines/pipeline_i2vgen_xl.py:2054) on one PIL image: resize by the
    smaller of the two width / height ratios so the image covers `resolution` = (width, height), then crop the
    centre.  The BOX filter is that of diffusers 0.27.2."""
    from PIL import Image

    scale = min(image.size[0] / resolution[0], image.size[1] / resolution[1])
    image = image.resize((round(image.width // scale), round(image.height // scale)), resample=Image.BOX)
    x1 = (image.width - resolution[0]) // 2
    y1 = (image.height - resolution[1]) // 2
    return image.crop((x1, y1, x1 + resolution[0], y1 + resolution[1]))


def pil_to_model_input(images) -> torch.Tensor:
    """One PIL image or a list of them (same size) -> [n, 3, H, W] fp32 in [-1, 1]: uint8 x -> x / 127.5 - 1."""
    import numpy as np

    images = images if isinstance(images, (list, tuple)) else [images]
    a = np.stack([np.asarray(im.convert("RGB"), dtype=np.float32) for im in images])
    return torch.from_numpy(a).permute(0, 3, 1, 2).contiguous() / 127.5 - 1.0


FRAME_EXTENSIONS = (".png", ".jpg", ".jpeg")


def load_frames(frame_dir: str, n_frames: int, image_size) -> torch.Tensor:
    """The first `n_frames` image files of `frame_dir` (.png / .jpg, sorted by name), each through center_crop_wide
    to `image_size` = (width, height) -> [n_frames, 3, height, width] fp32 in [-1, 1]."""
    from PIL import Image

    if not os.path.isdir(frame_dir):
        raise FileNotFoundError(f"frame directory {frame_dir!r} not found")
    names = sorted(n for n in os.listdir(frame_dir) if n.lower().endswith(FRAME_EXTENSIONS))
    if len(names) < n_frames:
        raise FileNotFoundError(f"{frame_dir!r} holds {len(names)} frames (.png / .jpg), {n_frames} are needed")
    frames = []
    for n in names[:n_frames]:
        with Image.open(os.path.join(frame_dir, n)) as im:
            frames.append(center_crop_wide(im.convert("RGB"), tuple(image_size)))
    return pil_to_model_input(frames)


def frames_to_uint8(video: torch.Tensor) -> torch.Tensor:
    """[3, T, H, W] decoded video in [-1, 1] -> uint8 [T, H, W, 3], the mapping of the reference's tensor2vid /
    VaeImageProcessor.postprocess: round(clamp(x / 2 + 0.5, 0, 1) * 255), halves to even (numpy's round)."""
    x = (video.detach().float().cpu() / 2 + 0.5).clamp(0, 1)
    return (x * 255).round().to(torch.uint8).permute(1, 2, 3, 0).contiguous()


def save_frames(video: torch.Tensor, out_dir: str, first_index: int = 0) -> list:
    """One RGB PNG per frame of a [3, T, H, W] video: out_dir/000.png, 001.png, ...  The files are numbered from
    `first_index`, so that a slice of a longer video keeps its frames' numbers."""
    from PIL import Image

    os.makedirs(out_dir, exist_ok=True)
    paths = []
    for i, frame in enumerate(frames_to_uint8(video).numpy()):
        p = os.path.join(out_dir, f"{first_index + i:03d}.png")
        Image.fromarray(frame).save(p)
        paths.append(p)
    return paths
