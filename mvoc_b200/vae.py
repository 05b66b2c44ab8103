"""AutoencoderKL decoder, product side: latents -> frames on the library's kernels (bf16 on one B200).

The module tree and parameter names are those of the decoder side of diffusers 0.27.2's ``AutoencoderKL`` (the
stabilityai/sd-vae architecture i2vgen-xl ships), so a checkpoint's state dict loads unchanged:
``post_quant_conv.*`` and ``decoder.{conv_in, mid_block, up_blocks, conv_norm_out, conv_out}.*``.  The reference
runs it from ``decode_latents`` (pipelines/pipeline_i2vgen_xl.py:771-791).

Activations are channels-last ``[n, H, W, C]`` from conv_in to conv_out.  The resnets, GroupNorms and
upsamplers are the UNet's (``unet3d.ResnetBlock2D`` without a time embedding, ``GroupNormAct``, ``Upsample2D``):
3x3 convs on the tcgen05 implicit GEMM with the 1x1 shortcut and the residual in its epilogue, GroupNorm(+SiLU)
with statistics per frame.  The mid-block attention is one head of width 512: GroupNorm, one fused QKV GEMM with
the three biases, ``mvoc_attn_d512_fwd``, then ``to_out[0]`` with bias and the block's residual in the epilogue.
conv_in (4 input channels), conv_out (3 output channels) and the 1x1 post_quant_conv run on cuDNN through torch,
the same choice the UNet makes for its 4- and 8-channel convs.
"""
from __future__ import annotations

import os
from typing import Sequence

import torch
import torch.nn as nn

from . import ops
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


def _read_state_dict(path: str) -> dict:
    if path.endswith(".safetensors"):
        from safetensors.torch import load_file

        return load_file(path, device="cpu")
    return torch.load(path, map_location="cpu", weights_only=True)


def load_vae_decoder(path: str, device, dtype=torch.bfloat16) -> AutoencoderKLDecoder:
    """AutoencoderKL decoder from a diffusers ``AutoencoderKL`` state dict (``.safetensors`` or a torch file).
    ``decoder.*`` and ``post_quant_conv.*`` are loaded, ``encoder.*`` and ``quant_conv.*`` ignored; a missing or
    unexpected decoder key, or a tensor of the wrong shape, raises an error that names it.  Only the key names of
    diffusers >= 0.14 are accepted (``to_q`` / ``to_k`` / ``to_v`` / ``to_out.0``)."""
    if not os.path.exists(path):
        raise FileNotFoundError(f"VAE state dict {path!r} not found")
    sd = _read_state_dict(path)
    with torch.device("meta"):
        model = AutoencoderKLDecoder()
    want = model.state_dict()
    keep = {}
    for k, v in sd.items():
        if k.startswith(("encoder.", "quant_conv.")):
            continue
        if k not in want:
            raise KeyError(f"{path}: unexpected decoder key {k!r}")
        if tuple(v.shape) != tuple(want[k].shape):
            raise ValueError(f"{path}: {k!r} has shape {tuple(v.shape)}, the decoder needs {tuple(want[k].shape)}")
        keep[k] = v
    missing = [k for k in want if k not in keep]
    if missing:
        raise KeyError(f"{path}: missing decoder key {missing[0]!r} ({len(missing)} missing)")
    model.load_state_dict(keep, strict=True, assign=True)
    model = model.to(device=device, dtype=dtype).eval().requires_grad_(False)
    return prepare(model)


def frames_to_uint8(video: torch.Tensor) -> torch.Tensor:
    """[3, T, H, W] decoded video in [-1, 1] -> uint8 [T, H, W, 3], the mapping of the reference's tensor2vid /
    VaeImageProcessor.postprocess: round(clamp(x / 2 + 0.5, 0, 1) * 255), halves to even (numpy's round)."""
    x = (video.detach().float().cpu() / 2 + 0.5).clamp(0, 1)
    return (x * 255).round().to(torch.uint8).permute(1, 2, 3, 0).contiguous()


def save_frames(video: torch.Tensor, out_dir: str) -> list:
    """One RGB PNG per frame of a [3, T, H, W] video: out_dir/000.png, 001.png, ..."""
    from PIL import Image

    os.makedirs(out_dir, exist_ok=True)
    paths = []
    for i, frame in enumerate(frames_to_uint8(video).numpy()):
        p = os.path.join(out_dir, f"{i:03d}.png")
        Image.fromarray(frame).save(p)
        paths.append(p)
    return paths
