"""ORACLE — test infrastructure only (never imported by mvoc_b200/).

Encoder side of diffusers 0.27.2 ``AutoencoderKL`` restated in fp32, next to the decoder of oracle/vae.py and
built from the same resnet and mid-block attention.  Random-init (seeded): there is no checkpoint here.

Layout: conv_in(3->C0) -> 4 down blocks of 2 resnets with channels C0, C1, C2, C3 (+ a downsampler after all but
the last: F.pad (0, 1, 0, 1), then Conv2d(3, stride 2, no padding)) -> mid (resnet, 1-head attention, resnet) ->
GroupNorm -> SiLU -> conv_out(C3->8) -> quant_conv(8->8, 1x1).  The output is the posterior's moments: mean and
logvar of 4 latent channels.  The real model has (C0..C3) = (128, 256, 512, 512); tests use a narrow one.
"""
from __future__ import annotations

from typing import Sequence

import torch
import torch.nn as nn
import torch.nn.functional as F

from .vae import _MidAttention, _Resnet


class _Downsample(nn.Module):
    def __init__(self, c: int):
        super().__init__()
        self.conv = nn.Conv2d(c, c, 3, stride=2, padding=0)

    def forward(self, x):
        return self.conv(F.pad(x, (0, 1, 0, 1)))


class _DownBlock(nn.Module):
    def __init__(self, cin: int, cout: int, groups: int, downsample: bool):
        super().__init__()
        self.resnets = nn.ModuleList([_Resnet(cin if i == 0 else cout, cout, groups) for i in range(2)])
        self.downsample = _Downsample(cout) if downsample else None

    def forward(self, x):
        for r in self.resnets:
            x = r(x)
        return x if self.downsample is None else self.downsample(x)


class EncoderKL(nn.Module):
    def __init__(self, block_out_channels: Sequence[int] = (128, 256, 512, 512), groups: int = 32):
        super().__init__()
        c = list(block_out_channels)
        self.conv_in = nn.Conv2d(3, c[0], 3, padding=1)
        self.down_blocks = nn.ModuleList(
            [_DownBlock(c[max(i - 1, 0)], c[i], groups, downsample=i < len(c) - 1) for i in range(len(c))])
        self.mid_resnet1 = _Resnet(c[-1], c[-1], groups)
        self.mid_attn = _MidAttention(c[-1], groups)
        self.mid_resnet2 = _Resnet(c[-1], c[-1], groups)
        self.conv_norm_out = nn.GroupNorm(groups, c[-1], eps=1e-6)
        self.conv_out = nn.Conv2d(c[-1], 8, 3, padding=1)
        self.quant_conv = nn.Conv2d(8, 8, 1)

    def forward(self, images):
        """images [n, 3, H, W] -> moments [n, 8, h, w]."""
        x = self.conv_in(images)
        for blk in self.down_blocks:
            x = blk(x)
        x = self.mid_resnet2(self.mid_attn(self.mid_resnet1(x)))
        return self.quant_conv(self.conv_out(F.silu(self.conv_norm_out(x))))


def build_encoder(narrow: bool = True, seed: int = 0) -> EncoderKL:
    torch.manual_seed(seed)
    m = EncoderKL((32, 64, 128, 128), groups=8) if narrow else EncoderKL()
    return m.eval().requires_grad_(False)
