"""CLIP image tower, product side: frames -> image embeddings on the library's kernels (bf16 on one B200).

The module tree and parameter names are those of transformers' ``CLIPVisionModelWithProjection`` (the reference's
``image_encoder/`` folder, a ViT-H/14: 32 layers, width 1280, 16 heads of 80, 257 tokens, projection 1024), so its
state dict loads unchanged.  The reference calls it from ``I2VGenXLPipeline._encode_image`` for every branch and
frame of a composition (pipelines/pipeline_i2vgen_xl.py:1391-1541) and once for the first frame of an inversion.

Per encoder layer: ``mvoc_layernorm``, one fused q/k/v ``mvoc_linear`` (1280 -> 3840, the three biases in its
epilogue), ``mvoc_attn_d80_fwd`` on the three column slices, ``out_proj`` with the residual in the epilogue,
``mvoc_layernorm``, ``mlp.fc1`` with the exact GELU in the epilogue (``mvoc_linear_gelu``), ``mlp.fc2`` with the
residual in the epilogue.  The 14x14 stride-14 patch convolution does not overlap: the patches are a host reshape and
the convolution one ``mvoc_linear`` with K = 3*14*14 = 588 zero-padded to 640 (the weight once, the patches per call).
The class token and the position embedding are two torch adds; ``pre_layrnorm`` and ``post_layernorm`` (on the pooled
CLS token only) are ``mvoc_layernorm``, and ``visual_projection`` (no bias) is ``mvoc_linear``.  ``image_embeds`` is
not L2-normalised.  Nothing on this path goes to cuDNN or cuBLAS.
"""
from __future__ import annotations

from dataclasses import dataclass

import torch
import torch.nn as nn

from . import ops
from .unet3d import derived

CLIP_MEAN = (0.48145466, 0.4578275, 0.40821073)
CLIP_STD = (0.26862954, 0.26130258, 0.27577711)
K_ALIGN = 64   # the tcgen05 GEMM's K granularity


@dataclass
class CLIPVisionConfig:
    """The reference checkpoint's CLIPVisionConfig (image_encoder/config.json of i2vgen-xl); LayerNorm eps 1e-5 and the
    erf GELU (hidden_act "gelu") are fixed."""
    hidden_size: int = 1280
    intermediate_size: int = 5120
    num_hidden_layers: int = 32
    num_attention_heads: int = 16
    patch_size: int = 14
    image_size: int = 224
    projection_dim: int = 1024
    num_channels: int = 3
    layer_norm_eps: float = 1e-5

    @property
    def num_patches(self) -> int:
        return (self.image_size // self.patch_size) ** 2


class CLIPVisionEmbeddings(nn.Module):
    def __init__(self, cfg: CLIPVisionConfig):
        super().__init__()
        self.cfg = cfg
        self.class_embedding = nn.Parameter(torch.empty(cfg.hidden_size))
        self.patch_embedding = nn.Conv2d(cfg.num_channels, cfg.hidden_size, cfg.patch_size, cfg.patch_size, bias=False)
        self.position_embedding = nn.Embedding(cfg.num_patches + 1, cfg.hidden_size)

    def forward(self, pixel_values: torch.Tensor) -> torch.Tensor:
        cfg = self.cfg
        n, c, hh, ww = pixel_values.shape
        p = cfg.patch_size
        if (hh, ww) != (cfg.image_size, cfg.image_size) or c != cfg.num_channels:
            raise ValueError(f"CLIP image tower: pixel_values must be [n, {cfg.num_channels}, {cfg.image_size}, "
                             f"{cfg.image_size}], got {tuple(pixel_values.shape)}")
        w = self.patch_embedding.weight
        k = c * p * p
        kp = -(-k // K_ALIGN) * K_ALIGN
        w_pad = derived(self, "w_patch", (w,), lambda: nn.functional.pad(w.reshape(w.shape[0], k), (0, kp - k)))
        gh, gw = hh // p, ww // p
        # [n, c, gh, p, gw, p] -> rows (image, patch row, patch col), columns (channel, ky, kx): Conv2d's weight order
        patches = torch.zeros((n, gh * gw, kp), dtype=w.dtype, device=w.device)
        patches[..., :k] = pixel_values.reshape(n, c, gh, p, gw, p).permute(0, 2, 4, 1, 3, 5).reshape(n, gh * gw, k)
        emb = ops.linear(patches, w_pad)
        cls = self.class_embedding.to(emb.dtype).expand(n, 1, -1)
        return torch.cat([cls, emb], dim=1) + self.position_embedding.weight


class CLIPAttention(nn.Module):
    """Self-attention of both CLIP towers: dense at head_dim 80 (image) or causal at head_dim 64 (text, `causal`)."""

    def __init__(self, cfg, causal: bool = False):
        super().__init__()
        d = cfg.hidden_size
        self.heads = cfg.num_attention_heads
        self.head_dim = d // self.heads
        self.causal = causal
        self.k_proj = nn.Linear(d, d)
        self.v_proj = nn.Linear(d, d)
        self.q_proj = nn.Linear(d, d)
        self.out_proj = nn.Linear(d, d)

    def forward(self, h: torch.Tensor, residual: torch.Tensor) -> torch.Tensor:
        d = h.shape[-1]
        ws = (self.q_proj.weight, self.k_proj.weight, self.v_proj.weight)
        bs = (self.q_proj.bias, self.k_proj.bias, self.v_proj.bias)
        w_qkv = derived(self, "w_qkv", ws, lambda: torch.cat(ws, dim=0).contiguous())
        b_qkv = derived(self, "b_qkv", bs, lambda: torch.cat(bs, dim=0).contiguous())
        qkv = ops.linear(h, w_qkv, b_qkv)
        attend = ops.attention_causal if self.causal else ops.attention_d80
        a = attend(qkv[..., :d], qkv[..., d:2 * d], qkv[..., 2 * d:], self.heads, scale=self.head_dim ** -0.5)
        return ops.linear(a, self.out_proj.weight, self.out_proj.bias, residual)


class CLIPMLP(nn.Module):
    def __init__(self, cfg):
        super().__init__()
        self.fc1 = nn.Linear(cfg.hidden_size, cfg.intermediate_size)
        self.fc2 = nn.Linear(cfg.intermediate_size, cfg.hidden_size)

    def forward(self, h: torch.Tensor, residual: torch.Tensor) -> torch.Tensor:
        return ops.linear(ops.linear_gelu(h, self.fc1.weight, self.fc1.bias), self.fc2.weight, self.fc2.bias, residual)


def _layernorm(ln: nn.LayerNorm, x: torch.Tensor) -> torch.Tensor:
    return ops.layernorm(x.contiguous(), ln.weight, ln.bias, ln.eps)


class CLIPEncoderLayer(nn.Module):
    def __init__(self, cfg, causal: bool = False):
        super().__init__()
        self.self_attn = CLIPAttention(cfg, causal)
        self.layer_norm1 = nn.LayerNorm(cfg.hidden_size, eps=cfg.layer_norm_eps)
        self.mlp = CLIPMLP(cfg)
        self.layer_norm2 = nn.LayerNorm(cfg.hidden_size, eps=cfg.layer_norm_eps)

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        x = self.self_attn(_layernorm(self.layer_norm1, x), x)
        return self.mlp(_layernorm(self.layer_norm2, x), x)


class CLIPEncoder(nn.Module):
    def __init__(self, cfg, causal: bool = False):
        super().__init__()
        self.layers = nn.ModuleList([CLIPEncoderLayer(cfg, causal) for _ in range(cfg.num_hidden_layers)])


class CLIPVisionTransformer(nn.Module):
    def __init__(self, cfg: CLIPVisionConfig):
        super().__init__()
        self.embeddings = CLIPVisionEmbeddings(cfg)
        self.pre_layrnorm = nn.LayerNorm(cfg.hidden_size, eps=cfg.layer_norm_eps)   # transformers' spelling
        self.encoder = CLIPEncoder(cfg)
        self.post_layernorm = nn.LayerNorm(cfg.hidden_size, eps=cfg.layer_norm_eps)


class CLIPVisionEncoder(nn.Module):
    """transformers' CLIPVisionModelWithProjection (same module tree and state-dict names): pixel_values
    [n, 3, 224, 224] (CLIP-normalised, see clip_image_input) -> image_embeds [n, projection_dim] in the weights' dtype."""

    def __init__(self, cfg: CLIPVisionConfig = None):
        super().__init__()
        self.cfg = cfg or CLIPVisionConfig()
        self.vision_model = CLIPVisionTransformer(self.cfg)
        self.visual_projection = nn.Linear(self.cfg.hidden_size, self.cfg.projection_dim, bias=False)

    @property
    def dtype(self):
        return self.visual_projection.weight.dtype

    def forward(self, pixel_values: torch.Tensor) -> torch.Tensor:
        vm = self.vision_model
        x = vm.embeddings(pixel_values.to(self.dtype))
        x = _layernorm(vm.pre_layrnorm, x)
        for layer in vm.encoder.layers:
            x = layer(x)
        pooled = _layernorm(vm.post_layernorm, x[:, 0])   # post_layernorm on the CLS token only
        return ops.linear(pooled, self.visual_projection.weight)


# keys of a full CLIPModel / older transformers checkpoints that the image tower does not use
_IGNORED = ("text_model.", "text_projection.", "logit_scale", "vision_model.embeddings.position_ids")


def load_clip_image_encoder(path: str, device, dtype=torch.bfloat16, cfg: CLIPVisionConfig = None) -> CLIPVisionEncoder:
    """CLIP image tower from a transformers ``CLIPVisionModelWithProjection`` state dict (``.safetensors`` or a torch
    file): ``vision_model.*`` and ``visual_projection.weight``.  The text tower's keys and the position_ids buffer of
    older checkpoints are ignored; a missing or unexpected key, or a tensor of the wrong shape, raises an error that
    names it.  `cfg` defaults to the reference checkpoint's configuration."""
    from .vae import _load_part

    return _load_part(path, lambda: CLIPVisionEncoder(cfg), "CLIP image encoder", _IGNORED, device, dtype,
                      kind="CLIP image encoder")


def clip_image_input(images, width: int, size: int = 224) -> torch.Tensor:
    """The image preprocessing of diffusers 0.27.2's I2VGenXLPipeline (``__call__`` step 3.2.1, ``_encode_image``):
    each PIL image is centre-cropped by ``_center_crop_wide`` to (width, width) (BOX resize, centre crop), resized by
    ``_resize_bilinear`` to the feature extractor's crop size (size x size, PIL BILINEAR), scaled to [0, 1]
    (``pil_to_numpy``) and normalised with the CLIP mean and std (CLIPImageProcessor with do_resize, do_center_crop
    and do_rescale False).  One PIL image or a list -> [n, 3, size, size] fp32."""
    import numpy as np
    from PIL import Image

    from .vae import center_crop_wide

    images = images if isinstance(images, (list, tuple)) else [images]
    arrs = []
    for im in images:
        im = center_crop_wide(im.convert("RGB"), (width, width)).resize((size, size), resample=Image.BILINEAR)
        arrs.append(np.asarray(im, dtype=np.float32) / 255.0)
    x = torch.from_numpy(np.stack(arrs)).permute(0, 3, 1, 2).contiguous()
    mean = torch.tensor(CLIP_MEAN).view(1, 3, 1, 1)
    std = torch.tensor(CLIP_STD).view(1, 3, 1, 1)
    return (x - mean) / std


def first_frame(path: str):
    """The PIL image at `path`, or the first image file (.png / .jpg, sorted by name) of the directory `path`."""
    import os

    from PIL import Image

    from .vae import FRAME_EXTENSIONS

    if os.path.isdir(path):
        names = sorted(n for n in os.listdir(path) if n.lower().endswith(FRAME_EXTENSIONS))
        if not names:
            raise FileNotFoundError(f"{path!r} holds no .png / .jpg frame")
        path = os.path.join(path, names[0])
    if not os.path.isfile(path):
        raise FileNotFoundError(f"frame {path!r} not found")
    with Image.open(path) as im:
        return im.convert("RGB")
