"""I2VGenXL-architecture UNet3D, product side (bf16 on one B200).

Module/attribute names and the state-dict layout follow diffusers' ``I2VGenXLUNet`` so that MVOC's
hook functions (``mvoc_b200.pnp_utils.register_*``, mirroring i2vgen-xl/pnp_utils.py) address the same
objects — ``unet.up_blocks[i].attentions[j].transformer_blocks[0].attn1.processor`` etc. — and a real
checkpoint's state dict loads unchanged.

What runs underneath is this repo's C-ABI library (``mvoc_b200.ops``): every attention
(tcgen05 flash attention / warp-per-pixel temporal attention), every GroupNorm(+SiLU), the GEGLU
gate, the mask blends and the latent/DDIM updates are sm_100a kernels, and so is the dense work (SURVEY §2.2 K9,
§8f-1): 3x3 convolutions, temporal convolutions and every Linear / 1x1 conv with 64-aligned channel counts run on
the tcgen05 implicit-GEMM kernel (csrc/gemm_tc.cu) with bias / residual / GEGLU / shortcut-conv fused into its
epilogue.  What stays on cuDNN / cuBLAS through torch: conv_in (8 input channels), conv_out (4 output channels),
the three stride-2 downsamplers, the time / fps embeddings (M <= 80 rows) and the once-per-run conditioning stem.
There is no CPU path: tensors must be CUDA.

Data layout: activations are channels-last ``[B*T, H, W, C]`` (frames outermost) from conv_in to
conv_out.  In that layout every 1x1 conv / Linear / LayerNorm is a row-wise op on ``[B*T*H*W, C]``,
the spatial transformer's NCHW<->NLC permutes (pnp_utils.py:434, :502) are views, and the temporal
transformer needs no ``[(b t) c h w] <-> [(b h w) t c]`` permute (pnp_utils.py:189, :207-213) at all:
its row-wise ops do not care about row order and the temporal attention kernel walks the frames of a
pixel with a stride.  The first NCHW version of this file spent ~40 % of a step in cuDNN
nchw<->nhwc conversions and strided elementwise copies (profiles/r01_launches_v1_nchw_summary.txt).

Forward bodies restate the functions MVOC re-points (i2vgen-xl/pnp_utils.py:170-548) and the stock
diffusers blocks; citations are on each method.
"""
from __future__ import annotations

import inspect
import math
import os
from typing import Optional, Tuple

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import ops



class UNetConfig:
    def __init__(self, block_out_channels=(320, 640, 1280, 1280),
                 down_block_types=("CrossAttnDownBlock3D",) * 3 + ("DownBlock3D",),
                 up_block_types=("UpBlock3D",) + ("CrossAttnUpBlock3D",) * 3,
                 layers_per_block=2, norm_num_groups=32, cross_attention_dim=1024, attention_head_dim=64,
                 in_channels=4, out_channels=4, transformer_in_heads=8):
        self.block_out_channels = tuple(block_out_channels)
        self.down_block_types = tuple(down_block_types)
        self.up_block_types = tuple(up_block_types)
        self.layers_per_block = layers_per_block
        self.norm_num_groups = norm_num_groups
        self.cross_attention_dim = cross_attention_dim
        self.attention_head_dim = attention_head_dim
        self.in_channels = in_channels
        self.out_channels = out_channels
        self.transformer_in_heads = transformer_in_heads

    @staticmethod
    def full():
        return UNetConfig()

    @staticmethod
    def reduced():
        return UNetConfig(block_out_channels=(64, 128), down_block_types=("CrossAttnDownBlock3D", "DownBlock3D"),
                          up_block_types=("UpBlock3D", "CrossAttnUpBlock3D"), transformer_in_heads=2)

    @staticmethod
    def tiny4():
        """Full 4-level layout with narrow channels (the golden-vector model of tests/golden)."""
        return UNetConfig(block_out_channels=(64, 128, 256, 256), transformer_in_heads=2)

    @staticmethod
    def named(kind: str):
        try:
            return {"full": UNetConfig.full, "reduced": UNetConfig.reduced, "tiny4": UNetConfig.tiny4}[kind]()
        except KeyError:
            raise ValueError(f"unknown UNet config {kind!r}") from None


# ------------------------------------------------------------------ small pieces
class _Ctx:
    """Per-UNet execution context shared by its modules: the (optional) multi-GPU partition."""

    def __init__(self):
        self.parallel = None   # mvoc_b200.parallel.FrameParallel or None
        self.full_hw = None    # (h, w) of the un-sharded frame while a temporal operator runs on pixel shards
        self.temb_act = None   # (emb, SiLU(emb)) of the running forward: every resnet's time_emb_proj reads the same


# MVOC_DENSE=lib sends the dense work to cuDNN / cuBLAS instead of this repo's tcgen05 kernels: the A/B baseline
# of bench.py (recorded in its `switches`), never the product configuration.
_DENSE_TC = os.environ.get("MVOC_DENSE", "tc") != "lib"
_TC_DTYPES = (torch.bfloat16, torch.float16)


def _temb_act(ctx: Optional[_Ctx], temb: torch.Tensor) -> torch.Tensor:
    """SiLU(temb) of a resnet's time_emb_proj (pnp_utils.py:941-948).  Every resnet of one UNet forward gets the same
    temb, so I2VGenXLUNet.body computes the SiLU once and the resnets read it (the same values: one launch instead of
    one per resnet)."""
    act = ctx.temb_act if ctx is not None else None
    return act[1] if act is not None and act[0] is temb else F.silu(temb)


def cat_channels(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    """torch.cat([a, b], dim=-1) of two channels-last activations (the up blocks' skip connections): the library's
    copy kernel (mvoc_concat_lastdim, bit-identical) on the bf16 / fp16 product path, like Upsample2D's; the fp32
    host-layer tests run torch.cat."""
    if a.dtype in _TC_DTYPES and a.is_contiguous() and b.is_contiguous() and a.shape[-1] % 8 == 0 \
            and b.shape[-1] % 8 == 0:
        return ops.concat_lastdim(a, b)
    return torch.cat([a, b], dim=-1)


def derived(module: nn.Module, name: str, sources, build):
    """Weight re-layouts (tap-major conv filters, fused QKV, ...) cached on the module and rebuilt when a source
    parameter is replaced, moved, cast or edited in place (load_state_dict copies in place and bumps _version)."""
    store = module.__dict__.setdefault("_derived", {})
    key = tuple((p.data_ptr(), p._version) for p in sources)
    hit = store.get(name)
    if hit is None or hit[0] != key:
        with torch.no_grad():
            hit = (key, build())
        store[name] = hit
    return hit[1]


def invalidate_derived(root: nn.Module) -> None:
    """Drop every cached weight re-layout under `root` (load_state_dict post-hook; captured CUDA graphs that
    baked their addresses in are dropped by the pipeline through `derived_epoch`)."""
    for m in root.modules():
        m.__dict__.pop("_derived", None)
    root.__dict__["derived_epoch"] = root.__dict__.get("derived_epoch", 0) + 1


def _tc_ok(x: torch.Tensor, k: int, n: int) -> bool:
    return _DENSE_TC and x.is_cuda and x.dtype in _TC_DTYPES and k % 64 == 0 and n % 64 == 0


def dense_linear(x, weight, bias=None, residual=None):
    """x [..., K] @ weight[N, K]^T (+ bias) (+ residual): mvoc_linear, bias and residual in the epilogue."""
    n, k = weight.shape[0], weight.shape[1]
    if _tc_ok(x, k, n):
        return ops.linear(x, weight, bias, residual)
    y = F.linear(x, weight, bias)
    return y if residual is None else y.add_(residual)


def conv_nhwc(x: torch.Tensor, conv: nn.Conv2d, bias: Optional[torch.Tensor] = None,
              residual: Optional[torch.Tensor] = None, shortcut=None) -> torch.Tensor:
    """Conv2d on a channels-last activation [N, H, W, C] -> [N, H', W', C'].  `residual` (shaped like the result)
    is added to it; `shortcut` = (x2 [N, H, W, C2], conv1x1) accumulates the resnet's 1x1 shortcut conv of x2 into
    the same output tile (its bias must already be folded into `bias`).
    3x3 / stride 1 / pad 1 with 64-aligned channels: mvoc_conv3x3_nhwc (implicit GEMM on tcgen05).  Anything else
    (conv_in, conv_out, the stride-2 downsamplers): cuDNN NHWC kernels on the permuted view, which IS torch's
    channels_last memory format, so no nchw<->nhwc conversion runs."""
    b = conv.bias if bias is None else bias
    if (conv.kernel_size == (3, 3) and conv.stride == (1, 1) and conv.padding == (1, 1) and conv.dilation == (1, 1)
            and conv.groups == 1 and _tc_ok(x, conv.in_channels, conv.out_channels)
            and (shortcut is None or shortcut[1].in_channels % 64 == 0)):
        wt = derived(conv, "w_taps", (conv.weight,), lambda: ops.conv_taps(conv.weight))
        x2 = w2 = None
        if shortcut is not None:
            x2, sc = shortcut
            w2 = derived(sc, "w_rows", (sc.weight,),
                         lambda: sc.weight.reshape(sc.out_channels, sc.in_channels).contiguous())
        return ops.conv3x3(x if x.is_contiguous() else x.contiguous(), wt, b, residual, x2, w2)
    y = F.conv2d(x.permute(0, 3, 1, 2), conv.weight, b, conv.stride, conv.padding).permute(0, 2, 3, 1)
    y = y if y.is_contiguous() else y.contiguous()
    if shortcut is not None:
        x2, sc = shortcut
        co, c2 = sc.out_channels, sc.in_channels
        y.view(-1, co).addmm_(x2.reshape(-1, c2), sc.weight.view(co, c2).t())
    return y if residual is None else y.add_(residual)


class GroupNormAct(nn.GroupNorm):
    """nn.GroupNorm parameters, executed by the channels-last GroupNorm kernels (optionally fused SiLU,
    fused per-(frame, channel) add, statistics over the T frames of a video)."""

    def forward(self, x, silu: bool = False, frames_per_stat: int = 1, add=None, out=None, gather=None):
        return ops.groupnorm_nhwc(x, self.weight, self.bias, self.num_groups, self.eps, silu, frames_per_stat,
                                  add, out, gather)


class Timesteps(nn.Module):
    def __init__(self, num_channels: int):
        super().__init__()
        self.num_channels = num_channels

    def forward(self, timesteps):
        half = self.num_channels // 2
        exponent = -math.log(10000) * torch.arange(half, dtype=torch.float32, device=timesteps.device) / half
        emb = timesteps[:, None].float() * torch.exp(exponent)[None, :]
        return torch.cat([torch.cos(emb), torch.sin(emb)], dim=-1)


class TimestepEmbedding(nn.Module):
    def __init__(self, in_channels: int, time_embed_dim: int):
        super().__init__()
        self.linear_1 = nn.Linear(in_channels, time_embed_dim)
        self.act = nn.SiLU()
        self.linear_2 = nn.Linear(time_embed_dim, time_embed_dim)

    def forward(self, sample, condition=None):
        return self.linear_2(self.act(self.linear_1(sample)))


# ------------------------------------------------------------------ attention
class TemporalShape:
    """Marks hidden_states [B*T, S, C] as frame-major tokens whose attention runs over the T frames of
    each (video, pixel) — what the reference expresses by permuting to [(b h w), T, C] (pnp_utils.py:189)."""

    __slots__ = ("videos", "frames", "pixels")

    def __init__(self, videos: int, frames: int, pixels: int):
        self.videos, self.frames, self.pixels = videos, frames, pixels


def run_attention(q, k, v, heads, temporal: Optional[TemporalShape]):
    """q [N, Sq, C], k/v [N, Sk, C] (any row stride).  Spatial / cross: tcgen05 kernel over the S axis.
    Temporal: warp-per-(pixel, head) kernel over the frame axis, reading the frame-major rows in place."""
    if temporal is None:
        return ops.attention(q, k, v, heads)
    C = q.shape[-1]
    rows = q.shape[0] * q.shape[1]
    o = ops.temporal_attention_frames(q.view(rows, C), k.view(rows, C), v.view(rows, C), heads,
                                      temporal.videos, temporal.frames, temporal.pixels)
    return o.view(q.shape[0], q.shape[1], C)


class AttnProcessor2_0:
    """Stock processor (diffusers AttnProcessor2_0 == pnp_utils.py:576-612 + :674-704 minus the
    injection block) over the C-ABI attention kernels."""

    def __call__(self, attn, hidden_states, encoder_hidden_states=None, attention_mask=None, temb=None,
                 scale: float = 1.0):
        if attention_mask is not None:
            raise NotImplementedError("attention_mask is never set on this path (pnp_utils.py:594)")
        if encoder_hidden_states is None:
            q, k, v = attn.qkv_self(hidden_states)
        else:
            q = dense_linear(hidden_states, attn.to_q.weight)
            k, v = attn.kv_cross(encoder_hidden_states)
        out = run_attention(q, k, v, attn.heads, attn.temporal if encoder_hidden_states is None else None)
        return attn.out_proj(out)


class Attention(nn.Module):
    def __init__(self, query_dim: int, cross_attention_dim: Optional[int] = None, heads: int = 8,
                 dim_head: int = 64, bias: bool = False, out_bias: bool = True):
        super().__init__()
        self.inner_dim = dim_head * heads
        self.heads = heads
        self.dim_head = dim_head
        kv_dim = cross_attention_dim if cross_attention_dim is not None else query_dim
        self.is_cross = cross_attention_dim is not None
        self.scale = dim_head ** -0.5
        self.rescale_output_factor = 1.0
        self.residual_connection = False
        self.spatial_norm = self.group_norm = self.norm_cross = None
        self.to_q = nn.Linear(query_dim, self.inner_dim, bias=bias)
        self.to_k = nn.Linear(kv_dim, self.inner_dim, bias=bias)
        self.to_v = nn.Linear(kv_dim, self.inner_dim, bias=bias)
        self.to_out = nn.ModuleList([nn.Linear(self.inner_dim, query_dim, bias=out_bias), nn.Dropout(0.0)])
        self._processor = None
        self._accepts_hw = False
        self._residual = None        # offered by the transformer block, consumed by out_proj
        self.temporal: Optional[TemporalShape] = None   # set per call by the temporal transformer
        self.ctx: Optional[_Ctx] = None
        self.processor = AttnProcessor2_0()

    # `module.processor = obj` is how MVOC installs its processors (pnp_utils.py:715, :897)
    @property
    def processor(self):
        return self._processor

    @processor.setter
    def processor(self, p):
        object.__setattr__(self, "_processor", p)
        # attention_forward (pnp_utils.py:357-365) inspects the processor on every call; the
        # answer only changes when the processor does, so it is computed here once.
        object.__setattr__(self, "_accepts_hw", "height" in inspect.signature(p.__call__).parameters)

    def qkv_self(self, x):
        """One GEMM for the three self-attention projections; q, k, v are strided views."""
        ws = (self.to_q.weight, self.to_k.weight, self.to_v.weight)
        w = derived(self, "w_qkv", ws, lambda: torch.cat(ws, dim=0).contiguous())
        qkv = dense_linear(x, w)
        c = self.inner_dim
        return qkv[..., :c], qkv[..., c:2 * c], qkv[..., 2 * c:]

    def kv_cross(self, ctx):
        ws = (self.to_k.weight, self.to_v.weight)
        w = derived(self, "w_kv", ws, lambda: torch.cat(ws, dim=0).contiguous())
        kv = dense_linear(ctx, w)
        c = self.inner_dim
        return kv[..., :c], kv[..., c:]

    def out_proj(self, x):
        """to_out[0] (+ the no-op dropout, pnp_utils.py:692-694).  When the transformer block has offered its
        residual (`_residual`), the skip add of pnp_utils.py:283 / :315 rides in the GEMM epilogue."""
        res, self._residual = self._residual, None
        return dense_linear(x, self.to_out[0].weight, self.to_out[0].bias, res)

    def forward(self, hidden_states, encoder_hidden_states=None, attention_mask=None, height=None, width=None,
                **cross_attention_kwargs):
        """attention_forward, pnp_utils.py:348-385."""
        if self._accepts_hw:
            return self._processor(self, hidden_states, encoder_hidden_states=encoder_hidden_states,
                                   attention_mask=attention_mask, height=height, width=width)
        return self._processor(self, hidden_states, encoder_hidden_states=encoder_hidden_states,
                               attention_mask=attention_mask)


class LayerNormK(nn.LayerNorm):
    """nn.LayerNorm parameters, executed by mvoc_layernorm (warp per row)."""

    def forward(self, x):
        return ops.layernorm(x, self.weight, self.bias, self.eps)


class GEGLU(nn.Module):
    def __init__(self, dim_in: int, dim_out: int):
        super().__init__()
        self.proj = nn.Linear(dim_in, dim_out * 2)

    def forward(self, x):
        k, f2 = self.proj.in_features, self.proj.out_features
        if _tc_ok(x, k, f2 // 2) and x.is_contiguous():
            return ops.linear_geglu(x, self.proj.weight, self.proj.bias)   # gate in the GEMM epilogue
        return ops.geglu(self.proj(x))      # x * gelu(gate) in one pass (mvoc_geglu)


class GELU(nn.Module):
    def __init__(self, dim_in: int, dim_out: int):
        super().__init__()
        self.proj = nn.Linear(dim_in, dim_out)

    def forward(self, x):
        return F.gelu(self.proj(x))


class FeedForward(nn.Module):
    def __init__(self, dim: int, mult: int = 4, activation_fn: str = "geglu"):
        super().__init__()
        inner = dim * mult
        self.net = nn.ModuleList([GEGLU(dim, inner) if activation_fn == "geglu" else GELU(dim, inner),
                                  nn.Dropout(0.0), nn.Linear(inner, dim)])

    def forward(self, x, residual=None):
        out = self.net[2]
        return dense_linear(self.net[0](x), out.weight, out.bias, residual)


class BasicTransformerBlock(nn.Module):
    """basic_transformer_block_forward, pnp_utils.py:222-346 (norm_type 'layer_norm').  Row-wise except for
    the two attention cores; `temporal` selects the frame axis for them."""

    def __init__(self, dim, num_attention_heads, attention_head_dim, cross_attention_dim=None,
                 double_self_attention=False):
        super().__init__()
        self.only_cross_attention = False
        self.norm_type = "layer_norm"
        self.norm1 = LayerNormK(dim, eps=1e-5)
        self.attn1 = Attention(dim, None, num_attention_heads, attention_head_dim, bias=False)
        self.norm2 = LayerNormK(dim, eps=1e-5)
        self.attn2 = Attention(dim, None if double_self_attention else cross_attention_dim,
                               num_attention_heads, attention_head_dim, bias=False)
        self.norm3 = LayerNormK(dim, eps=1e-5)
        self.ff = FeedForward(dim, activation_fn="geglu")

    def forward(self, hidden_states, encoder_hidden_states=None, height=None, width=None,
                temporal: Optional[TemporalShape] = None):
        self.attn1.temporal = temporal
        self.attn2.temporal = temporal
        hidden_states = self._attend(self.attn1, self.norm1(hidden_states), hidden_states,
                                     encoder_hidden_states=None, height=height, width=width)       # :283
        hidden_states = self._attend(self.attn2, self.norm2(hidden_states), hidden_states,
                                     encoder_hidden_states=encoder_hidden_states)                   # :315
        return self.ff(self.norm3(hidden_states), residual=hidden_states)       # :322-342

    @staticmethod
    def _attend(attn, normed, residual, **kw):
        """attn(normed) + residual.  The residual is offered to the processor's output projection
        (Attention.out_proj fuses it into the GEMM epilogue); a processor that projects on its own leaves it
        unconsumed and the add runs here."""
        attn._residual = residual
        h = attn(normed, **kw)
        if attn._residual is None:
            return h
        attn._residual = None
        return h.add_(residual)


class Transformer2DModel(nn.Module):
    """transformer2dmodel_forward live branch, pnp_utils.py:426-434 and :462-508, on channels-last
    activations: the NCHW->NLC permute (:434) and its inverse (:502) are views and the two 1x1 convs are
    row-wise GEMMs."""

    def __init__(self, num_attention_heads, attention_head_dim, in_channels, cross_attention_dim, norm_num_groups=32):
        super().__init__()
        inner = num_attention_heads * attention_head_dim
        self.is_input_continuous, self.use_linear_projection = True, False
        self.norm = GroupNormAct(norm_num_groups, in_channels, eps=1e-6, affine=True)
        self.proj_in = nn.Conv2d(in_channels, inner, kernel_size=1)
        self.transformer_blocks = nn.ModuleList(
            [BasicTransformerBlock(inner, num_attention_heads, attention_head_dim, cross_attention_dim)])
        self.proj_out = nn.Conv2d(inner, in_channels, kernel_size=1)

    def forward(self, hidden_states, encoder_hidden_states=None, **kwargs):
        n, height, width, C = hidden_states.shape
        inner = self.proj_in.out_channels
        x = self.norm(hidden_states)                                            # :430
        tokens = dense_linear(x.view(n, height * width, C), self.proj_in.weight.view(inner, C), self.proj_in.bias)
        for block in self.transformer_blocks:                                   # :487-497
            tokens = block(tokens, encoder_hidden_states=encoder_hidden_states, height=height, width=width)
        out = dense_linear(tokens, self.proj_out.weight.view(C, inner), self.proj_out.bias,
                           hidden_states.view(n, height * width, C))            # :503 + the skip add of :508
        return (out.view(n, height, width, C),)


class TransformerTemporalModel(nn.Module):
    """transformer_temporal_model_forward, pnp_utils.py:170-220, on frame-major channels-last rows."""

    def __init__(self, num_attention_heads, attention_head_dim, in_channels, cross_attention_dim, norm_num_groups=32):
        super().__init__()
        inner = num_attention_heads * attention_head_dim
        self.norm = GroupNormAct(norm_num_groups, in_channels, eps=1e-6, affine=True)
        self.proj_in = nn.Linear(in_channels, inner)
        self.transformer_blocks = nn.ModuleList(
            [BasicTransformerBlock(inner, num_attention_heads, attention_head_dim, cross_attention_dim,
                                   double_self_attention=True)])
        self.proj_out = nn.Linear(inner, in_channels)
        self.ctx: Optional[_Ctx] = None

    def forward(self, hidden_states, encoder_hidden_states=None, num_frames: int = 1, **kwargs):
        par = self.ctx.parallel if self.ctx is not None else None
        if par is not None and par.world > 1:
            return (par.temporal_transformer(self, hidden_states, num_frames),)
        return (self.forward_local(hidden_states, num_frames, None),)

    def forward_local(self, hidden_states, num_frames, gather):
        """hidden_states [(b t), h, w, C] holding ALL frames of its pixels (h*w may be a pixel shard)."""
        bt, height, width, C = hidden_states.shape
        b, S = bt // num_frames, height * width
        x = self.norm(hidden_states, frames_per_stat=num_frames, gather=gather)  # 5-D GroupNorm, :185-188
        x = dense_linear(x.view(bt, S, C), self.proj_in.weight, self.proj_in.bias)   # :191 (permute :189 implicit)
        shape = TemporalShape(b, num_frames, S)
        for block in self.transformer_blocks:                                   # :194-203
            x = block(x, encoder_hidden_states=None, height=height, width=width, temporal=shape)
        x = dense_linear(x, self.proj_out.weight, self.proj_out.bias, hidden_states.view(bt, S, C))   # :206-215
        return x.view(bt, height, width, C)


# ------------------------------------------------------------------ conv blocks
class ResnetBlock2D(nn.Module):
    """Stock ResnetBlock2D forward == the closure at pnp_utils.py:902-1020 without the injection block.
    temb_channels=None builds the VAE's resnet: no time_emb_proj, called as forward(x, None)."""

    def __init__(self, in_channels, out_channels, temb_channels, groups=32, eps=1e-5):
        super().__init__()
        self.norm1 = GroupNormAct(groups, in_channels, eps=eps, affine=True)
        self.conv1 = nn.Conv2d(in_channels, out_channels, 3, padding=1)
        self.time_emb_proj = nn.Linear(temb_channels, out_channels) if temb_channels is not None else None
        self.norm2 = GroupNormAct(groups, out_channels, eps=eps, affine=True)
        self.dropout = nn.Dropout(0.0)
        self.conv2 = nn.Conv2d(out_channels, out_channels, 3, padding=1)
        self.nonlinearity = nn.SiLU()
        self.upsample = self.downsample = None
        self.output_scale_factor = 1.0
        self.conv_shortcut = nn.Conv2d(in_channels, out_channels, 1) if in_channels != out_channels else None
        self.feature_hook = None  # set by register_resnet_injection
        self.ctx: Optional[_Ctx] = None

    def forward(self, input_tensor, temb, scale: float = 1.0):
        n, H, W, cin = input_tensor.shape
        h = self.norm1(input_tensor, silu=True)                                 # :909-910
        h = conv_nhwc(h, self.conv1)                                            # :939
        t = None if self.time_emb_proj is None else self.time_emb_proj(_temb_act(self.ctx, temb))   # :941-948
        h = self.norm2(h, silu=True, add=t, out=h)                              # `+ temb` :952 fused into norm2 :953, :965
        if self.conv_shortcut is None:
            if self.feature_hook is None:
                return conv_nhwc(h, self.conv2, residual=input_tensor)          # :968 + :1018 (scale factor 1)
            h = conv_nhwc(h, self.conv2)                                        # :968
            self.feature_hook(self, h)                                          # :970-1004
            return h.add_(input_tensor)                                         # :1018
        # 1x1 shortcut conv (:1011-1016) == extra K chunks of conv2's implicit GEMM; its bias rides on
        # conv2's (a per-channel constant commutes with the per-pixel select of the injection)
        sc = self.conv_shortcut
        bias2 = derived(self, "bias2", (self.conv2.bias, sc.bias), lambda: (self.conv2.bias + sc.bias).detach())
        if self.feature_hook is None:
            return conv_nhwc(h, self.conv2, bias=bias2, shortcut=(input_tensor, sc))
        h = conv_nhwc(h, self.conv2, bias=bias2)
        self.feature_hook(self, h)                                              # blend BEFORE the shortcut add
        cout = h.shape[-1]
        return dense_linear(input_tensor.view(-1, cin), sc.weight.view(cout, cin), None,
                            h.view(-1, cout)).view(n, H, W, cout)


class _TemporalTap(nn.Sequential):
    """[GroupNorm, SiLU, (Dropout), Conv3d(k=(3,1,1))] — an nn.Sequential so the state-dict names equal
    diffusers' ("conv1.0.weight", "conv1.2.weight", "conv2.3.weight", ...); executed as GroupNorm(5-D
    statistics)+SiLU in one kernel and the 3-tap temporal conv as accumulating row GEMMs on frame-shifted
    row ranges (no [B,C,T,H,W] permute and no im2col copy)."""

    def __init__(self, dim_in, dim_out, groups, with_dropout):
        mods = [GroupNormAct(groups, dim_in), nn.SiLU()]
        if with_dropout:
            mods.append(nn.Dropout(0.0))
        mods.append(nn.Conv3d(dim_in, dim_out, (3, 1, 1), padding=(1, 0, 0)))
        super().__init__(*mods)

    @property
    def norm(self):
        return self[0]

    @property
    def conv(self):
        return self[len(self) - 1]

    def forward(self, x, num_frames, gather=None, residual=None):
        """x: [(b t), h, w, C] frame-major channels-last -> same layout (+ residual, the layer's identity)."""
        bt, h, w, C = x.shape
        b, S = bt // num_frames, h * w
        y = self.norm(x, silu=True, frames_per_stat=num_frames, gather=gather)
        conv = self.conv
        co = conv.out_channels
        if _tc_ok(y, C, co):
            wt = derived(self, "w_taps", (conv.weight,), lambda: ops.conv_taps(conv.weight))
            return ops.temporal_conv3(y, wt, conv.bias, b, num_frames, residual)
        # [co, ci, 3, 1, 1] -> [tap, ci, co] (right-hand operands of accumulating row GEMMs on frame-shifted rows)
        taps = derived(self, "taps_t", (conv.weight,), lambda: conv.weight.view(co, C, 3).permute(2, 1, 0).contiguous())
        wp, wc, wn = taps[0], taps[1], taps[2]
        y2 = y.view(bt * S, C)
        out = torch.addmm(conv.bias, y2, wc)                                    # centre tap, all frames
        rows = num_frames * S
        if num_frames > 1:
            for i in range(b):
                r0, r1 = i * rows, (i + 1) * rows
                out[r0 + S:r1].addmm_(y2[r0:r1 - S], wp)                        # tap on frame t-1
                out[r0:r1 - S].addmm_(y2[r0 + S:r1], wn)                        # tap on frame t+1
        out = out.view(bt, h, w, co)
        return out if residual is None else out.add_(residual)


class TemporalConvLayer(nn.Module):
    """Stock TemporalConvLayer forward == the closure at pnp_utils.py:1042-1057 without the injection."""

    def __init__(self, in_dim, out_dim=None, dropout=0.1, norm_num_groups=32):
        super().__init__()
        out_dim = out_dim or in_dim
        self.conv1 = _TemporalTap(in_dim, out_dim, norm_num_groups, False)
        self.conv2 = _TemporalTap(out_dim, in_dim, norm_num_groups, True)
        self.conv3 = _TemporalTap(out_dim, in_dim, norm_num_groups, True)
        self.conv4 = _TemporalTap(out_dim, in_dim, norm_num_groups, True)
        nn.init.zeros_(self.conv4.conv.weight)
        nn.init.zeros_(self.conv4.conv.bias)
        self.feature_hook = None  # set by register_temp_conv_injection
        self.ctx: Optional[_Ctx] = None

    def forward(self, hidden_states, num_frames: int = 1):
        par = self.ctx.parallel if self.ctx is not None else None
        if par is not None and par.world > 1:
            h = par.temporal_conv(self, hidden_states, num_frames)
        else:
            h = self.forward_local(hidden_states, num_frames, None)
        if self.feature_hook is not None:
            self.feature_hook(self, h)                                          # :1059-1082
        return h

    def forward_local(self, hidden_states, num_frames, gather):
        h = self.conv1(hidden_states, num_frames, gather)                       # :1048
        h = self.conv2(h, num_frames, gather)
        h = self.conv3(h, num_frames, gather)
        return self.conv4(h, num_frames, gather, residual=hidden_states)        # :1051 + identity :1053


class Downsample2D(nn.Module):
    def __init__(self, channels):
        super().__init__()
        self.conv = nn.Conv2d(channels, channels, 3, stride=2, padding=1)

    def forward(self, x, scale: float = 1.0):
        return conv_nhwc(x, self.conv)


class Upsample2D(nn.Module):
    def __init__(self, channels):
        super().__init__()
        self.conv = nn.Conv2d(channels, channels, 3, padding=1)

    def forward(self, x, output_size=None, scale: float = 1.0):
        n, h, w, c = x.shape
        if (output_size is None or tuple(output_size) == (2 * h, 2 * w)) and c % 8 == 0 and x.is_contiguous() \
                and x.dtype in (torch.bfloat16, torch.float16):
            return conv_nhwc(ops.upsample_nearest2x(x), self.conv)               # the library's kernel
        xc = x.permute(0, 3, 1, 2)                                              # channels_last view
        if output_size is None:
            xc = F.interpolate(xc, scale_factor=2.0, mode="nearest")
        else:
            xc = F.interpolate(xc, size=output_size, mode="nearest")
        return conv_nhwc(xc.permute(0, 2, 3, 1), self.conv)


class _Block3D(nn.Module):
    has_cross_attention = False

    def _make(self, n, in_chs, out_ch, temb, head_dim, cross_dim, groups, attn):
        self.resnets = nn.ModuleList([ResnetBlock2D(ic, out_ch, temb, groups) for ic in in_chs])
        self.temp_convs = nn.ModuleList([TemporalConvLayer(out_ch, out_ch, 0.1, groups) for _ in range(n)])
        if attn:
            heads = out_ch // head_dim
            self.attentions = nn.ModuleList(
                [Transformer2DModel(heads, head_dim, out_ch, cross_dim, groups) for _ in range(n)])
            self.temp_attentions = nn.ModuleList(
                [TransformerTemporalModel(heads, head_dim, out_ch, cross_dim, groups) for _ in range(n)])


class CrossAttnDownBlock3D(_Block3D):
    has_cross_attention = True

    def __init__(self, in_ch, out_ch, temb, n_layers, head_dim, cross_dim, groups, add_downsample):
        super().__init__()
        self._make(n_layers, [in_ch] + [out_ch] * (n_layers - 1), out_ch, temb, head_dim, cross_dim, groups, True)
        self.downsamplers = nn.ModuleList([Downsample2D(out_ch)]) if add_downsample else None

    def forward(self, hidden_states, temb=None, encoder_hidden_states=None, num_frames=1, **kw):
        outs = ()
        for resnet, temp_conv, attn, temp_attn in zip(self.resnets, self.temp_convs, self.attentions,
                                                      self.temp_attentions):
            hidden_states = resnet(hidden_states, temb)
            hidden_states = temp_conv(hidden_states, num_frames=num_frames)
            hidden_states = attn(hidden_states, encoder_hidden_states=encoder_hidden_states)[0]
            hidden_states = temp_attn(hidden_states, num_frames=num_frames)[0]
            outs += (hidden_states,)
        if self.downsamplers is not None:
            for d in self.downsamplers:
                hidden_states = d(hidden_states)
            outs += (hidden_states,)
        return hidden_states, outs


class DownBlock3D(_Block3D):
    def __init__(self, in_ch, out_ch, temb, n_layers, groups, add_downsample):
        super().__init__()
        self._make(n_layers, [in_ch] + [out_ch] * (n_layers - 1), out_ch, temb, 0, 0, groups, False)
        self.downsamplers = nn.ModuleList([Downsample2D(out_ch)]) if add_downsample else None

    def forward(self, hidden_states, temb=None, num_frames=1, **kw):
        outs = ()
        for resnet, temp_conv in zip(self.resnets, self.temp_convs):
            hidden_states = resnet(hidden_states, temb)
            hidden_states = temp_conv(hidden_states, num_frames=num_frames)
            outs += (hidden_states,)
        if self.downsamplers is not None:
            for d in self.downsamplers:
                hidden_states = d(hidden_states)
            outs += (hidden_states,)
        return hidden_states, outs


class UNetMidBlock3DCrossAttn(_Block3D):
    has_cross_attention = True

    def __init__(self, ch, temb, head_dim, cross_dim, groups):
        super().__init__()
        self.resnets = nn.ModuleList([ResnetBlock2D(ch, ch, temb, groups) for _ in range(2)])
        self.temp_convs = nn.ModuleList([TemporalConvLayer(ch, ch, 0.1, groups) for _ in range(2)])
        heads = ch // head_dim
        self.attentions = nn.ModuleList([Transformer2DModel(heads, head_dim, ch, cross_dim, groups)])
        self.temp_attentions = nn.ModuleList([TransformerTemporalModel(heads, head_dim, ch, cross_dim, groups)])

    def forward(self, hidden_states, temb=None, encoder_hidden_states=None, num_frames=1, **kw):
        hidden_states = self.resnets[0](hidden_states, temb)
        hidden_states = self.temp_convs[0](hidden_states, num_frames=num_frames)
        for attn, temp_attn, resnet, temp_conv in zip(self.attentions, self.temp_attentions, self.resnets[1:],
                                                      self.temp_convs[1:]):
            hidden_states = attn(hidden_states, encoder_hidden_states=encoder_hidden_states)[0]
            hidden_states = temp_attn(hidden_states, num_frames=num_frames)[0]
            hidden_states = resnet(hidden_states, temb)
            hidden_states = temp_conv(hidden_states, num_frames=num_frames)
        return hidden_states


def _up_in_channels(in_ch, out_ch, prev_out, n_layers):
    ins = []
    for i in range(n_layers):
        res_skip = in_ch if i == n_layers - 1 else out_ch
        res_in = prev_out if i == 0 else out_ch
        ins.append(res_in + res_skip)
    return ins


class CrossAttnUpBlock3D(_Block3D):
    has_cross_attention = True

    def __init__(self, in_ch, out_ch, prev_out, temb, n_layers, head_dim, cross_dim, groups, add_upsample):
        super().__init__()
        self._make(n_layers, _up_in_channels(in_ch, out_ch, prev_out, n_layers), out_ch, temb, head_dim, cross_dim,
                   groups, True)
        self.upsamplers = nn.ModuleList([Upsample2D(out_ch)]) if add_upsample else None

    def forward(self, hidden_states, res_hidden_states_tuple, temb=None, encoder_hidden_states=None,
                upsample_size=None, num_frames=1, **kw):
        for resnet, temp_conv, attn, temp_attn in zip(self.resnets, self.temp_convs, self.attentions,
                                                      self.temp_attentions):
            res = res_hidden_states_tuple[-1]
            res_hidden_states_tuple = res_hidden_states_tuple[:-1]
            hidden_states = cat_channels(hidden_states, res)
            hidden_states = resnet(hidden_states, temb)
            hidden_states = temp_conv(hidden_states, num_frames=num_frames)
            hidden_states = attn(hidden_states, encoder_hidden_states=encoder_hidden_states)[0]
            hidden_states = temp_attn(hidden_states, num_frames=num_frames)[0]
        if self.upsamplers is not None:
            for u in self.upsamplers:
                hidden_states = u(hidden_states, upsample_size)
        return hidden_states


class UpBlock3D(_Block3D):
    def __init__(self, in_ch, out_ch, prev_out, temb, n_layers, groups, add_upsample):
        super().__init__()
        self._make(n_layers, _up_in_channels(in_ch, out_ch, prev_out, n_layers), out_ch, temb, 0, 0, groups, False)
        self.upsamplers = nn.ModuleList([Upsample2D(out_ch)]) if add_upsample else None

    def forward(self, hidden_states, res_hidden_states_tuple, temb=None, upsample_size=None, num_frames=1, **kw):
        for resnet, temp_conv in zip(self.resnets, self.temp_convs):
            res = res_hidden_states_tuple[-1]
            res_hidden_states_tuple = res_hidden_states_tuple[:-1]
            hidden_states = cat_channels(hidden_states, res)
            hidden_states = resnet(hidden_states, temb)
            hidden_states = temp_conv(hidden_states, num_frames=num_frames)
        if self.upsamplers is not None:
            for u in self.upsamplers:
                hidden_states = u(hidden_states, upsample_size)
        return hidden_states


class TinyAttention(nn.Module):
    """Attention(query_dim=4, heads=2, dim_head=4) of I2VGenXLTransformerTemporalEncoder: head_dim 4 is
    below any tensor-core tile; 0.0002 % of the FLOPs.  Computed with explicit matmuls (no SDPA library)."""

    def __init__(self, dim, heads, dim_head):
        super().__init__()
        inner = heads * dim_head
        self.heads, self.dim_head = heads, dim_head
        self.to_q = nn.Linear(dim, inner, bias=False)
        self.to_k = nn.Linear(dim, inner, bias=False)
        self.to_v = nn.Linear(dim, inner, bias=False)
        self.to_out = nn.ModuleList([nn.Linear(inner, dim, bias=True), nn.Dropout(0.0)])

    def forward(self, x):
        B, N, _ = x.shape
        q = self.to_q(x).view(B, N, self.heads, self.dim_head).transpose(1, 2).float()
        k = self.to_k(x).view(B, N, self.heads, self.dim_head).transpose(1, 2).float()
        v = self.to_v(x).view(B, N, self.heads, self.dim_head).transpose(1, 2).float()
        p = torch.softmax(q @ k.transpose(-1, -2) * (self.dim_head ** -0.5), dim=-1)
        o = (p @ v).transpose(1, 2).reshape(B, N, self.heads * self.dim_head).to(x.dtype)
        return self.to_out[0](o)


class I2VGenXLTransformerTemporalEncoder(nn.Module):
    def __init__(self, dim, num_attention_heads=2, attention_head_dim=4):
        super().__init__()
        self.norm1 = nn.LayerNorm(dim, eps=1e-5)
        self.attn1 = TinyAttention(dim, num_attention_heads, attention_head_dim)
        self.ff = FeedForward(dim, activation_fn="gelu")

    def forward(self, hidden_states):
        hidden_states = self.attn1(self.norm1(hidden_states)) + hidden_states
        return self.ff(hidden_states) + hidden_states


class _Cfg:
    def __init__(self, c):
        self.in_channels = c.in_channels
        self.cross_attention_dim = c.cross_attention_dim


class I2VGenXLUNet(nn.Module):
    def __init__(self, cfg: Optional[UNetConfig] = None):
        super().__init__()
        cfg = cfg or UNetConfig()
        self.cfg = cfg
        self.config = _Cfg(cfg)
        boc = cfg.block_out_channels
        temb = boc[0] * 4
        g, hd, cd, ic = cfg.norm_num_groups, cfg.attention_head_dim, cfg.cross_attention_dim, cfg.in_channels
        self.conv_in = nn.Conv2d(ic + ic, boc[0], 3, padding=1)
        self.transformer_in = TransformerTemporalModel(cfg.transformer_in_heads, hd, boc[0], cd, g)
        self.image_latents_proj_in = nn.Sequential(
            nn.Conv2d(4, ic * 4, 3, padding=1), nn.SiLU(), nn.Conv2d(ic * 4, ic * 4, 3, padding=1), nn.SiLU(),
            nn.Conv2d(ic * 4, ic, 3, padding=1))
        self.image_latents_temporal_encoder = I2VGenXLTransformerTemporalEncoder(ic, 2, ic)
        self.image_latents_context_embedding = nn.Sequential(
            nn.Conv2d(4, ic * 8, 3, padding=1), nn.SiLU(), nn.AdaptiveAvgPool2d((32, 32)),
            nn.Conv2d(ic * 8, ic * 16, 3, stride=2, padding=1), nn.SiLU(),
            nn.Conv2d(ic * 16, cd, 3, stride=2, padding=1))
        self.time_proj = Timesteps(boc[0])
        self.time_embedding = TimestepEmbedding(boc[0], temb)
        self.context_embedding = nn.Sequential(nn.Linear(cd, temb), nn.SiLU(), nn.Linear(temb, cd * ic))
        self.fps_embedding = nn.Sequential(nn.Linear(boc[0], temb), nn.SiLU(), nn.Linear(temb, temb))
        self.down_blocks = nn.ModuleList()
        out_ch = boc[0]
        for i, t in enumerate(cfg.down_block_types):
            in_ch, out_ch = out_ch, boc[i]
            final = i == len(boc) - 1
            if t == "CrossAttnDownBlock3D":
                self.down_blocks.append(CrossAttnDownBlock3D(in_ch, out_ch, temb, cfg.layers_per_block, hd, cd, g,
                                                             not final))
            else:
                self.down_blocks.append(DownBlock3D(in_ch, out_ch, temb, cfg.layers_per_block, g, not final))
        self.mid_block = UNetMidBlock3DCrossAttn(boc[-1], temb, hd, cd, g)
        self.num_upsamplers = 0
        self.up_blocks = nn.ModuleList()
        rev = list(reversed(boc))
        out_ch = rev[0]
        for i, t in enumerate(cfg.up_block_types):
            final = i == len(boc) - 1
            prev_out, out_ch = out_ch, rev[i]
            in_ch = rev[min(i + 1, len(boc) - 1)]
            if not final:
                self.num_upsamplers += 1
            if t == "CrossAttnUpBlock3D":
                self.up_blocks.append(CrossAttnUpBlock3D(in_ch, out_ch, prev_out, temb, cfg.layers_per_block + 1,
                                                         hd, cd, g, not final))
            else:
                self.up_blocks.append(UpBlock3D(in_ch, out_ch, prev_out, temb, cfg.layers_per_block + 1, g,
                                                not final))
        self.conv_norm_out = GroupNormAct(g, boc[0], eps=1e-5)
        self.conv_act = nn.SiLU()
        self.conv_out = nn.Conv2d(boc[0], cfg.out_channels, 3, padding=1)
        self.conv_out.feature_hook = None  # set by register_out_conv_injection
        self.ctx = _Ctx()
        for m in self.modules():
            if isinstance(m, (TransformerTemporalModel, TemporalConvLayer, Attention, ResnetBlock2D)):
                m.ctx = self.ctx
        # weights edited after the first forward: drop the cached re-layouts (and, through derived_epoch, the
        # CUDA graphs that captured their addresses)
        self.register_load_state_dict_post_hook(lambda module, incompatible: invalidate_derived(module))

    @property
    def dtype(self):
        return self.conv_in.weight.dtype

    # ------------------------------------------------------------------
    def _embeddings(self, sample, timestep, fps):
        timesteps = timestep
        if not torch.is_tensor(timesteps):
            timesteps = torch.tensor([timesteps], dtype=torch.int64, device=sample.device)
        elif timesteps.dim() == 0:
            timesteps = timesteps[None].to(sample.device)
        timesteps = timesteps.expand(sample.shape[0])
        t_emb = self.time_embedding(self.time_proj(timesteps).to(self.dtype))
        fps_emb = self.fps_embedding(self.time_proj(fps.expand(fps.shape[0])).to(self.dtype))
        return t_emb + fps_emb

    def context(self, encoder_hidden_states, image_latents, image_embeddings):
        """Context tokens [B, 77 + 64 + 4, 1024] of ONE frame per video (pipeline_i2vgen_xl.py:204-240 with
        multi_frame_guidance False computes the same tensor T times; it only depends on frame 0)."""
        il = image_latents[:, :, 0]
        il = self.image_latents_context_embedding(il)
        b, c, h, w = il.shape
        il = il.permute(0, 2, 3, 1).reshape(b, h * w, c)
        image_emb = self.context_embedding(image_embeddings[:, 0:1, :])
        image_emb = image_emb.view(-1, self.config.in_channels, self.config.cross_attention_dim)
        return torch.cat([encoder_hidden_states, il, image_emb], dim=1)

    def stem_condition(self, image_latents_first):
        """Image-latent conditioning channels [(b t), c, h, w] (pipeline_i2vgen_xl.py:264-279); independent
        of the timestep, so the step loop computes it once."""
        b, c, T, h, w = image_latents_first.shape
        il = image_latents_first.permute(0, 2, 1, 3, 4).reshape(b * T, c, h, w)
        il = self.image_latents_proj_in(il)
        il = il.view(b, T, c, h, w).permute(0, 3, 4, 1, 2).reshape(b * h * w, T, c)
        il = self.image_latents_temporal_encoder(il)
        return il.reshape(b, h, w, T, c).permute(0, 3, 4, 1, 2).reshape(b * T, c, h, w).contiguous()

    def stem(self, sample_frames, il_frames, num_frames):
        """cat + conv_in + transformer_in (pipeline_i2vgen_xl.py:282-290).  sample_frames, il_frames:
        [(b t), c, h, w] (the frames this rank owns); returns channels-last [(b t), h, w, C0]."""
        x = torch.cat([sample_frames, il_frames], dim=1).permute(0, 2, 3, 1).contiguous()
        x = conv_nhwc(x, self.conv_in)
        return self.transformer_in(x, num_frames=num_frames)[0]

    def body(self, sample, emb, context_emb, num_frames, forward_upsample_size):
        """down / mid / up / out, pipeline_i2vgen_xl.py:292-357, on channels-last [(b t), h, w, C].
        Returns the noise prediction as [(b t), 4, h, w] (contiguous NCHW)."""
        self.ctx.temb_act = (emb, F.silu(emb))                                  # read by every resnet
        try:
            return self._body(sample, emb, context_emb, num_frames, forward_upsample_size)
        finally:
            self.ctx.temb_act = None

    def _body(self, sample, emb, context_emb, num_frames, forward_upsample_size):
        upsample_size = None
        res_samples = (sample,)
        for blk in self.down_blocks:
            if blk.has_cross_attention:
                sample, res = blk(sample, temb=emb, encoder_hidden_states=context_emb, num_frames=num_frames)
            else:
                sample, res = blk(sample, temb=emb, num_frames=num_frames)
            res_samples += res
        sample = self.mid_block(sample, emb, encoder_hidden_states=context_emb, num_frames=num_frames)
        for i, blk in enumerate(self.up_blocks):
            n = len(blk.resnets)
            res = res_samples[-n:]
            res_samples = res_samples[:-n]
            if i != len(self.up_blocks) - 1 and forward_upsample_size:
                upsample_size = res_samples[-1].shape[1:3]
            if blk.has_cross_attention:
                sample = blk(sample, res, temb=emb, encoder_hidden_states=context_emb, upsample_size=upsample_size,
                             num_frames=num_frames)
            else:
                sample = blk(sample, res, temb=emb, upsample_size=upsample_size, num_frames=num_frames)
        sample = self.conv_norm_out(sample, silu=True, out=sample)              # :351-352
        sample = conv_nhwc(sample, self.conv_out).permute(0, 3, 1, 2).contiguous()   # :354 -> [(b t), 4, h, w]
        if self.conv_out.feature_hook is not None:
            self.conv_out.feature_hook(self.conv_out, sample)                   # pnp_utils.py:1114-1146
        return sample

    def forward(self, sample, timestep, fps, image_latents, image_embeddings=None, encoder_hidden_states=None,
                image_latents_first=None, return_dict: bool = False, **kwargs):
        """Stock signature (diffusers I2VGenXLUNet.forward) plus MVOC's `image_latents_first`
        (I2VGenXLUnetExtension.forward, pipeline_i2vgen_xl.py:109-122).  Single-GPU convenience entry; the
        step loops use the pieces directly (mvoc_b200/pipeline.py).  Returns a 1-tuple [b, 4, T, h, w]."""
        if not sample.is_cuda:
            raise RuntimeError("mvoc_b200.I2VGenXLUNet runs on CUDA tensors only (no CPU fallback)")
        if image_latents_first is None:
            image_latents_first = image_latents
        b, c, T, h, w = sample.shape
        fwd_up = any(s % (2 ** self.num_upsamplers) != 0 for s in (h, w))
        emb = self._embeddings(sample, timestep, fps).repeat_interleave(T, dim=0)
        ctx = self.context(encoder_hidden_states, image_latents, image_embeddings)
        ctx = ctx.repeat_interleave(T, dim=0)
        frames = sample.permute(0, 2, 1, 3, 4).reshape(b * T, c, h, w)
        x = self.stem(frames, self.stem_condition(image_latents_first), T)
        out = self.body(x, emb, ctx, T, fwd_up)
        return (out.view(b, T, *out.shape[1:]).permute(0, 2, 1, 3, 4),)


def build_unet(kind: str = "full", seed: int = 0, device="cuda", dtype=torch.bfloat16) -> I2VGenXLUNet:
    """Random-init weights of the named architecture: torch.manual_seed(seed) + PyTorch default inits on the
    CPU in fp32, then cast/moved.  (Parity tests do not rely on RNG order: they load the oracle's state dict.)"""
    torch.manual_seed(seed)
    m = I2VGenXLUNet(UNetConfig.named(kind)).eval().requires_grad_(False)
    return prepare(m.to(device=device, dtype=dtype))


def prepare(unet: I2VGenXLUNet) -> I2VGenXLUNet:
    """Put the conv weights in channels_last memory format once (cuDNN then runs its NHWC kernels with no
    per-call filter transform)."""
    for m in unet.modules():
        if isinstance(m, nn.Conv2d) and m.kernel_size != (1, 1):
            m.weight.data = m.weight.data.contiguous(memory_format=torch.channels_last)
    return unet
