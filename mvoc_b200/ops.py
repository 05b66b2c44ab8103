"""Tensor-facing wrappers over the C-ABI (include/mvoc_b200.h).

PyTorch is used here only as the owner of device memory and streams: every
function marshals ``data_ptr()``, shapes, strides and the current CUDA stream
into one C call.  None of them has a torch/CPU fallback — a non-CUDA tensor or a
missing library raises.
"""
from __future__ import annotations

import os
from typing import Optional, Sequence

import torch

from . import _cabi
from ._cabi import MVOC_MASK_F32, MVOC_MASK_U8

_DT = {torch.bfloat16: _cabi.MVOC_BF16, torch.float16: _cabi.MVOC_F16, torch.float32: _cabi.MVOC_F32}
HEAD_DIM = 64

# number of C-ABI kernel launches issued through this module (bench.py's gpu_launches)
launch_count = 0


def _count(n: int = 1) -> None:
    global launch_count
    launch_count += n


class KernelTimer:
    """Per-launch device timing with CUDA events on the launching stream (bench.py's roofline leg).
    records[key] = list of (start_event, end_event, work) where work is algorithmic FLOPs or bytes."""

    def __init__(self):
        self.records = {}

    def add(self, key, ev0, ev1, work):
        self.records.setdefault(key, []).append((ev0, ev1, work))

    def summary(self):
        """key -> (launches, total_ms, total_work); call after torch.cuda.synchronize()."""
        out = {}
        for key, recs in self.records.items():
            ms = sum(a.elapsed_time(b) for a, b, _ in recs)
            out[key] = (len(recs), ms, sum(w for _, _, w in recs))
        return out


_timer: Optional[KernelTimer] = None


def set_timer(t: Optional[KernelTimer]) -> None:
    global _timer
    _timer = t


class _Timed:
    __slots__ = ("key", "work", "ev0")

    def __init__(self, key, work):
        self.key, self.work, self.ev0 = key, work, None

    def __enter__(self):
        if _timer is not None:
            self.ev0 = torch.cuda.Event(enable_timing=True)
            self.ev0.record()
        return self

    def __exit__(self, *exc):
        if self.ev0 is not None and _timer is not None:
            ev1 = torch.cuda.Event(enable_timing=True)
            ev1.record()
            _timer.add(self.key, self.ev0, ev1, self.work)
        return False


def _dt(t: torch.Tensor) -> int:
    try:
        return _DT[t.dtype]
    except KeyError:
        raise TypeError(f"mvoc_b200: unsupported dtype {t.dtype}") from None


def _need_cuda(*ts: Optional[torch.Tensor]) -> None:
    """Every tensor must live on the CURRENT CUDA device: the C-ABI launches on the current device and on its
    current stream, so a tensor of another GPU would be an illegal address there.  (One process per GPU is the
    deployment model; scripts call torch.cuda.set_device before touching the pipeline.)"""
    cur = -1
    for t in ts:
        if t is None:
            continue
        if not t.is_cuda:
            raise RuntimeError(
                "mvoc_b200 ops run on CUDA tensors only (sm_100a kernels; there is no CPU fallback)"
            )
        if cur < 0:
            cur = torch.cuda.current_device()
        if t.device.index != cur:
            raise RuntimeError(
                f"mvoc_b200 ops launch on the current CUDA device (cuda:{cur}) but got a tensor on {t.device}; "
                "call torch.cuda.set_device(device) first (one process per GPU)"
            )


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _bnc_strides(t: torch.Tensor, heads: int):
    """(batch, token, head) element strides of a [B, N, heads*64] tensor."""
    if t.dim() != 3 or t.shape[-1] != heads * HEAD_DIM or t.stride(-1) != 1:
        raise ValueError(
            f"expected [B, N, {heads}*{HEAD_DIM}] with a contiguous last dim, got {tuple(t.shape)} "
            f"strides {t.stride()}"
        )
    return t.stride(0), t.stride(1), HEAD_DIM


def _check_io(what: str, out: torch.Tensor, shape, *inputs: torch.Tensor) -> None:
    """The kernels take one dtype code (q's) for every operand and write `shape` through `out`'s strides: inputs and
    out must share q's dtype, and out must be exactly `shape` with a contiguous last dim."""
    dt = inputs[0].dtype
    for name, t in zip(("q", "k", "v", "out"), (*inputs, out)):
        if t.dtype != dt:
            raise ValueError(f"{what}: {name} is {t.dtype}, q is {dt}")
    if tuple(out.shape) != tuple(shape) or out.stride(-1) != 1:
        raise ValueError(f"{what}: out must be {tuple(shape)} with a contiguous last dim, got {tuple(out.shape)} "
                         f"strides {out.stride()}")


def attention(
    q: torch.Tensor,
    k: torch.Tensor,
    v: torch.Tensor,
    heads: int,
    scale: Optional[float] = None,
    out: Optional[torch.Tensor] = None,
    variant: int = 0,
) -> torch.Tensor:
    """softmax(Q K^T * scale) V for q [B,Nq,H*64], k/v [B,Nk,H*64] -> [B,Nq,H*64] (tcgen05 kernel)."""
    _need_cuda(q, k, v, out)
    B, Nq, C = q.shape
    Nk = k.shape[1]
    if k.shape[0] != B or v.shape != k.shape:
        raise ValueError(f"attention: q {tuple(q.shape)} k {tuple(k.shape)} v {tuple(v.shape)} mismatch")
    if out is None:
        out = torch.empty((B, Nq, C), dtype=q.dtype, device=q.device)
    _check_io("attention", out, (B, Nq, C), q, k, v)
    if scale is None:
        scale = HEAD_DIM ** -0.5
    lib = _cabi.load()
    with _Timed(("attn", B, heads, Nq, Nk), 4.0 * B * heads * Nq * Nk * HEAD_DIM):
        st = lib.mvoc_attn_fwd(
            q.data_ptr(), k.data_ptr(), v.data_ptr(), out.data_ptr(),
            B, heads, Nq, Nk, HEAD_DIM,
            *_bnc_strides(q, heads), *_bnc_strides(k, heads), *_bnc_strides(v, heads),
            *_bnc_strides(out, heads),
            float(scale), _dt(q), int(variant), _stream(),
        )
    _cabi.check(st, "mvoc_attn_fwd")
    _count()
    return out


def attention_causal(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, heads: int, scale: Optional[float] = None,
                     out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Causal softmax(Q K^T * scale) V with head_dim 64 (the CLIP text tower's self-attention, mvoc_attn_causal_fwd):
    query row r attends to keys 0..r.  q, k, v [B, N, H*64] (any batch / token strides, e.g. column slices of a fused
    QKV output) -> [B, N, H*64]."""
    _need_cuda(q, k, v, out)
    if q.dim() != 3 or q.shape != k.shape or v.shape != k.shape:
        raise ValueError(f"attention_causal: q {tuple(q.shape)} k {tuple(k.shape)} v {tuple(v.shape)} must be one "
                         "[B, N, H*64] shape")
    B, N, C = q.shape
    if out is None:
        out = torch.empty((B, N, C), dtype=q.dtype, device=q.device)
    _check_io("attention_causal", out, (B, N, C), q, k, v)
    if scale is None:
        scale = HEAD_DIM ** -0.5
    with _Timed(("attn_causal", B, heads, N), 2.0 * B * heads * N * (N + 1) * HEAD_DIM):
        rc = _cabi.load().mvoc_attn_causal_fwd(
            q.data_ptr(), k.data_ptr(), v.data_ptr(), out.data_ptr(), B, heads, N, N, HEAD_DIM,
            *_bnc_strides(q, heads), *_bnc_strides(k, heads), *_bnc_strides(v, heads), *_bnc_strides(out, heads),
            float(scale), _dt(q), _stream())
    _cabi.check(rc, "mvoc_attn_causal_fwd")
    _count()
    return out


WIDE_HEAD_DIM = 512


def _bn_strides(t: torch.Tensor, what: str, B: int, N: int):
    """(batch, token) element strides of a [B, N, 512] tensor with a contiguous last dim."""
    if tuple(t.shape) != (B, N, WIDE_HEAD_DIM) or t.stride(-1) != 1:
        raise ValueError(f"attention_d512: {what} must be [{B}, {N}, {WIDE_HEAD_DIM}] with a contiguous last dim, "
                         f"got {tuple(t.shape)} strides {t.stride()}")
    return t.stride(0), t.stride(1)


def attention_d512(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, scale: Optional[float] = None,
                   out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Single-head softmax(Q K^T * scale) V with head_dim 512 (the VAE decoder's mid-block attention):
    q, k, v [B, N, 512] (any batch / token strides, e.g. column slices of a fused QKV output) -> [B, N, 512]."""
    _need_cuda(q, k, v, out)
    if q.dim() != 3:
        raise ValueError(f"attention_d512: need q, k, v [B, N, 512], got {tuple(q.shape)}")
    B, N = q.shape[0], q.shape[1]
    if out is None:
        out = torch.empty((B, N, WIDE_HEAD_DIM), dtype=q.dtype, device=q.device)
    _check_io("attention_d512", out, (B, N, WIDE_HEAD_DIM), q, k, v)
    st = [s for t, nm in ((q, "q"), (k, "k"), (v, "v"), (out, "out")) for s in _bn_strides(t, nm, B, N)]
    if scale is None:
        scale = WIDE_HEAD_DIM ** -0.5
    with _Timed(("attn_d512", B, N), 4.0 * B * N * N * WIDE_HEAD_DIM):
        rc = _cabi.load().mvoc_attn_d512_fwd(q.data_ptr(), k.data_ptr(), v.data_ptr(), out.data_ptr(), B, N,
                                             WIDE_HEAD_DIM, *st, float(scale), _dt(q), _stream())
    _cabi.check(rc, "mvoc_attn_d512_fwd")
    _count()
    return out


CLIP_HEAD_DIM = 80


def _bnh80_strides(t: torch.Tensor, what: str, heads: int):
    """(batch, token, head) element strides of a [B, N, heads*80] view with a contiguous last dim."""
    if t.dim() != 3 or t.shape[-1] != heads * CLIP_HEAD_DIM or t.stride(-1) != 1:
        raise ValueError(f"attention_d80: {what} must be [B, N, {heads}*{CLIP_HEAD_DIM}] with a contiguous last dim, "
                         f"got {tuple(t.shape)} strides {t.stride()}")
    return t.stride(0), t.stride(1), CLIP_HEAD_DIM


def attention_d80(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, heads: int, scale: Optional[float] = None,
                  out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """softmax(Q K^T * scale) V with head_dim 80 (the CLIP image tower's self-attention, mvoc_attn_d80_fwd):
    q [B, Nq, H*80], k / v [B, Nk, H*80] (any batch / token strides, e.g. column slices of a fused QKV output)
    -> [B, Nq, H*80]."""
    _need_cuda(q, k, v, out)
    if q.dim() != 3 or k.dim() != 3 or k.shape[0] != q.shape[0] or v.shape != k.shape:
        raise ValueError(f"attention_d80: q {tuple(q.shape)} k {tuple(k.shape)} v {tuple(v.shape)} mismatch")
    B, Nq, C = q.shape
    Nk = k.shape[1]
    if out is None:
        out = torch.empty((B, Nq, C), dtype=q.dtype, device=q.device)
    _check_io("attention_d80", out, (B, Nq, C), q, k, v)
    st = [s for t, nm in ((q, "q"), (k, "k"), (v, "v"), (out, "out")) for s in _bnh80_strides(t, nm, heads)]
    if scale is None:
        scale = CLIP_HEAD_DIM ** -0.5
    with _Timed(("attn_d80", B, heads, Nq, Nk), 4.0 * B * heads * Nq * Nk * CLIP_HEAD_DIM):
        rc = _cabi.load().mvoc_attn_d80_fwd(q.data_ptr(), k.data_ptr(), v.data_ptr(), out.data_ptr(), B, heads, Nq,
                                            Nk, CLIP_HEAD_DIM, *st, float(scale), _dt(q), _stream())
    _cabi.check(rc, "mvoc_attn_d80_fwd")
    _count()
    return out


def temporal_attention(
    q: torch.Tensor,
    k: torch.Tensor,
    v: torch.Tensor,
    heads: int,
    scale: Optional[float] = None,
    out: Optional[torch.Tensor] = None,
) -> torch.Tensor:
    """Attention over frames: q,k,v [P, T, H*64] with T <= 32 (warp-per-problem kernel)."""
    _need_cuda(q, k, v, out)
    P, T, C = q.shape
    if k.shape != q.shape or v.shape != q.shape:
        raise ValueError("temporal_attention: q, k, v must have the same shape")
    if out is None:
        out = torch.empty((P, T, C), dtype=q.dtype, device=q.device)
    _check_io("temporal_attention", out, (P, T, C), q, k, v)
    if scale is None:
        scale = HEAD_DIM ** -0.5
    lib = _cabi.load()
    with _Timed(("attn_temporal", P, heads, T), 4.0 * P * T * C * q.element_size()):
        st = lib.mvoc_attn_temporal_fwd(
            q.data_ptr(), k.data_ptr(), v.data_ptr(), out.data_ptr(),
            P, T, heads, HEAD_DIM,
            *_bnc_strides(q, heads), *_bnc_strides(k, heads), *_bnc_strides(v, heads),
            *_bnc_strides(out, heads),
            float(scale), _dt(q), _stream(),
        )
    _cabi.check(st, "mvoc_attn_temporal_fwd")
    _count()
    return out


def qk_blend_(
    q: torch.Tensor,
    k: Optional[torch.Tensor],
    mask: torch.Tensor,
    n_obj: int,
    inject_background: bool,
) -> None:
    """In-place Q/K injection.  q,k: contiguous [n_branches*c, ...] whose slot-major flattening is
    [n_branches, tokens, C]; mask [n_obj, tokens] uint8 (select) or float32 (lerp), same token order."""
    _need_cuda(q, k, mask)
    nb = n_obj + 3
    C = q.shape[-1]
    if not q.is_contiguous() or (k is not None and not k.is_contiguous()):
        raise ValueError("qk_blend_: q and k must be contiguous")
    if q.numel() % (nb * C) != 0:
        raise ValueError(f"qk_blend_: {tuple(q.shape)} is not divisible into {nb} slots")
    tokens = q.numel() // (nb * C)
    if mask.dtype == torch.uint8:
        kind = MVOC_MASK_U8
    elif mask.dtype == torch.float32:
        kind = MVOC_MASK_F32
    else:
        raise TypeError(f"qk_blend_: mask dtype {mask.dtype} (need uint8 or float32)")
    if tuple(mask.shape) != (n_obj, tokens) or not mask.is_contiguous():
        raise ValueError(f"qk_blend_: mask must be contiguous [{n_obj}, {tokens}], got {tuple(mask.shape)}")
    base = 0 if inject_background else n_obj + 2
    lib = _cabi.load()
    st = lib.mvoc_qk_blend(q.data_ptr(), _ptr(k), n_obj, tokens, C, mask.data_ptr(), kind, base,
                           _dt(q), _stream())
    _cabi.check(st, "mvoc_qk_blend")
    _count()


def attention_pair(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, heads: int, pair_batches: int,
                   scale: Optional[float] = None, out: Optional[torch.Tensor] = None, variant: int = 0) -> torch.Tensor:
    """Two branches that share Q and K (mvoc_attn_pair_fwd): q, k [B, N, H*64]; v [B + pair_batches, N, H*64];
    out[b] = softmax(q[b] k[b]^T) v[b], out[b + pair_batches] = the same softmax times v[b + pair_batches].
    pair_batches >= B (fewer would make two CTAs write one output batch); out batches [B, pair_batches) are not
    written."""
    _need_cuda(q, k, v, out)
    B, Nq, C = q.shape
    Nk = k.shape[1]
    if k.shape[0] != B or v.shape[0] != B + pair_batches or v.shape[1] != Nk or pair_batches < B:
        raise ValueError(f"attention_pair: q {tuple(q.shape)} k {tuple(k.shape)} v {tuple(v.shape)} pair {pair_batches}")
    if out is None:
        out = torch.empty((B + pair_batches, Nq, C), dtype=q.dtype, device=q.device)
    _check_io("attention_pair", out, (B + pair_batches, Nq, C), q, k, v)
    if scale is None:
        scale = HEAD_DIM ** -0.5
    with _Timed(("attn_pair", B, heads, Nq, Nk), 2 * 4.0 * B * heads * Nq * Nk * HEAD_DIM):
        st = _cabi.load().mvoc_attn_pair_fwd(
            q.data_ptr(), k.data_ptr(), v.data_ptr(), out.data_ptr(), B, heads, Nq, Nk, HEAD_DIM,
            *_bnc_strides(q, heads), *_bnc_strides(k, heads), *_bnc_strides(v, heads), *_bnc_strides(out, heads),
            int(pair_batches), float(scale), _dt(q), int(variant), _stream())
    _cabi.check(st, "mvoc_attn_pair_fwd")
    _count()
    return out


def _token_rows(t: torch.Tensor, what: str, batches: int, pixels: int, C: int) -> int:
    """Row stride (elements) of a [batches, pixels, C] tensor whose (batch, pixel) rows are uniformly strided — a
    contiguous tensor or a column slice of a wider row-major buffer (e.g. one third of a fused QKV output)."""
    if tuple(t.shape) != (batches, pixels, C) or t.stride(2) != 1 or t.stride(0) != pixels * t.stride(1):
        raise ValueError(f"attention_inject_: {what} must be [{batches}, {pixels}, {C}] with uniformly strided rows, "
                         f"got {tuple(t.shape)} strides {t.stride()}")
    return t.stride(1)


def attention_inject_(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, mask: torch.Tensor, heads: int, n_obj: int,
                      frames: int, inject_background: bool, temporal: bool, scale: Optional[float] = None,
                      out: Optional[torch.Tensor] = None, variant: int = 0, share_p: Optional[bool] = None) -> torch.Tensor:
    """Q/K injection + attention of all branches through the single C-ABI call mvoc_attn_inject_fwd.
    q, k, v: [(n_obj+3)*frames, pixels, H*64], rows in (branch, frame, pixel) order for the spatial AND the temporal
    mode, uniformly strided (they may be the column slices of one fused QKV GEMM output); mask [n_obj,
    frames*pixels] uint8 / float32.  q and k are modified in place.  share_p (default: on for the spatial mode): one
    softmax for the uncond / cond pair, which receive the same blended Q', K'."""
    _need_cuda(q, k, v, mask, out)
    nb = n_obj + 3
    if q.dim() != 3 or q.shape[0] != nb * frames:
        raise ValueError(f"attention_inject_: need q, k, v [{nb}*{frames}, pixels, C], got {tuple(q.shape)}")
    pixels, C = q.shape[1], q.shape[2]
    if C != heads * HEAD_DIM:
        raise ValueError(f"attention_inject_: C={C} != heads*{HEAD_DIM}")
    if mask.dtype == torch.uint8:
        kind = MVOC_MASK_U8
    elif mask.dtype == torch.float32:
        kind = MVOC_MASK_F32
    else:
        raise TypeError(f"attention_inject_: mask dtype {mask.dtype} (need uint8 or float32)")
    if tuple(mask.shape) != (n_obj, frames * pixels) or not mask.is_contiguous():
        raise ValueError(f"attention_inject_: mask must be contiguous [{n_obj}, {frames * pixels}]")
    if out is None:
        out = torch.empty((nb * frames, pixels, C), dtype=q.dtype, device=q.device)
    _check_io("attention_inject_", out, (nb * frames, pixels, C), q, k, v)
    lds = [_token_rows(t, nm, nb * frames, pixels, C) for t, nm in ((q, "q"), (k, "k"), (v, "v"), (out, "out"))]
    if scale is None:
        scale = HEAD_DIM ** -0.5
    if share_p is None:
        share_p = not temporal
    base = 0 if inject_background else n_obj + 2
    rows = nb * frames * pixels
    if temporal:
        timed = _Timed(("attn_temporal", nb * pixels, heads, frames), 4.0 * rows * C * q.element_size())
    else:   # algorithmic FLOPs of the reference: every branch runs its own softmax (pnp_utils.py:684)
        timed = _Timed(("attn_inject", nb * frames, heads, pixels, pixels, int(bool(share_p))),
                       4.0 * nb * frames * heads * pixels * pixels * HEAD_DIM)
    with timed:
        rc = _cabi.load().mvoc_attn_inject_fwd(q.data_ptr(), k.data_ptr(), v.data_ptr(), out.data_ptr(), *lds, n_obj,
                                               frames, pixels, heads, HEAD_DIM, mask.data_ptr(), kind, base,
                                               int(bool(temporal)), int(bool(share_p)), float(scale), _dt(q),
                                               int(variant), _stream())
    _cabi.check(rc, "mvoc_attn_inject_fwd")
    _count(3 if (share_p and not temporal) else 2)
    return out


def feature_blend_(x: torch.Tensor, mask: torch.Tensor, n_obj: int, frames: int) -> None:
    """In-place hidden-state injection on x [n_branches*T, C, H, W]; mask [n_obj, T, H*W] uint8."""
    _need_cuda(x, mask)
    nb = n_obj + 3
    if x.dim() != 4 or not x.is_contiguous() or x.shape[0] != nb * frames:
        raise ValueError(f"feature_blend_: need contiguous [{nb}*{frames}, C, H, W], got {tuple(x.shape)}")
    C, HW = x.shape[1], x.shape[2] * x.shape[3]
    if mask.dtype != torch.uint8 or tuple(mask.shape) != (n_obj, frames, HW) or not mask.is_contiguous():
        raise ValueError(f"feature_blend_: mask must be contiguous uint8 [{n_obj}, {frames}, {HW}]")
    lib = _cabi.load()
    st = lib.mvoc_feature_blend(x.data_ptr(), n_obj, frames, C, HW, mask.data_ptr(), _dt(x), _stream())
    _cabi.check(st, "mvoc_feature_blend")
    _count()


_gn_ws: dict = {}


def groupnorm_silu(
    x: torch.Tensor,
    weight: torch.Tensor,
    bias: torch.Tensor,
    groups: int,
    eps: float,
    silu: bool,
    frames_per_stat: int = 1,
    out: Optional[torch.Tensor] = None,
) -> torch.Tensor:
    """GroupNorm(+SiLU) over x [N, C, *spatial]; statistics shared by `frames_per_stat` consecutive n."""
    _need_cuda(x, weight, bias, out)
    if not x.is_contiguous():
        raise ValueError("groupnorm_silu: x must be contiguous")
    N, C = x.shape[0], x.shape[1]
    S = x.numel() // (N * C)
    if out is None:
        out = torch.empty_like(x)
    lib = _cabi.load()
    need = lib.mvoc_groupnorm_workspace_bytes(N, groups)
    key = x.device.index
    ws = _gn_ws.get(key)
    if ws is None or ws.numel() < need:
        ws = torch.empty(max(need, 1 << 20), dtype=torch.uint8, device=x.device)
        _gn_ws[key] = ws
    if weight.dtype != x.dtype or bias.dtype != x.dtype:
        raise TypeError("groupnorm_silu: weight/bias dtype must match x")
    with _Timed(("groupnorm", N, C, S, frames_per_stat), 2.0 * x.numel() * x.element_size()):
        st = lib.mvoc_groupnorm_silu(x.data_ptr(), out.data_ptr(), weight.data_ptr(), bias.data_ptr(),
                                     N, C, S, groups, frames_per_stat, float(eps), int(bool(silu)),
                                     _dt(x), ws.data_ptr(), _stream())
    _cabi.check(st, "mvoc_groupnorm_silu")
    _count()
    return out


def latent_composite_(
    z: torch.Tensor,
    bg: torch.Tensor,
    objs: torch.Tensor,
    mask: Optional[torch.Tensor],
    unet_in: Optional[torch.Tensor],
    ratio: float,
    do_fusion: bool,
    obj_noise_fusion: bool = False,
) -> None:
    """Noise fusion of z [4,T,h,w]-shaped latents + concat into unet_in [n_obj+3, ...] (one launch)."""
    _need_cuda(z, bg, objs, mask, unet_in)
    E = z.numel()
    n_obj = objs.numel() // E
    for t in (z, bg, objs):
        if not t.is_contiguous():
            raise ValueError("latent_composite_: latents must be contiguous")
    thw = E // 4
    if mask is not None and (mask.dtype != torch.float32 or mask.numel() != n_obj * thw or not mask.is_contiguous()):
        raise ValueError(f"latent_composite_: mask must be contiguous float32 [{n_obj}, {thw}]")
    if unet_in is not None and (unet_in.numel() != (n_obj + 3) * E or not unet_in.is_contiguous()):
        raise ValueError("latent_composite_: unet_in must be contiguous [n_obj+3, E]")
    lib = _cabi.load()
    st = lib.mvoc_latent_composite(z.data_ptr(), bg.data_ptr(), objs.data_ptr(), _ptr(mask),
                                   _ptr(unet_in), n_obj, E, thw, float(ratio), int(bool(do_fusion)),
                                   int(bool(obj_noise_fusion)), _dt(z),
                                   _dt(unet_in) if unet_in is not None else _dt(z), _stream())
    _cabi.check(st, "mvoc_latent_composite")
    _count()


def cfg_ddim_step_(pred_uncond: torch.Tensor, pred_cond: Optional[torch.Tensor], x: torch.Tensor,
                   guidance: float, alpha_t: float, alpha_prev: float) -> None:
    """x <- DDIM(v-pred, eta=0) step using v = u + g (c - u); in place on x."""
    _need_cuda(pred_uncond, pred_cond, x)
    if not (pred_uncond.is_contiguous() and x.is_contiguous() and (pred_cond is None or pred_cond.is_contiguous())):
        raise ValueError("cfg_ddim_step_: tensors must be contiguous")
    lib = _cabi.load()
    st = lib.mvoc_cfg_ddim_step(pred_uncond.data_ptr(), _ptr(pred_cond), x.data_ptr(), x.numel(),
                                float(guidance), float(alpha_t), float(alpha_prev),
                                _dt(pred_uncond), _dt(x), _stream())
    _cabi.check(st, "mvoc_cfg_ddim_step")
    _count()


def ddim_inverse_step_(pred_uncond: torch.Tensor, pred_cond: Optional[torch.Tensor], x: torch.Tensor,
                       guidance: float, alpha_src: float, alpha_dst: float) -> None:
    """x <- inverse-DDIM step from level alpha_src to alpha_dst; in place on x."""
    _need_cuda(pred_uncond, pred_cond, x)
    if not (pred_uncond.is_contiguous() and x.is_contiguous() and (pred_cond is None or pred_cond.is_contiguous())):
        raise ValueError("ddim_inverse_step_: tensors must be contiguous")
    lib = _cabi.load()
    st = lib.mvoc_ddim_inverse_step(pred_uncond.data_ptr(), _ptr(pred_cond), x.data_ptr(), x.numel(),
                                    float(guidance), float(alpha_src), float(alpha_dst),
                                    _dt(pred_uncond), _dt(x), _stream())
    _cabi.check(st, "mvoc_ddim_inverse_step")
    _count()


# --------------------------------------------------------------------------
# channels-last (NHWC) path
# --------------------------------------------------------------------------
_gnh_geom: dict = {}
_gnh_bufs: dict = {}


def _gnh_geometry(S: int, C: int, dt: int):
    key = (S, C, dt)
    g = _gnh_geom.get(key)
    if g is None:
        import ctypes

        chunks, tpc = ctypes.c_int(0), ctypes.c_int64(0)
        _cabi.check(_cabi.load().mvoc_groupnorm_nhwc_geometry(S, C, dt, ctypes.byref(chunks), ctypes.byref(tpc)),
                    "mvoc_groupnorm_nhwc_geometry")
        g = (chunks.value, tpc.value)
        _gnh_geom[key] = g
    return g


def _groupnorm_nhwc_slab(
    x: torch.Tensor,
    weight: torch.Tensor,
    bias: torch.Tensor,
    groups: int,
    eps: float,
    silu: bool,
    frames_per_stat: int = 1,
    add: Optional[torch.Tensor] = None,
    out: Optional[torch.Tensor] = None,
    gather=None,
) -> torch.Tensor:
    """GroupNorm(+SiLU) over channels-last x [N, S, C] (or [N, H, W, C]); `add` [N, C] is added to x first
    (the resnet time embedding).  `gather(partial [N,G,chunks,2]) -> [sets,N,G,chunks,2]` merges the
    statistics of pixel shards living on other GPUs (mvoc_b200.parallel); None on a single GPU."""
    _need_cuda(x, weight, bias, add, out)
    if not x.is_contiguous():
        raise ValueError("groupnorm_nhwc: x must be contiguous [N, ..., C]")
    N, C = x.shape[0], x.shape[-1]
    S = x.numel() // (N * C)
    if out is None:
        out = torch.empty_like(x)
    if add is not None and (tuple(add.shape) != (N, C) or not add.is_contiguous() or add.dtype != x.dtype):
        raise ValueError(f"groupnorm_nhwc: add must be contiguous [{N}, {C}] of x's dtype")
    dt = _dt(x)
    lib = _cabi.load()
    chunks, tpc = _gnh_geometry(S, C, dt)
    partial = torch.empty((N, groups, chunks, 2), dtype=torch.float32, device=x.device)
    with _Timed(("groupnorm", N, C, S, frames_per_stat), 2.0 * x.numel() * x.element_size()):
        _cabi.check(lib.mvoc_groupnorm_nhwc_stats(x.data_ptr(), _ptr(add), partial.data_ptr(), N, S, C, groups, dt,
                                                  _stream()), "mvoc_groupnorm_nhwc_stats")
        sets = 1
        if gather is not None:
            partial = gather(partial)
            sets = partial.shape[0]
        ckey = (x.device.index, S, C, groups, sets)
        counts = _gnh_bufs.get(ckey)
        if counts is None:
            cg = C // groups
            per = [float(max(0, min(S, (c + 1) * tpc) - c * tpc) * cg) for c in range(chunks)]
            counts = torch.tensor(per * sets, dtype=torch.float32, device=x.device)
            _gnh_bufs[ckey] = counts
        stat = torch.empty((N // frames_per_stat, groups, 2), dtype=torch.float32, device=x.device)
        _cabi.check(lib.mvoc_groupnorm_nhwc_finalize(partial.data_ptr(), counts.data_ptr(), stat.data_ptr(), N, groups,
                                                     chunks, frames_per_stat, sets, float(eps), _stream()),
                    "mvoc_groupnorm_nhwc_finalize")
        _cabi.check(lib.mvoc_groupnorm_nhwc_apply(x.data_ptr(), out.data_ptr(), weight.data_ptr(), bias.data_ptr(),
                                                  _ptr(add), stat.data_ptr(), N, S, C, groups, frames_per_stat,
                                                  int(bool(silu)), dt, _stream()), "mvoc_groupnorm_nhwc_apply")
    _count(3)
    return out


def groupnorm_nhwc(
    x: torch.Tensor,
    weight: torch.Tensor,
    bias: torch.Tensor,
    groups: int,
    eps: float,
    silu: bool,
    frames_per_stat: int = 1,
    add: Optional[torch.Tensor] = None,
    out: Optional[torch.Tensor] = None,
    gather=None,
) -> torch.Tensor:
    """GroupNorm(+SiLU) over channels-last x [N, S, C] (or [N, H, W, C]); see _groupnorm_nhwc_slab."""
    return _groupnorm_nhwc_slab(x, weight, bias, groups, eps, silu, frames_per_stat, add, out, gather)


def geglu(x: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """x [..., 2F] -> x[..., :F] * gelu(x[..., F:]) in one pass."""
    _need_cuda(x, out)
    if not x.is_contiguous():
        raise ValueError("geglu: x must be contiguous")
    F2 = x.shape[-1]
    F = F2 // 2
    M = x.numel() // F2
    if out is None:
        out = torch.empty(x.shape[:-1] + (F,), dtype=x.dtype, device=x.device)
    with _Timed(("geglu", M, F), 3.0 * M * F * x.element_size()):
        _cabi.check(_cabi.load().mvoc_geglu(x.data_ptr(), out.data_ptr(), M, F, _dt(x), _stream()), "mvoc_geglu")
    _count()
    return out


def upsample_nearest2x(x: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """x [N, H, W, C] channels-last -> [N, 2H, 2W, C], nearest neighbour (Upsample2D of the up blocks)."""
    _need_cuda(x, out)
    if x.dim() != 4 or not x.is_contiguous():
        raise ValueError("upsample_nearest2x: x must be a contiguous [N, H, W, C] tensor")
    N, H, W, C = x.shape
    if out is None:
        out = torch.empty((N, 2 * H, 2 * W, C), dtype=x.dtype, device=x.device)
    elif tuple(out.shape) != (N, 2 * H, 2 * W, C) or not out.is_contiguous() or out.dtype != x.dtype:
        raise ValueError("upsample_nearest2x: out must be a contiguous [N, 2H, 2W, C] tensor of x's dtype")
    with _Timed(("upsample2x", N, H, W, C), 5.0 * x.numel() * x.element_size()):
        _cabi.check(_cabi.load().mvoc_upsample_nearest2x_nhwc(x.data_ptr(), out.data_ptr(), N, H, W, C, _dt(x), _stream()),
                    "mvoc_upsample_nearest2x_nhwc")
    _count()
    return out


def concat_lastdim(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    """torch.cat([a, b], dim=-1) of two contiguous channels-last tensors [..., CA], [..., CB] (the up blocks' skip
    connections): one library copy kernel, bit-identical to torch.cat."""
    _need_cuda(a, b)
    if not (a.is_contiguous() and b.is_contiguous()) or a.shape[:-1] != b.shape[:-1] or a.dtype != b.dtype:
        raise ValueError(f"concat_lastdim: need contiguous tensors of one dtype with equal leading dims, got "
                         f"{tuple(a.shape)} {a.dtype} and {tuple(b.shape)} {b.dtype}")
    CA, CB = a.shape[-1], b.shape[-1]
    out = torch.empty(tuple(a.shape[:-1]) + (CA + CB,), dtype=a.dtype, device=a.device)
    rows = a.numel() // CA
    if rows == 0:
        return out                    # nothing to copy (an empty tensor has no data pointer to hand the kernel)
    with _Timed(("concat_lastdim", rows, CA, CB), 2.0 * out.numel() * out.element_size()):
        _cabi.check(_cabi.load().mvoc_concat_lastdim(a.data_ptr(), b.data_ptr(), out.data_ptr(), rows, CA, CB, _dt(a),
                                                     _stream()), "mvoc_concat_lastdim")
    _count()
    return out


def layernorm(x: torch.Tensor, weight: torch.Tensor, bias: torch.Tensor, eps: float,
              out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Row-wise LayerNorm over the last dim of a contiguous [..., C] tensor (warp per row)."""
    _need_cuda(x, weight, bias, out)
    if not x.is_contiguous():
        raise ValueError("layernorm: x must be contiguous")
    C = x.shape[-1]
    M = x.numel() // C
    if out is None:
        out = torch.empty_like(x)
    with _Timed(("layernorm", M, C), 2.0 * x.numel() * x.element_size()):
        _cabi.check(_cabi.load().mvoc_layernorm(x.data_ptr(), out.data_ptr(), weight.data_ptr(), bias.data_ptr(),
                                                M, C, float(eps), _dt(x), _stream()), "mvoc_layernorm")
    _count()
    return out


def temporal_attention_frames(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, heads: int, B: int, T: int,
                              S: int, scale: Optional[float] = None, out: Optional[torch.Tensor] = None):
    """Attention over the T frames of every (video, pixel) for row-major tokens in (b, t, pixel) order.
    q, k, v: [B*T*S, H*64] 2-D views (row stride arbitrary, e.g. slices of a fused QKV GEMM output);
    returns [B*T*S, H*64] in the same order — no (b t) <-> (b hw) permute is materialised."""
    import ctypes

    _need_cuda(q, k, v, out)
    C = heads * HEAD_DIM
    rows = B * T * S
    for t in (q, k, v):
        if t.dim() != 2 or t.shape[0] != rows or t.shape[1] != C or t.stride(1) != 1:
            raise ValueError(f"temporal_attention_frames: expected [{rows}, {C}] row-major views, got {tuple(t.shape)}")
    if out is None:
        out = torch.empty((rows, C), dtype=q.dtype, device=q.device)
    _check_io("temporal_attention_frames", out, (rows, C), q, k, v)
    if scale is None:
        scale = HEAD_DIM ** -0.5
    st = []
    for t in (q, k, v, out):
        rs = t.stride(0)
        st += [T * S * rs, rs, S * rs, HEAD_DIM]
    arr = (ctypes.c_int64 * 16)(*st)
    with _Timed(("attn_temporal", B * S, heads, T), 4.0 * rows * C * q.element_size()):
        rc = _cabi.load().mvoc_attn_temporal_strided_fwd(q.data_ptr(), k.data_ptr(), v.data_ptr(), out.data_ptr(),
                                                        B, S, T, heads, HEAD_DIM, arr, float(scale), _dt(q), _stream())
    _cabi.check(rc, "mvoc_attn_temporal_strided_fwd")
    _count()
    return out


# --------------------------------------------------------------------------
# dense work on tcgen05 tensor cores (csrc/gemm_tc.cu): convolutions, temporal convolutions, Linears
# --------------------------------------------------------------------------
# bit 0 = CTA pairs (tcgen05 cta_group::2); bits 8.. = tile-width override.  An experiment switch for A/B
# measurements (bench.py records it); the default is the configuration the product numbers were measured with.
GEMM_VARIANT = int(os.environ.get("MVOC_GEMM_VARIANT", "1") or 0)


def _rows(t: torch.Tensor, what: str):
    """(rows, row stride in elements) of a tensor whose leading dims collapse into uniformly strided rows."""
    if t.dim() < 2 or t.stride(-1) != 1:
        raise ValueError(f"{what}: need [..., C] with a contiguous last dim, got {tuple(t.shape)} strides {t.stride()}")
    ld = t.stride(-2)
    rows = t.shape[-2]
    for i in range(t.dim() - 3, -1, -1):
        if t.shape[i] != 1 and t.stride(i) != t.stride(i + 1) * t.shape[i + 1]:
            raise ValueError(f"{what}: leading dims of {tuple(t.shape)} (strides {t.stride()}) do not collapse into rows")
        rows *= t.shape[i]
    return rows, ld


def linear(x: torch.Tensor, weight: torch.Tensor, bias: Optional[torch.Tensor] = None,
           residual: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None,
           variant: Optional[int] = None) -> torch.Tensor:
    """out[..., N] = x[..., K] @ weight[N, K]^T (+ bias) (+ residual) in one tcgen05 kernel (mvoc_linear)."""
    _need_cuda(x, weight, bias, residual, out)
    N, K = weight.shape
    if x.shape[-1] != K or not weight.is_contiguous():
        raise ValueError(f"linear: x {tuple(x.shape)} vs contiguous weight {tuple(weight.shape)}")
    M, ldx = _rows(x, "linear x")
    if out is None:
        out = torch.empty(x.shape[:-1] + (N,), dtype=x.dtype, device=x.device)
    Mo, ldo = _rows(out, "linear out")
    ldr = 0
    if residual is not None:
        Mr, ldr = _rows(residual, "linear residual")
        if Mr != M or residual.shape[-1] != N:
            raise ValueError(f"linear: residual {tuple(residual.shape)} does not match [{M}, {N}]")
    if Mo != M or out.shape[-1] != N:
        raise ValueError(f"linear: out {tuple(out.shape)} does not match [{M}, {N}]")
    v = GEMM_VARIANT if variant is None else variant
    with _Timed(("gemm", "linear", M, K, N), 2.0 * M * K * N):
        rc = _cabi.load().mvoc_linear(x.data_ptr(), weight.data_ptr(), _ptr(bias), _ptr(residual), out.data_ptr(),
                                      M, K, N, ldx, ldr, ldo, _dt(x), int(v), _stream())
    _cabi.check(rc, "mvoc_linear")
    _count()
    return out


def linear_geglu(x: torch.Tensor, weight: torch.Tensor, bias: Optional[torch.Tensor] = None,
                 out: Optional[torch.Tensor] = None, variant: Optional[int] = None) -> torch.Tensor:
    """GEGLU projection with the gate in the GEMM epilogue: x [..., K], weight [2F, K] -> [..., F]."""
    _need_cuda(x, weight, bias, out)
    F2, K = weight.shape
    F = F2 // 2
    if x.shape[-1] != K or not x.is_contiguous() or not weight.is_contiguous():
        raise ValueError(f"linear_geglu: contiguous x {tuple(x.shape)} vs weight {tuple(weight.shape)}")
    M = x.numel() // K
    if out is None:
        out = torch.empty(x.shape[:-1] + (F,), dtype=x.dtype, device=x.device)
    v = GEMM_VARIANT if variant is None else variant
    with _Timed(("gemm", "geglu", M, K, F2), 2.0 * M * K * F2):
        rc = _cabi.load().mvoc_linear_geglu(x.data_ptr(), weight.data_ptr(), _ptr(bias), out.data_ptr(), M, K, F,
                                            _dt(x), int(v), _stream())
    _cabi.check(rc, "mvoc_linear_geglu")
    _count()
    return out


def linear_gelu(x: torch.Tensor, weight: torch.Tensor, bias: Optional[torch.Tensor] = None,
                out: Optional[torch.Tensor] = None, variant: Optional[int] = None) -> torch.Tensor:
    """out[..., N] = gelu(x[..., K] @ weight[N, K]^T (+ bias)) with the exact (erf) GELU in the tcgen05 GEMM epilogue
    (mvoc_linear_gelu): the CLIP image tower's mlp.fc1 + activation."""
    _need_cuda(x, weight, bias, out)
    N, K = weight.shape
    if x.shape[-1] != K or not weight.is_contiguous():
        raise ValueError(f"linear_gelu: x {tuple(x.shape)} vs contiguous weight {tuple(weight.shape)}")
    M, ldx = _rows(x, "linear_gelu x")
    if out is None:
        out = torch.empty(x.shape[:-1] + (N,), dtype=x.dtype, device=x.device)
    Mo, ldo = _rows(out, "linear_gelu out")
    if Mo != M or out.shape[-1] != N:
        raise ValueError(f"linear_gelu: out {tuple(out.shape)} does not match [{M}, {N}]")
    v = GEMM_VARIANT if variant is None else variant
    with _Timed(("gemm", "gelu", M, K, N), 2.0 * M * K * N):
        rc = _cabi.load().mvoc_linear_gelu(x.data_ptr(), weight.data_ptr(), _ptr(bias), out.data_ptr(), M, K, N, ldx,
                                           ldo, _dt(x), int(v), _stream())
    _cabi.check(rc, "mvoc_linear_gelu")
    _count()
    return out


def conv_taps(weight: torch.Tensor) -> torch.Tensor:
    """Conv2d weight [Cout, Cin, 3, 3] -> tap-major K-major [9, Cout, Cin]; Conv3d weight [Cout, Cin, 3, 1, 1] ->
    [3, Cout, Cin] (the operand layout of mvoc_conv3x3_nhwc / mvoc_temporal_conv3)."""
    if weight.dim() == 5:
        co, ci, kt, kh, kw = weight.shape
        if (kt, kh, kw) != (3, 1, 1):
            raise ValueError("conv_taps: Conv3d kernels must be (3, 1, 1)")
        return weight.reshape(co, ci, 3).permute(2, 0, 1).contiguous()
    co, ci, kh, kw = weight.shape
    if (kh, kw) != (3, 3):
        raise ValueError("conv_taps: Conv2d kernels must be 3x3")
    return weight.permute(2, 3, 0, 1).reshape(9, co, ci).contiguous()


def conv3x3(x: torch.Tensor, w_taps: torch.Tensor, bias: Optional[torch.Tensor] = None,
            residual: Optional[torch.Tensor] = None, x2: Optional[torch.Tensor] = None,
            w2: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None,
            variant: Optional[int] = None) -> torch.Tensor:
    """3x3 / stride 1 / pad 1 convolution on channels-last x [N, H, W, Cin] with w_taps [9, Cout, Cin]
    (+ bias) (+ x2 [N, H, W, Cin2] @ w2 [Cout, Cin2]^T, the 1x1 shortcut) (+ residual [N, H, W, Cout])."""
    _need_cuda(x, w_taps, bias, residual, x2, w2, out)
    if x.dim() != 4 or not x.is_contiguous():
        raise ValueError(f"conv3x3: need contiguous [N, H, W, Cin], got {tuple(x.shape)}")
    N, H, W, ci = x.shape
    if w_taps.dim() != 3 or w_taps.shape[0] != 9 or w_taps.shape[2] != ci or not w_taps.is_contiguous():
        raise ValueError(f"conv3x3: w_taps must be contiguous [9, Cout, {ci}], got {tuple(w_taps.shape)}")
    co = w_taps.shape[1]
    ci2 = 0
    if (x2 is None) != (w2 is None):
        raise ValueError("conv3x3: x2 and w2 go together")
    if x2 is not None:
        ci2 = x2.shape[-1]
        if tuple(x2.shape) != (N, H, W, ci2) or not x2.is_contiguous() or tuple(w2.shape) != (co, ci2) \
                or not w2.is_contiguous():
            raise ValueError("conv3x3: x2 must be contiguous [N, H, W, Cin2] and w2 contiguous [Cout, Cin2]")
    if out is None:
        out = torch.empty((N, H, W, co), dtype=x.dtype, device=x.device)
    for t, nm in ((out, "out"), (residual, "residual")):
        if t is not None and (tuple(t.shape) != (N, H, W, co) or not t.is_contiguous()):
            raise ValueError(f"conv3x3: {nm} must be contiguous [{N}, {H}, {W}, {co}]")
    v = GEMM_VARIANT if variant is None else variant
    with _Timed(("gemm", "conv3x3", N * H * W, 9 * ci + ci2, co), 2.0 * N * H * W * co * (9 * ci + ci2)):
        rc = _cabi.load().mvoc_conv3x3_nhwc(x.data_ptr(), w_taps.data_ptr(), _ptr(bias), _ptr(residual), _ptr(x2),
                                            _ptr(w2), ci2, out.data_ptr(), N, H, W, ci, co, _dt(x), int(v), _stream())
    _cabi.check(rc, "mvoc_conv3x3_nhwc")
    _count()
    return out


def conv3x3_s2(x: torch.Tensor, w_taps: torch.Tensor, bias: Optional[torch.Tensor] = None,
               pad: Sequence[int] = (0, 1), out: Optional[torch.Tensor] = None,
               variant: Optional[int] = None) -> torch.Tensor:
    """3x3 / stride 2 convolution on channels-last x [N, H, W, Cin] with w_taps [9, Cout, Cin] (+ bias) ->
    [N, Ho, Wo, Cout], Ho = (H + pad[0] + pad[1] - 3) // 2 + 1.  pad = (zeros before, zeros after) each axis:
    (0, 1) is the VAE's Downsample2D (F.pad (0, 1, 0, 1), then an unpadded conv), (1, 1) torch's padding=1."""
    _need_cuda(x, w_taps, bias, out)
    if x.dim() != 4 or not x.is_contiguous():
        raise ValueError(f"conv3x3_s2: need contiguous [N, H, W, Cin], got {tuple(x.shape)}")
    N, H, W, ci = x.shape
    if w_taps.dim() != 3 or w_taps.shape[0] != 9 or w_taps.shape[2] != ci or not w_taps.is_contiguous():
        raise ValueError(f"conv3x3_s2: w_taps must be contiguous [9, Cout, {ci}], got {tuple(w_taps.shape)}")
    pb, pe = (int(p) for p in pad)
    if pb not in (0, 1) or pe not in (0, 1):
        raise ValueError(f"conv3x3_s2: pad {tuple(pad)} must be (0 or 1, 0 or 1)")
    Ho, Wo = ((n + pb + pe - 3) // 2 + 1 for n in (H, W))
    if Ho < 1 or Wo < 1:
        raise ValueError(f"conv3x3_s2: {H}x{W} with pad {tuple(pad)} leaves an empty output")
    co = w_taps.shape[1]
    if out is None:
        out = torch.empty((N, Ho, Wo, co), dtype=x.dtype, device=x.device)
    elif tuple(out.shape) != (N, Ho, Wo, co) or not out.is_contiguous():
        raise ValueError(f"conv3x3_s2: out must be contiguous [{N}, {Ho}, {Wo}, {co}]")
    v = GEMM_VARIANT if variant is None else variant
    with _Timed(("gemm", "conv3x3_s2", N * Ho * Wo, 9 * ci, co), 2.0 * N * Ho * Wo * co * 9 * ci):
        rc = _cabi.load().mvoc_conv3x3_s2_nhwc(x.data_ptr(), w_taps.data_ptr(), _ptr(bias), out.data_ptr(), N, H, W,
                                               ci, co, pb, pe, _dt(x), int(v), _stream())
    _cabi.check(rc, "mvoc_conv3x3_s2_nhwc")
    _count()
    return out


def temporal_conv3(x: torch.Tensor, w_taps: torch.Tensor, bias: Optional[torch.Tensor], videos: int, frames: int,
                   residual: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None,
                   variant: Optional[int] = None) -> torch.Tensor:
    """Conv3d (3,1,1) over the frames of frame-major channels-last rows: x [(b t), ..., Cin] -> [(b t), ..., Cout]."""
    _need_cuda(x, w_taps, bias, residual, out)
    if not x.is_contiguous() or x.shape[0] != videos * frames:
        raise ValueError(f"temporal_conv3: need contiguous [{videos}*{frames}, ..., Cin], got {tuple(x.shape)}")
    ci = x.shape[-1]
    if w_taps.dim() != 3 or w_taps.shape[0] != 3 or w_taps.shape[2] != ci or not w_taps.is_contiguous():
        raise ValueError(f"temporal_conv3: w_taps must be contiguous [3, Cout, {ci}], got {tuple(w_taps.shape)}")
    co = w_taps.shape[1]
    S = x.numel() // (videos * frames * ci)
    if out is None:
        out = torch.empty(x.shape[:-1] + (co,), dtype=x.dtype, device=x.device)
    for t, nm in ((out, "out"), (residual, "residual")):
        if t is not None and (t.numel() != videos * frames * S * co or not t.is_contiguous()):
            raise ValueError(f"temporal_conv3: {nm} must be contiguous with {videos * frames * S} rows of {co}")
    v = GEMM_VARIANT if variant is None else variant
    with _Timed(("gemm", "tconv3", videos * frames * S, 3 * ci, co), 2.0 * videos * frames * S * co * 3 * ci):
        rc = _cabi.load().mvoc_temporal_conv3(x.data_ptr(), w_taps.data_ptr(), _ptr(bias), _ptr(residual),
                                              out.data_ptr(), videos, frames, S, ci, co, _dt(x), int(v), _stream())
    _cabi.check(rc, "mvoc_temporal_conv3")
    _count()
    return out
