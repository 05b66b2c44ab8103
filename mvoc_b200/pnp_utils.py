"""MVOC's hook layer (i2vgen-xl/pnp_utils.py) over the B200 kernels — the drop-in boundary.

Same entry points, argument meaning and out-of-band state as the reference:
  register_time_all(model, t, mask)                         pnp_utils.py:48-166
  modify_diffuser_attention_forward(unet)                   pnp_utils.py:169-560
  register_spatial_attention_pnp(model, schedule, inject_background)   :563-715
  register_temp_attention_pnp(model, schedule, inject_background)      :718-897
  register_resnet_injection(model, schedule)                :900-1037
  register_temp_conv_injection(model, schedule)             :1040-1105
  register_out_conv_injection(model, schedule)              :1108-1159
Processors keep the diffusers AttnProcessor call signature (:565-575) and the attributes
``injection_schedule``, ``inject_background``, ``t``, ``mask``.

Differences that are deliberate (SURVEY App. B): ``// 5`` is generalised to ``n_obj + 3`` branches
(D1; identical for two objects); binary-mask blends are exact selects on u8 masks and the float-mask
blend is one fp32 lerp rounded once (D2); module indices are derived from the UNet layout instead of
being hard-coded, so reduced UNets work.  The blend + attention run as sm_100a kernels
(mvoc_qk_blend, mvoc_attn_fwd / mvoc_attn_temporal_fwd, mvoc_feature_blend); nothing here falls back
to torch math.
"""
from __future__ import annotations

from typing import List, Optional, Sequence, Tuple

import torch
import torch.nn.functional as F

from . import ops
from .unet3d import AttnProcessor2_0

MaskPair = Tuple[torch.Tensor, torch.Tensor]
SHARE_P_MIN_TOKENS = 2048      # spatial layers at least this long run the composite pair through the pair kernel


# --------------------------------------------------------------------------
# mask preparation (once per resolution, cached): token-ordered masks for the kernels
# --------------------------------------------------------------------------
class _MaskCache:
    """The reference re-materialises a [T,h,w,C] mask per object per layer per step
    (pnp_utils.py:648-656, :805-809).  The kernels read one value per token, so the nearest-resized,
    token-ordered masks are built once per (mask list, resolution, kind, shard) and reused.
    Token order is (frame, pixel) everywhere — the row order of the channels-last activations.

    Entries are found by the IDENTITY of the mask tensors (and their in-place version counters) and hold
    strong references to them, so an address recycled by the allocator can never alias a dead entry; every
    entry carries a serial number that CUDA-graph keys use (mvoc_b200.pipeline).  The store is a small LRU
    and is emptied by init_pnp."""

    MAX_ENTRIES = 8

    class _Entry:
        __slots__ = ("tensors", "versions", "serial", "derived")

        def __init__(self, tensors, serial):
            self.tensors = tensors
            self.versions = tuple(t._version for t in tensors)
            self.serial = serial
            self.derived = {}

        def matches(self, tensors) -> bool:
            return (len(tensors) == len(self.tensors)
                    and all(a is b for a, b in zip(tensors, self.tensors))
                    and all(t._version == v for t, v in zip(tensors, self.versions)))

    def __init__(self):
        self._entries = []
        self._serial = 0

    def clear(self) -> None:
        self._entries.clear()

    def __len__(self) -> int:
        return len(self._entries)

    def _entry(self, mask: Sequence[MaskPair]) -> "_MaskCache._Entry":
        tensors = tuple(t for pair in mask for t in (pair[0], pair[1]))
        for i, e in enumerate(self._entries):
            if e.matches(tensors):
                if i:
                    self._entries.insert(0, self._entries.pop(i))
                return e
        self._serial += 1
        e = self._Entry(tensors, self._serial)
        self._entries.insert(0, e)
        del self._entries[self.MAX_ENTRIES:]
        return e

    def handle(self, mask: Sequence[MaskPair]) -> "_MaskCache._Entry":
        """The cache entry of a mask list.  Captured CUDA graphs bake in the addresses of the derived token
        masks: they key on `handle.serial` and keep the handle alive so that an LRU eviction cannot free them."""
        return self._entry(mask)

    def tokens(self, mask, h, w, soft: bool, frames=None, pixels=None) -> torch.Tensor:
        """[n_obj, T'*S'] in (frame, pixel) order.  soft=False: uint8 from the BINARY masks
        (pnp_utils.py:648-651, :986-994); soft=True: float32 from the FLOAT masks (:805-809).  Both are
        nearest-resized from the latent resolution to (h, w); `frames` / `pixels` = (lo, hi) shard ranges."""
        store = self._entry(mask).derived
        key = ("soft" if soft else "bin", h, w, frames, pixels)
        out = store.get(key)
        if out is None:
            rows = []
            for mf, mb in mask:
                m = (mf if soft else mb)[0].to(torch.float32)            # [4,T,H,W]
                m = F.interpolate(m, size=(h, w), mode="nearest")[0]      # channel 0: [T,h,w]
                m = m.reshape(m.shape[0], h * w)
                if frames is not None:
                    m = m[frames[0]:frames[1]]
                if pixels is not None:
                    m = m[:, pixels[0]:pixels[1]]
                rows.append(m.reshape(-1) if soft else (m != 0).to(torch.uint8).reshape(-1))
            out = torch.stack(rows).contiguous()
            store[key] = out
        return out

    def feature_planes(self, mask, frames=None) -> torch.Tensor:
        """[n_obj, T', H*W] uint8 from the BINARY masks at full latent resolution (pnp_utils.py:986-994)."""
        store = self._entry(mask).derived
        key = ("feat", frames)
        out = store.get(key)
        if out is None:
            planes = [mb[0, 0].reshape(mb.shape[2], -1).to(torch.uint8) for _, mb in mask]
            if frames is not None:
                planes = [p_[frames[0]:frames[1]] for p_ in planes]
            out = torch.stack(planes).contiguous()
            store[key] = out
        return out


_MASKS = _MaskCache()


def _fires(obj) -> bool:
    """`self.t in self.injection_schedule or self.t == 1000` (pnp_utils.py:624, :778, :970, :1059, :1114)
    without a device sync: the schedule is turned into a Python set once."""
    sched = getattr(obj, "injection_schedule", None)
    if sched is None:
        return False
    cached = getattr(obj, "_schedule_cache", None)
    if cached is None or cached[0] is not sched:
        vals = sched.tolist() if isinstance(sched, torch.Tensor) else list(sched)
        cached = (sched, frozenset(int(v) for v in vals))
        obj._schedule_cache = cached
    t = int(obj.t)
    return t in cached[1] or t == 1000


def _partition(module):
    ctx = getattr(module, "ctx", None)
    par = ctx.parallel if ctx is not None else None
    return par if (par is not None and par.world > 1) else None


# --------------------------------------------------------------------------
# processors
# --------------------------------------------------------------------------
class _InjectingProcessor(AttnProcessor2_0):
    temporal = False

    def __call__(self, attn, hidden_states, encoder_hidden_states=None, attention_mask=None, temb=None,
                 height=None, width=None, scale: float = 1.0):
        """hidden_states: [n_branches * T', S', C] channels-last tokens, frames outermost inside a branch
        (spatial: T' = this rank's frames, S' = h*w; temporal: T' = all frames, S' = this rank's pixels)."""
        if encoder_hidden_states is not None or not _fires(self):
            return super().__call__(attn, hidden_states, encoder_hidden_states, attention_mask, temb, scale)
        mask = self.mask
        n_obj = len(mask)
        nb = n_obj + 3
        if hidden_states.shape[0] % nb != 0:
            raise ValueError(f"batch {hidden_states.shape[0]} is not divisible into n_obj+3={nb} branches")
        # ONE fused QKV projection, as on the stock layers: the kernels take the three column slices with their
        # row stride (the reference projects three times, :604-612)
        q, k, v = attn.qkv_self(hidden_states)
        par = _partition(attn)
        n_frames_total = mask[0][0].shape[2]
        frames = hidden_states.shape[0] // nb
        if self.temporal:
            if par is not None and attn.ctx.full_hw is not None:   # rows are this rank's pixel shard of (fh x fw)
                fh, fw = attn.ctx.full_hw
                tokens = _MASKS.tokens(mask, fh, fw, soft=True, pixels=par.pixel_range(fh * fw))
            else:
                tokens = _MASKS.tokens(mask, height, width, soft=True)           # float mask (:805)
        else:
            frm = par.frame_range(n_frames_total) if par is not None else None
            tokens = _MASKS.tokens(mask, height, width, soft=False, frames=frm)  # binary mask (:648)
        # blend (:628-672 / :782-850) + attention of every branch (:684 / :862) in one C-ABI call; on the large
        # spatial layers the uncond / cond pair shares one softmax (they receive the same Q', K': :664-668).  Measured
        # on B200 (profiles/r02_attn_pair.txt): 2.06 -> 1.91 ms per layer at 4096 tokens, a loss below 2048 tokens
        # (64-key blocks and a second launch cost more than the saved exponentials there).
        share_p = (not self.temporal) and hidden_states.shape[1] >= SHARE_P_MIN_TOKENS
        out = ops.attention_inject_(q, k, v, tokens, attn.heads, n_obj, frames, bool(self.inject_background),
                                    self.temporal, share_p=share_p)
        return attn.out_proj(out)                                               # :692 (+ the block's skip add)


def register_spatial_attention_pnp(model, injection_schedule, inject_background=False):
    class ModifiedSpaAttnProcessor(_InjectingProcessor):
        temporal = False

    for bi, li in injected_attention_sites(model.unet):
        module = model.unet.up_blocks[bi].attentions[li].transformer_blocks[0].attn1
        p = ModifiedSpaAttnProcessor()
        setattr(p, "injection_schedule", injection_schedule)
        setattr(p, "inject_background", inject_background)
        module.processor = p


def register_temp_attention_pnp(model, injection_schedule, inject_background=False):
    class ModifiedTmpAttnProcessor(_InjectingProcessor):
        temporal = True

    for bi, li in injected_attention_sites(model.unet):
        module = model.unet.up_blocks[bi].temp_attentions[li].transformer_blocks[0].attn1
        p = ModifiedTmpAttnProcessor()
        setattr(p, "injection_schedule", injection_schedule)
        setattr(p, "inject_background", inject_background)
        module.processor = p


def injected_attention_sites(unet):
    """res_dict = {1: [1, 2], 2: [0, 1, 2], 3: [0, 1, 2]} (pnp_utils.py:706, :889) expressed on the layout:
    every cross-attention up block, skipping layer 0 of the lowest-resolution one (comment at :707)."""
    sites, first = [], True
    for bi, blk in enumerate(unet.up_blocks):
        if not getattr(blk, "has_cross_attention", False):
            continue
        for li in range(len(blk.attentions)):
            if first and li == 0:
                continue
            sites.append((bi, li))
        first = False
    return sites


# --------------------------------------------------------------------------
# feature (conv) injection
# --------------------------------------------------------------------------
def _feature_hook(module, hidden_states):
    """Blend of the composite slots from the background slot + objects, in place
    (pnp_utils.py:970-1004 / :1059-1082 / :1114-1146).  hidden_states is channels-last
    [n_branches*T', H, W, C] (resnet / temporal conv) or NCHW [n_branches*T', 4, H, W] (conv_out)."""
    if not _fires(module):
        return
    mask = module.mask
    n_obj = len(mask)
    nb = n_obj + 3
    if hidden_states.shape[0] % nb != 0:
        raise ValueError(f"batch {hidden_states.shape[0]} is not divisible into n_obj+3={nb} branches")
    frames = hidden_states.shape[0] // nb
    n_frames_total = mask[0][0].shape[2]
    par = _partition(module)
    frm = par.frame_range(n_frames_total) if par is not None else None
    if getattr(module, "feature_layout", "nhwc") == "nchw":
        ops.feature_blend_(hidden_states, _MASKS.feature_planes(mask, frm), n_obj, frames)
    else:
        H, W = hidden_states.shape[1], hidden_states.shape[2]
        # a binary-mask blend of channels-last rows is the same select as the Q/K blend with base = slot 0
        ops.qk_blend_(hidden_states, None, _MASKS.tokens(mask, H, W, soft=False, frames=frm), n_obj, True)


def register_resnet_injection(model, injection_schedule):
    blk = model.unet.up_blocks[-1]          # up_blocks_id = [3]  (pnp_utils.py:1031)
    for m in blk.resnets:
        m.feature_hook = _feature_hook
        setattr(m, "injection_schedule", injection_schedule)


def register_temp_conv_injection(model, injection_schedule):
    blk = model.unet.up_blocks[-1]          # pnp_utils.py:1099
    for m in blk.temp_convs:
        m.feature_hook = _feature_hook
        setattr(m, "injection_schedule", injection_schedule)


def register_out_conv_injection(model, injection_schedule):
    m = model.unet.conv_out                 # pnp_utils.py:1157
    m.feature_hook = _feature_hook
    m.feature_layout = "nchw"               # 4 channels: blended after the cast back to [N,4,H,W]
    m.ctx = model.unet.ctx
    setattr(m, "injection_schedule", injection_schedule)


def modify_diffuser_attention_forward(unet):
    """The reference re-points the forward of every TransformerTemporalModel / BasicTransformerBlock /
    Attention / Transformer2DModel so that height/width reach the processors (pnp_utils.py:550-560).
    The modules of mvoc_b200.unet3d already implement exactly those forwards; this validates the tree
    instead of patching it."""
    from .unet3d import Attention, BasicTransformerBlock, Transformer2DModel, TransformerTemporalModel

    n = 0
    for _, module in unet.named_modules():
        if isinstance(module, (Attention, BasicTransformerBlock, Transformer2DModel, TransformerTemporalModel)):
            n += 1
    if n == 0:
        raise TypeError("modify_diffuser_attention_forward: not an mvoc_b200.unet3d.I2VGenXLUNet")
    return unet


# --------------------------------------------------------------------------
# per-step state broadcast
# --------------------------------------------------------------------------
def register_time_all(model, t, mask):
    """setattr(module, 't'/'mask') on every hook site (pnp_utils.py:48-166), walking the layout."""
    unet = model.unet
    t = int(t)
    for blk in unet.up_blocks:                                   # :50-62
        for m in list(blk.resnets) + list(blk.temp_convs):
            setattr(m, "t", t)
            setattr(m, "mask", mask)
    for blk in list(unet.down_blocks) + [unet.mid_block] + list(unet.up_blocks):   # :64-156
        if not getattr(blk, "has_cross_attention", False):
            continue
        for tr in list(blk.attentions) + list(blk.temp_attentions):
            tb = tr.transformer_blocks[0]
            for a in (tb.attn1, tb.attn2):
                setattr(a.processor, "t", t)
                setattr(a.processor, "mask", mask)
    for m in (unet.conv_out, unet.conv_in):                      # :158-166
        setattr(m, "t", t)
        setattr(m, "mask", mask)


def _hook_sites(unet, pred) -> tuple:
    """One bool per hook site, in one fixed order: whether the site carries an injection hook and `pred(site)`."""
    sig = []
    blk = unet.up_blocks[-1]
    for m in list(blk.resnets) + list(blk.temp_convs) + [unet.conv_out]:
        sig.append(getattr(m, "feature_hook", None) is not None and pred(m))
    for bi, li in injected_attention_sites(unet):
        for grp in ("attentions", "temp_attentions"):
            p = getattr(unet.up_blocks[bi], grp)[li].transformer_blocks[0].attn1.processor
            sig.append(isinstance(p, _InjectingProcessor) and pred(p))
    return tuple(sig)


def hook_signature(unet) -> tuple:
    """Which hooks fire at the `t` last pushed by register_time_all — the control-flow key of one UNet
    forward (CUDA-graph capture in mvoc_b200.pipeline is keyed on it)."""
    return _hook_sites(unet, lambda m: hasattr(m, "t") and _fires(m))


def _scheduled(obj) -> bool:
    sched = getattr(obj, "injection_schedule", None)
    return sched is not None and len(sched) > 0


def injection_installed(unet) -> tuple:
    """Per hook site of hook_signature (the same walk, the same order): whether an injection hook with a non-empty
    schedule is installed, whatever `t` was pushed last.  The plain sampling loop (I2VGenXLPipeline.sample) refuses a
    UNet where any is."""
    return _hook_sites(unet, _scheduled)


def register_time(model, t):
    """Older helper kept for API parity (pnp_utils.py:36-45)."""
    for bi, li in injected_attention_sites(model.unet):
        for grp in ("attentions", "temp_attentions"):
            p = getattr(model.unet.up_blocks[bi], grp)[li].transformer_blocks[0].attn1.processor
            setattr(p, "t", int(t))
