"""CPU-side tests: C-ABI surface, host logic (scheduler, config, injection sites), oracle unit pins."""
import argparse
import ctypes
import json
import os
import re
from types import SimpleNamespace

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ------------------------------------------------------------------ C-ABI
def test_library_exports_every_declared_symbol():
    """The .so loads (no GPU needed) and exports exactly what include/mvoc_b200.h declares."""
    from mvoc_b200 import _cabi

    hdr = open(os.path.join(ROOT, "include", "mvoc_b200.h")).read()
    declared = set(re.findall(r"\b(mvoc_[a-z0-9_]+)\s*\(", hdr))
    assert declared, "no declarations found"
    assert declared == set(_cabi.SIGNATURES), (declared ^ set(_cabi.SIGNATURES))
    lib = _cabi.load()
    for name in declared:
        assert hasattr(lib, name), name
    assert "sm_100a" in _cabi.version()
    assert lib.mvoc_groupnorm_workspace_bytes(80, 32) >= 80 * 32 * 8


def test_argument_errors_are_reported_without_a_gpu():
    """Validation happens before any CUDA call: bad arguments return an error code + message."""
    from mvoc_b200 import _cabi

    lib = _cabi.load()
    rc = lib.mvoc_attn_fwd(None, None, None, None, 1, 1, 128, 128, 64, *([0] * 12), 0.125, 0, 0, None)
    assert rc == -1 and b"null pointer" in lib.mvoc_last_error()
    rc = lib.mvoc_attn_fwd(16, 16, 16, 16, 1, 1, 128, 128, 48, *([0] * 12), 0.125, 0, 0, None)
    assert rc == -2 and b"head_dim" in lib.mvoc_last_error()
    rc = lib.mvoc_qk_blend(16, 16, 0, 10, 64, 16, 0, 2, 0, None)
    assert rc == -1 and b"n_obj" in lib.mvoc_last_error()
    rc = lib.mvoc_cfg_ddim_step(16, 16, 16, 7, 1.0, 0.5, 0.6, 0, 2, None)
    assert rc == -2 and b"multiple of 8" in lib.mvoc_last_error()
    inj = lambda **kw: lib.mvoc_attn_inject_fwd(*[{**dict(q=16, k=16, v=16, o=16, ldq=128, ldk=128, ldv=128, ldo=128,
                                                          n_obj=2, frames=2, pixels=256, H=2, D=64, mask=16, kind=0,
                                                          base=4, mode=0, share_p=0, scale=0.125, dtype=0, variant=0,
                                                          stream=None), **kw}[n] for n in
                                                  ("q", "k", "v", "o", "ldq", "ldk", "ldv", "ldo", "n_obj", "frames",
                                                   "pixels", "H", "D", "mask", "kind", "base", "mode", "share_p", "scale",
                                                   "dtype", "variant", "stream")])
    assert inj(q=None) == -1 and b"null pointer" in lib.mvoc_last_error()
    assert inj(n_obj=0) == -1 and b"n_obj" in lib.mvoc_last_error()
    assert inj(mode=2) == -1 and b"mode" in lib.mvoc_last_error()
    assert inj(mode=1, share_p=1) == -2 and b"share_p" in lib.mvoc_last_error()     # temporal kernel is HBM-bound
    assert inj(ldq=100) == -1 and b"row stride" in lib.mvoc_last_error()
    rc = lib.mvoc_attn_pair_fwd(16, 16, 16, 16, 1, 1, 128, 128, 64, *([0] * 12), 0, 0.125, 0, 0, None)
    assert rc == -1 and b"pair_batches" in lib.mvoc_last_error()
    # the tcgen05 GEMM family validates shapes before touching the device
    rc = lib.mvoc_linear(16, 16, None, None, 16, 128, 100, 64, 100, 0, 64, 0, 0, None)
    assert rc == -2 and b"K=100" in lib.mvoc_last_error()
    rc = lib.mvoc_linear(16, 16, None, None, 16, 128, 64, 64, 32, 0, 64, 0, 0, None)
    assert rc == -1 and b"leading dimensions" in lib.mvoc_last_error()
    rc = lib.mvoc_conv3x3_nhwc(16, 16, None, None, None, None, 0, 16, 1, 8, 8, 48, 64, 0, 0, None)
    assert rc == -2 and b"multiple of 64" in lib.mvoc_last_error()
    rc = lib.mvoc_conv3x3_nhwc(16, 16, None, None, 16, None, 64, 16, 1, 8, 8, 64, 64, 0, 0, None)
    assert rc == -1 and b"x2 and w2" in lib.mvoc_last_error()
    rc = lib.mvoc_temporal_conv3(16, 16, None, None, 16, 1, 0, 64, 64, 64, 0, 0, None)
    assert rc == -1 and b"empty problem" in lib.mvoc_last_error()
    rc = lib.mvoc_linear_geglu(16, 16, None, 16, 128, 64, 96, 0, 0, None)
    assert rc == -2 and b"multiple of 64" in lib.mvoc_last_error()
    rc = lib.mvoc_linear(16, 16, None, None, 16, 128, 64, 64, 64, 0, 64, 2, 0, None)
    assert rc == -2 and b"dtype" in lib.mvoc_last_error()                           # fp32 storage is not supported
    rc = lib.mvoc_upsample_nearest2x_nhwc(16, 16, 2, 8, 8, 60, 0, None)
    assert rc == -2 and b"multiple of 8" in lib.mvoc_last_error()
    rc = lib.mvoc_upsample_nearest2x_nhwc(16, None, 2, 8, 8, 64, 0, None)
    assert rc == -1 and b"null pointer" in lib.mvoc_last_error()


@pytest.mark.parametrize("operand", [0, 1, 2])
def test_attention_rejects_zero_strides_where_the_extent_is_above_one(operand):
    """q, k and v are read through TMA, which cannot broadcast: a zero batch stride (B = 2) or token stride (N > 1) of
    q, k or v is refused before any CUDA call, whichever operand carries it."""
    from mvoc_b200 import _cabi

    lib = _cabi.load()
    name = b"qkv"[operand:operand + 1]

    def refused(entry):
        err = lib.mvoc_last_error()
        return entry in err and name + b" stride" in err

    B, H, N = 2, 2, 128
    st = [N * H * 64, H * 64, 64] * 4
    st[3 * operand] = 0                                                  # batch stride of q, k or v
    assert lib.mvoc_attn_fwd(16, 16, 16, 16, B, H, N, N, 64, *st, 0.125, 0, 0, None) == -2
    assert refused(b"mvoc_attn_fwd")
    assert lib.mvoc_attn_pair_fwd(16, 16, 16, 16, B, H, N, N, 64, *st, 1, 0.125, 0, 0, None) == -2
    assert refused(b"mvoc_attn_pair_fwd")
    for zero in (2 * operand, 2 * operand + 1):                          # batch, then token stride
        st = [N * 512, 512] * 4
        st[zero] = 0
        assert lib.mvoc_attn_d512_fwd(16, 16, 16, 16, B, N, 512, *st, 1.0, 0, None) == -2
        assert refused(b"mvoc_attn_d512_fwd")


def test_attention_pair_rejects_pair_batches_below_batches():
    """CTA b writes output batches b and b + pair_batches, so pair_batches < B would make two CTAs write one output
    batch: refused before any CUDA call by the pair entry and by the trace entry in pair mode."""
    from mvoc_b200 import _cabi

    lib = _cabi.load()
    B, H, N = 3, 2, 128
    st = [N * H * 64, H * 64, 64] * 4
    for pb in (1, 2):
        assert lib.mvoc_attn_pair_fwd(16, 16, 16, 16, B, H, N, N, 64, *st, pb, 0.125, 0, 0, None) == -1
        assert b"mvoc_attn_pair_fwd: pair_batches" in lib.mvoc_last_error()
        strides = (ctypes.c_int64 * 12)(*st)
        assert lib.mvoc_attn_fwd_trace(16, 16, 16, 16, B, H, N, N, 64, strides, pb, 0.125, 0, 0, 16, None) == -1
        assert b"mvoc_attn_fwd_trace: pair_batches" in lib.mvoc_last_error()


def test_gemm_tile_plan_host_logic():
    """mvoc_gemm_plan (no device call): what the GEMM entries choose.  On B200 a tcgen05.mma costs the same whatever
    N <= 256 is, so the plan minimises the NUMBER of column tiles: full 256-wide tiles plus one narrower tail tile;
    problems with fewer tiles than SMs get narrower tiles instead."""
    import ctypes

    from mvoc_b200 import _cabi

    lib = _cabi.load()

    def plan(rows, N, geglu=0, variant=1, sms=148):
        bn, pair, tail = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
        rc = lib.mvoc_gemm_plan(rows, N, geglu, variant, sms, ctypes.byref(bn), ctypes.byref(pair), ctypes.byref(tail))
        return rc, bn.value, pair.value, tail.value

    for rows in (327680, 81920, 20480):                      # config 2's levels 0-2 on one GPU
        assert plan(rows, 640) == (0, 256, 1, 128)           # 256 + 256 + 128, not 4 x 160
        assert plan(rows, 960) == (0, 256, 1, 192)
        assert plan(rows, 1920) == (0, 256, 1, 128)
        assert plan(rows, 1280) == (0, 256, 1, 0)
        rc, bn, pair, tail = plan(rows, 320)                 # two column tiles whichever way
        assert rc == 0 and pair == 1 and (tail == 320 - bn or (bn == 160 and tail == 0))
    assert plan(81920, 640, variant=3) == (0, 160, 1, 0)     # bit 1: only widths that divide N
    assert plan(81920, 640, variant=0)[2] == 0               # bit 0 clear: no CTA pairs
    assert plan(81920, 640, variant=1 | (192 << 8)) == (0, 192, 1, 64)   # forced width, tail covers the rest
    assert plan(327680, 1280, geglu=1) == (0, 256, 1, 0)     # GEGLU: value + gate columns share one 256-wide tile
    # the per-rank shapes of an 8-GPU run have fewer row tiles than the chip has SMs: narrower tiles fill more of them
    assert plan(640, 1280)[1] == 64 and plan(2560, 320)[1] == 64
    assert plan(640, 1280, sms=16)[1] == 256                 # ... unless the chip is small
    rc = plan(100, 100)[0]
    assert rc == -1 and b"multiple of 64" in lib.mvoc_last_error()


def test_product_ops_refuse_cpu_tensors():
    """No CPU fallback: the product raises instead of computing with torch."""
    from mvoc_b200 import ops

    q = torch.randn(1, 128, 64).bfloat16()
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.attention(q, q, q, 1)
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.groupnorm_silu(torch.randn(2, 32, 4, 4).bfloat16(), torch.ones(32).bfloat16(), torch.zeros(32).bfloat16(),
                           32, 1e-5, True)
    from mvoc_b200.unet3d import I2VGenXLUNet, UNetConfig

    m = I2VGenXLUNet(UNetConfig.reduced())
    with pytest.raises(RuntimeError, match="CUDA"):
        m(torch.randn(1, 4, 2, 8, 8), 1, torch.tensor([8]), torch.randn(1, 4, 2, 8, 8), torch.randn(1, 1, 1024),
          torch.randn(1, 77, 1024))


def test_product_never_imports_oracle():
    """Only tests/, __graft_entry__.smoke() and bench.py's CPU legs may touch oracle/."""
    for dirpath, _, files in os.walk(os.path.join(ROOT, "mvoc_b200")):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, re.M), f"{f} imports oracle"


# ------------------------------------------------------------------ scheduler
KNOWN_ALPHAS = {0: 0.999959, 1: 0.999913, 21: 0.997971, 501: 0.490706, 921: 0.0146935, 961: 0.00349756,
                981: 0.00078403, 999: 0.0}


def test_schedule_known_answers():
    """SURVEY App. A.6 known answers of the i2vgen-xl scheduler config."""
    from mvoc_b200.scheduler import DDIMSchedule
    from oracle import scheduler as osched

    s = DDIMSchedule(50)
    for t, a in KNOWN_ALPHAS.items():
        assert abs(s.alpha(t) - a) < 2e-6 * max(1.0, a / 1e-3), (t, s.alpha(t), a)
    assert s.timesteps[:4] == [981, 961, 941, 921] and s.timesteps[-1] == 1 and len(s.timesteps) == 50
    assert (s.alphas_cumprod == osched.alphas_cumprod().numpy()).all()
    inv = DDIMSchedule(500, inverse=True)
    assert inv.timesteps[:3] == [1, 3, 5] and inv.timesteps[-1] == 999
    assert set(s.timesteps) <= set(inv.timesteps)       # why inversion uses 500 steps
    assert inv.step_alphas(1) == (1.0, s.alpha(1))      # set_alpha_to_one below level 0
    o = osched.DDIMScheduler()
    o.set_timesteps(50)
    x = float(o.step(torch.tensor(0.5), 981, torch.tensor(1.0)))
    assert abs(x - 0.983932) < 2e-6                     # x=1, v=0.5, 981 -> 961
    # inverse then forward over the same pair of levels is the identity for a fixed prediction
    oi = osched.DDIMInverseScheduler()
    oi.set_timesteps(50)
    v = torch.tensor(0.3)
    x1 = oi.step(v, 21, torch.tensor(0.7))              # level 1 -> 21
    # map v (defined at level 1) to level 21 so that x0/eps are preserved, then step back
    a1, a21 = o.alphas_cumprod[1], o.alphas_cumprod[21]
    x0 = a1.sqrt() * 0.7 - (1 - a1).sqrt() * v
    eps = a1.sqrt() * v + (1 - a1).sqrt() * 0.7
    v21 = a21.sqrt() * eps - (1 - a21).sqrt() * x0
    back = o.step(v21, 21, x1)
    assert abs(float(back) - 0.7) < 1e-5


def test_init_pnp_schedules_follow_the_full_grid():
    """composite.py:39-52: k = int(n_steps * frac); schedule = timesteps[:k] of the FULL grid."""
    from mvoc_b200.pipeline import I2VGenXLPipeline, init_pnp
    from mvoc_b200.scheduler import DDIMSchedule
    from mvoc_b200.unet3d import I2VGenXLUNet, UNetConfig

    pipe = I2VGenXLPipeline(I2VGenXLUNet(UNetConfig.reduced()), "cpu")
    cfg = SimpleNamespace(n_steps=50, pnp_f_t=0.1, pnp_spatial_attn_t=0.5, pnp_temp_attn_t=0.0, inject_background=False)
    sch = init_pnp(pipe, DDIMSchedule(50), cfg)
    assert sch["conv"] == [981, 961, 941, 921, 901]
    assert len(sch["spatial"]) == 25 and sch["spatial"][-1] == 501
    assert sch["temporal"] == []          # an empty slice never fires
    from mvoc_b200 import pnp_utils

    blk = pipe.unet.up_blocks[-1]
    p = blk.attentions[1].transformer_blocks[0].attn1.processor
    assert type(p).__name__ == "ModifiedSpaAttnProcessor" and p.injection_schedule == sch["spatial"]
    # layer 0 of the lowest-resolution cross-attention up block keeps the stock processor (pnp_utils.py:706-707)
    assert type(blk.attentions[0].transformer_blocks[0].attn1.processor).__name__ == "AttnProcessor2_0"
    pnp_utils.register_time_all(pipe, 981, [])
    assert p.t == 981 and blk.resnets[0].t == 981 and pipe.unet.conv_out.t == 981
    p.t = 501
    assert pnp_utils._fires(p)
    p.t = 481
    assert not pnp_utils._fires(p)
    p.t = 1000
    assert pnp_utils._fires(p)            # `or self.t == 1000`


def test_full_unet_matches_published_parameter_count():
    from mvoc_b200.unet3d import I2VGenXLUNet, UNetConfig
    from oracle.unet import I2VGenXLUNet as OUNet, UNetConfig as OCfg

    with torch.device("meta"):
        p, o = I2VGenXLUNet(UNetConfig.full()), OUNet(OCfg.full())
    assert sum(x.numel() for x in p.parameters()) == 1_420_469_224
    assert sum(x.numel() for x in o.parameters()) == 1_420_469_224
    assert list(p.state_dict().keys()) == list(o.state_dict().keys())
    assert p.state_dict()["up_blocks.3.temp_convs.2.conv4.3.weight"].shape == (320, 320, 3, 1, 1)


# ------------------------------------------------------------------ config
def test_template_merge_and_interpolation(tmp_path):
    """OmegaConf subset used by the reference configs: deep merge, ${a} and ${a.b} interpolation, `active`."""
    from mvoc_b200 import config as cfg

    (tmp_path / "template.yaml").write_text(
        'seed: 6\ndata_dir: ".."\nmodel_name: "i2vgen-xl"\nvideo_name: "ReplaceMe"\n'
        'output_dir: "${data_dir}/Results/${model_name}/${video_name}/"\n'
        'n_steps: 50\npnp_f_t: 0.2\nfusion_step: [0, 3]\n'
        'frameinit_kwargs:\n  enable: true\n  filter_params:\n    method: "gaussian"\n    d_s: 0.25\n'
        'alias: "${frameinit_kwargs.filter_params.d_s}"\n')
    (tmp_path / "group.json").write_text(json.dumps([
        {"active": True, "video_name": "boat_surf", "pnp_f_t": 0.1, "fusion_step": [0, 1],
         "frameinit_kwargs": {"filter_params": {"d_s": 0.5}}},
        {"active": False, "video_name": "skipped"}]))
    out = list(cfg.iter_configs(str(tmp_path / "template.yaml"), str(tmp_path / "group.json")))
    assert len(out) == 1
    c = out[0]
    assert c.output_dir == "../Results/i2vgen-xl/boat_surf/"
    assert c.pnp_f_t == 0.1 and c.fusion_step == [0, 1] and c.n_steps == 50
    assert c.frameinit_kwargs.enable is True and c.frameinit_kwargs.filter_params.method == "gaussian"
    assert c.alias == 0.5                  # whole-value reference keeps the type


# ------------------------------------------------------------------ oracle unit pins
def _literal_two_object_spatial(query, key, masks, height, width, inject_background):
    """Literal transcription of pnp_utils.py:628-672 INCLUDING the hard-coded 5 (two objects only)."""
    import torch.nn.functional as F
    from einops import rearrange

    batch_size = query.shape[0]
    chunk_size = batch_size // 5
    query = rearrange(query.clone(), "b (h w) c -> b h w c", h=height)
    key = rearrange(key.clone(), "b (h w) c -> b h w c", h=height)
    if inject_background:
        q_inject, k_inject = query[:chunk_size], key[:chunk_size]
    else:
        q_inject, k_inject = query[4 * chunk_size:], key[4 * chunk_size:]
    for j, obj_mask_tensor in enumerate(masks):
        obj_q = query[chunk_size * (j + 1):chunk_size * (j + 2)]
        obj_k = key[chunk_size * (j + 1):chunk_size * (j + 2)]
        m = obj_mask_tensor[1].to(torch.float32)
        m = rearrange(m, "a b l h w -> (a b) l h w")
        m = F.interpolate(m, size=(height, width), mode="nearest")
        m = m[0]
        m = m.unsqueeze(-1).repeat(1, 1, 1, query.shape[-1])
        q_inject = q_inject * (1 - m) + obj_q * m
        k_inject = k_inject * (1 - m) + obj_k * m
    query[3 * chunk_size: 4 * chunk_size] = q_inject
    key[3 * chunk_size: 4 * chunk_size] = k_inject
    query[4 * chunk_size:] = q_inject
    key[4 * chunk_size:] = k_inject
    return rearrange(query, "b h w c -> b (h w) c"), rearrange(key, "b h w c -> b (h w) c")


@pytest.mark.parametrize("inject_background", [False, True])
def test_generalised_chunking_equals_the_hard_coded_five(inject_background):
    from mvoc_b200.synthetic import make_masks
    from oracle import ops_ref

    T, H, W, h, w, C = 4, 16, 16, 8, 8, 32
    masks = make_masks(2, T, H, W, seed=3)
    torch.manual_seed(0)
    q, k = torch.randn(5 * T, h * w, C), torch.randn(5 * T, h * w, C)
    a = ops_ref.spatial_qk_inject_ref(q, k, masks, h, w, inject_background)
    b = _literal_two_object_spatial(q, k, masks, h, w, inject_background)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    assert torch.equal(a[0][: 3 * T], q[: 3 * T])              # sources untouched
    assert torch.equal(a[0][3 * T: 4 * T], a[0][4 * T:])        # uncond == cond after injection


def test_nearest_resize_rule():
    """F.interpolate(mode='nearest') picks src = floor(dst * in / out), also for non-integer ratios."""
    from oracle import ops_ref

    m = torch.arange(2 * 32 * 32, dtype=torch.float32).view(2, 32, 32)
    for (h, w) in [(16, 16), (8, 8), (11, 20)]:
        r = ops_ref.nearest_mask(m, h, w)
        iy = torch.floor(torch.arange(h) * (32 / h)).long()
        ix = torch.floor(torch.arange(w) * (32 / w)).long()
        assert torch.equal(r, m[:, iy][:, :, ix])


def test_later_object_wins_on_overlap():
    from oracle import ops_ref

    T, H, W = 2, 8, 8
    full = torch.ones(1, 4, T, H, W, dtype=torch.bool)
    masks = [(full.float(), full), (full.float(), full)]
    x = torch.arange(5 * T, dtype=torch.float32).view(5 * T, 1, 1, 1).expand(5 * T, 3, H, W).contiguous()
    y = ops_ref.feature_inject_ref(x, masks)
    assert torch.equal(y[3 * T:4 * T], x[2 * T:3 * T]) and torch.equal(y[4 * T:], x[2 * T:3 * T])


def test_latent_fusion_keeps_background_outside_masks():
    from mvoc_b200.synthetic import make_masks
    from oracle import ops_ref

    masks = make_masks(2, 4, 16, 16, seed=1)
    z, bg = torch.randn(1, 4, 4, 16, 16), torch.randn(1, 4, 4, 16, 16)
    objs = [torch.randn(1, 4, 4, 16, 16) for _ in range(2)]
    out = ops_ref.latent_fusion_ref(z, bg, objs, [m for m, _ in masks], ratio=0.0)
    outside = (masks[0][0] == 0) & (masks[1][0] == 0)
    assert torch.equal(out[outside], bg[outside])              # r = 0: pure background outside every mask
    inside1 = masks[1][0] == 1
    assert torch.allclose(out[inside1], objs[1][inside1])


# ------------------------------------------------------------------ masks: host preparation vs reference / oracle
def test_mask_preprocess_matches_the_reference_function():
    """mvoc_b200.utils.mask_preprocess == the reference's utils.mask_preprocess (utils.py:92-154) on the PNG
    fixtures of tests/golden/masks (golden produced by the reference's own function, make_golden.py)."""
    from mvoc_b200.utils import mask_preprocess

    gdir = os.path.join(ROOT, "tests", "golden")
    gold = torch.load(os.path.join(gdir, "mask_preprocess.pt"), map_location="cpu")
    for name, path in (("dynamic", os.path.join(gdir, "masks", "dynamic")),
                       ("static", os.path.join(gdir, "masks", "static.png"))):
        mf, mb = mask_preprocess(path, "cpu", torch.float32, 1, 4, 4, downscale=8)
        rf, rb = gold[name]
        assert mf.shape == rf.shape == (1, 4, 4, 12, 16) and mb.dtype == torch.bool
        assert torch.equal(mf, rf) and torch.equal(mb, rb)
    # the dynamic folder holds 5 numbered files; frame 3 must be "003.png", not "010.png" (numeric sort + cut)
    assert not torch.equal(gold["dynamic"][0][0, 0, 3], gold["dynamic"][0][0, 0, 2])


def _emulate_qk_blend(x, tokens, n_obj, base_slot):
    """The contract of mvoc_qk_blend in include/mvoc_b200.h, in plain torch (test-side emulation)."""
    nb = n_obj + 3
    C = x.shape[-1]
    v = x.reshape(nb, -1, C).clone()
    acc = v[base_slot].clone()
    for j in range(n_obj):
        m = tokens[j].to(torch.float32)[:, None]
        if tokens.dtype == torch.uint8:
            acc = torch.where(m != 0, v[j + 1], acc)
        else:
            acc = acc * (1 - m) + v[j + 1] * m
    v[n_obj + 1] = acc
    v[n_obj + 2] = acc
    return v.reshape(x.shape)


@pytest.mark.parametrize("n_obj", [1, 2, 3])
@pytest.mark.parametrize("inject_background", [False, True])
def test_token_masks_reproduce_the_reference_injection(n_obj, inject_background):
    """Host-side mask preparation (nearest resize, (frame, pixel) token order, u8 / f32) fed through the
    kernel CONTRACT gives exactly the reference's spatial / temporal / feature injection."""
    from mvoc_b200 import pnp_utils
    from mvoc_b200.synthetic import make_masks
    from oracle import ops_ref

    T, H, W, h, w, C = 4, 16, 16, 8, 8, 16
    nb = n_obj + 3
    masks = make_masks(n_obj, T, H, W, seed=5)
    cache = pnp_utils._MaskCache()
    base = 0 if inject_background else n_obj + 2
    torch.manual_seed(1)
    # spatial: rows [nb*T, h*w, C]
    q = torch.randn(nb * T, h * w, C)
    ref_q, _ = ops_ref.spatial_qk_inject_ref(q, q.clone(), masks, h, w, inject_background)
    got = _emulate_qk_blend(q, cache.tokens(masks, h, w, soft=False), n_obj, base)
    assert torch.equal(got, ref_q)
    # temporal: the reference works on [(b h w), T, C]; the product keeps frame-major rows [(b t), h*w, C]
    qt = torch.randn(nb * h * w, T, C)
    ref_t, _ = ops_ref.temporal_qk_inject_ref(qt, qt.clone(), masks, h, w, inject_background)
    frame_major = qt.view(nb, h * w, T, C).permute(0, 2, 1, 3).reshape(nb * T, h * w, C)
    got_t = _emulate_qk_blend(frame_major, cache.tokens(masks, h, w, soft=True), n_obj, base)
    back = got_t.view(nb, T, h * w, C).permute(0, 2, 1, 3).reshape(nb * h * w, T, C)
    assert torch.allclose(back, ref_t, atol=1e-6)
    # features: NCHW in the reference, channels-last rows in the product, base = background always
    x = torch.randn(nb * T, C, H, W)
    ref_x = ops_ref.feature_inject_ref(x, masks)
    rows = x.permute(0, 2, 3, 1).reshape(nb * T, H * W, C)
    got_x = _emulate_qk_blend(rows, cache.tokens(masks, H, W, soft=False), n_obj, 0)
    assert torch.equal(got_x.view(nb * T, H, W, C).permute(0, 3, 1, 2), ref_x)
    planes = cache.feature_planes(masks)
    assert planes.shape == (n_obj, T, H * W) and planes.dtype == torch.uint8
    assert torch.equal(planes.view(n_obj, -1), cache.tokens(masks, H, W, soft=False))


def test_hook_signature_and_step_kinds():
    """Two hook configurations in the boat_surf schedule: conv + attention injection (steps 0-4), attention
    only (steps 5-49) => two captured graphs; computed without touching the GPU."""
    from mvoc_b200 import pnp_utils
    from mvoc_b200.pipeline import I2VGenXLPipeline, init_pnp
    from mvoc_b200.scheduler import DDIMSchedule
    from mvoc_b200.unet3d import I2VGenXLUNet, UNetConfig

    pipe = I2VGenXLPipeline(I2VGenXLUNet(UNetConfig.reduced()), "cpu")
    sched = DDIMSchedule(50)
    cfg = SimpleNamespace(n_steps=50, pnp_f_t=0.1, pnp_spatial_attn_t=1.0, pnp_temp_attn_t=1.0, inject_background=False)
    init_pnp(pipe, sched, cfg)
    assert pipe.step_kinds(sched.timesteps, []) == [0, 5]
    pnp_utils.register_time_all(pipe, 981, [])
    sig0 = pnp_utils.hook_signature(pipe.unet)
    pnp_utils.register_time_all(pipe, 21, [])
    sig1 = pnp_utils.hook_signature(pipe.unet)
    assert sig0 != sig1 and all(sig0) and any(sig1) and not all(sig1)
    cfg2 = SimpleNamespace(n_steps=50, pnp_f_t=0.2, pnp_spatial_attn_t=0.2, pnp_temp_attn_t=0.5, inject_background=False)
    init_pnp(pipe, sched, cfg2)
    assert pipe.step_kinds(sched.timesteps, []) == [0, 10, 25]


def test_latent_bank_and_wire_format(tmp_path):
    from mvoc_b200.pipeline import LatentBank, save_ddim_latents_at_t
    from mvoc_b200.utils import load_ddim_latents_at_T

    ts = [981, 961, 941]
    data = {t: torch.full((1, 4, 2, 4, 4), float(t)).half() for t in ts}
    for t, x in data.items():
        save_ddim_latents_at_t(x, t, str(tmp_path))
    assert sorted(os.listdir(tmp_path)) == ["ddim_latents_941.pt", "ddim_latents_961.pt", "ddim_latents_981.pt"]
    bank = LatentBank.from_dir(str(tmp_path), ts, "cpu")
    assert bank.data.shape == (3, 4, 2, 4, 4) and bank.data.dtype == torch.float32
    assert float(bank.at(961).mean()) == 961.0
    assert float(load_ddim_latents_at_T(str(tmp_path)).float().mean()) == 981.0


# ------------------------------------------------------------------ script / config contract
REF_CFG = os.path.join(ROOT, "tests", "golden", "reference_configs")


@pytest.mark.skipif(not os.path.isdir(REF_CFG), reason="the reference's config files are not stored under "
                    "tests/golden/reference_configs (tests/golden/make_golden.py copies them from a reference checkout)")
def test_reference_config_files_load_unchanged():
    """The reference's own template.yaml + group_config.json go through the loader and the path joins of
    composite.py:97-106 / inverse.py:143-150 without edits."""
    from mvoc_b200 import composite, config as cfgmod

    entries = list(cfgmod.iter_configs(f"{REF_CFG}/group_composite/template.yaml",
                                       f"{REF_CFG}/group_composite/group_config.json"))
    assert len(entries) == 7
    c = composite.resolve_paths(entries[0])
    assert c.video_name == "boat_surf" and c.image_size == [1280, 720]
    assert c.obj_mask_path == ["../demo/boat_surf/boat_mask", "../demo/boat_surf/surf_mask"]
    assert c.bg_ddim_latents_path == "../inversions/i2vgen-xl/boat_surf/ddim_latents"
    assert c.output_dir == "../Results/MVOC-Demo/i2vgen-xl/boat_surf/sailboat and surfing/"
    assert composite.latent_geometry(c) == (16, 90, 160)
    assert (c.pnp_f_t, c.pnp_spatial_attn_t, c.pnp_temp_attn_t, c.fusion_step) == (0.1, 1.0, 1.0, [0, 1])
    for e in entries:   # every shipped entry has exactly two objects (the reference's hard-coded // 5)
        assert len(e.obj_mask_path) == 2 and len(e.obj_ddim_latents_path) == 2
    inv = list(cfgmod.iter_configs(f"{REF_CFG}/group_inversion/template.yaml",
                                   f"{REF_CFG}/group_inversion/group_config.json"))
    assert inv and inv[0].inverse_config.n_steps == 500 and inv[0].inverse_config.cfg == 1.0
    assert inv[0].inverse_config.image_size == [1280, 720]          # ${image_size} keeps the list type
    assert inv[0].inverse_config.output_dir == "../inversions/i2vgen-xl/boat_surf/ddim_latents"
    assert inv[0].recon_config.ddim_latents_path == inv[0].inverse_config.output_dir


CFG = os.path.join(ROOT, "configs")


def test_shipped_config_files_load():
    """The template.yaml + group_config.json pairs under configs/ (the CLI defaults) go through the loader and the
    path joins of composite.py:97-106 / inverse.py:143-150 without edits."""
    from mvoc_b200 import composite, config as cfgmod

    entries = list(cfgmod.iter_configs(f"{CFG}/group_composite/template.yaml",
                                       f"{CFG}/group_composite/group_config.json"))
    assert len(entries) == 1                                        # the inactive entry is dropped
    c = composite.resolve_paths(entries[0])
    j = lambda *p: os.path.join(c.data_dir, *p)
    assert c.video_name == "synthetic_small" and c.image_size == [256, 128]
    assert c.obj_mask_path == [j("demo/synthetic_small/obj1_mask"), j("demo/synthetic_small/obj2_mask")]
    assert c.obj_ddim_latents_path == [j("inversions/i2vgen-xl/obj1/ddim_latents"),
                                       j("inversions/i2vgen-xl/obj2/ddim_latents")]
    assert c.bg_ddim_latents_path == j("inversions/i2vgen-xl/synthetic_small/ddim_latents")
    assert c.edited_first_frame_path == j("demo/synthetic_small/edited_first_frame/00000.png")
    assert c.video_path == j("demo", "synthetic_small.mp4")
    assert c.output_dir == f"{c.data_dir}/Results/MVOC-B200/i2vgen-xl/synthetic_small/bg plus two objects/"
    assert composite.latent_geometry(c) == (8, 16, 32)
    assert (c.pnp_f_t, c.pnp_spatial_attn_t, c.pnp_temp_attn_t, c.fusion_step) == (0.1, 1.0, 1.0, [0, 1])
    assert (c.n_steps, c.cfg, c.ddim_init_latents_t_idx, c.random_noise_ratio) == (50, 9.0, 0, 0.0)
    inv = list(cfgmod.iter_configs(f"{CFG}/group_inversion/template.yaml",
                                   f"{CFG}/group_inversion/group_config.json"))
    assert len(inv) == 1 and inv[0].video_name == "synthetic_small"
    assert inv[0].inverse_config.n_steps == 500 and inv[0].inverse_config.cfg == 1.0
    assert inv[0].inverse_config.image_size == [256, 128]           # ${image_size} keeps the list type
    assert inv[0].inverse_config.n_frames == 8                      # the entry's override reaches the nested key
    assert inv[0].inverse_config.output_dir == f"{inv[0].data_dir}/inversions/i2vgen-xl/synthetic_small/ddim_latents"
    assert inv[0].recon_config.ddim_latents_path == inv[0].inverse_config.output_dir


def test_cli_parsers_keep_the_reference_flags():
    from mvoc_b200 import composite, inverse

    a = composite.build_parser().parse_args(["--template_config", "t.yaml", "--configs_json", "c.json"])
    assert (a.template_config, a.configs_json) == ("t.yaml", "c.json")
    d = composite.build_parser().parse_args([])
    assert d.template_config == "./configs/group_composite/template.yaml"       # composite.py:229-235
    i = inverse.build_parser().parse_args([])
    assert i.configs_json == "./configs/group_inversion/group_config.json"      # inverse.py:231-235


def test_latent_bank_packed_round_trip(tmp_path):
    from mvoc_b200.pipeline import LatentBank

    data = {t: torch.randn(1, 4, 2, 4, 4) for t in (981, 1, 501)}
    bank = LatentBank(data, "cpu")
    p = str(tmp_path / "store" / "bank.pt")
    bank.save_packed(p)
    again = LatentBank.load_packed(p, "cpu")
    assert again.index == bank.index
    for t in data:
        assert torch.equal(again.at(t), data[t][0])


# ------------------------------------------------------------------ bench.py helpers (no GPU)
def test_bench_clock_sampler_parsing_and_peaks():
    import bench

    cs = bench.ClockSampler(0)
    cs.proc = SimpleNamespace(terminate=lambda: None, wait=lambda timeout=None: 0, kill=lambda: None)
    cs.lines = ["0, 1657, 1965, 990.12, Not Active, Not Active, Not Active, Active",
                "0, 1702, 1965, 975.00, Not Active, Not Active, Not Active, Active",
                "garbage line",
                "0, 1965, 1965, 300.00, Not Active, Not Active, Not Active, Not Active"]
    out = cs.stop()
    assert out["sm_mhz"] == 1702.0 and out["sm_max_mhz"] == 1965.0 and out["samples"] == 3
    assert out["reasons"] == ["sw_power_cap"]
    peaks = bench.measured_peaks()
    assert peaks["hbm_gbs"] > 1000 and peaks["bf16_tflops_sustained"] > 100 and peaks["_source"] in ("measured", "fallback")
    from mvoc_b200 import synthetic

    d = bench.workload_description(synthetic.WORKLOADS["config2"])
    assert "16 frames x 64x64" in d and "bg+2 objects" in d and "50-step" in d


def test_bench_reference_arm_contract(monkeypatch, capsys):
    """--impl reference prints the contract keys; non-zero ranks stay silent (the CPU work itself is faked)."""
    import json

    import bench
    from mvoc_b200 import synthetic

    class FakeSampler:
        def __init__(self, wl, budget):
            self.cores, self.desc, self.full = 4, "fake sample", synthetic.WORKLOADS[wl]

        def step(self):
            return 0.002, 0.5

    monkeypatch.setattr(bench, "CpuSampler", FakeSampler)
    args = SimpleNamespace(steps=3, warmup=1, gpus=2, workload="config2")
    monkeypatch.setenv("RANK", "1")
    bench.run_reference(args)
    assert capsys.readouterr().out == ""
    monkeypatch.setenv("RANK", "0")
    bench.run_reference(args)
    line = json.loads(capsys.readouterr().out)
    assert line["impl"] == "reference" and line["unit"] == "frames/s" and line["higher_is_better"] is True
    assert line["steps"] == 3 and line["value"] == pytest.approx(0.002)
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] == 4
    assert line["e2e"] == {"value": pytest.approx(0.002), "unit": "frames/s", "h2d_bytes_per_step": 0,
                           "d2h_bytes_per_step": 0}


def test_bench_steps_past_the_schedule_start_it_again():
    import bench

    assert bench.schedule_passes(3, 50) == [3]
    assert bench.schedule_passes(50, 50) == [50]
    assert bench.schedule_passes(120, 50) == [50, 50, 20]
    assert sum(bench.schedule_passes(1001, 500)) == 1001
    assert bench.positive_int("1") == 1
    with pytest.raises(argparse.ArgumentTypeError):
        bench.positive_int("0")


def test_bench_dump_outputs(tmp_path):
    import numpy as np

    import bench

    lat = torch.randn(1, 4, 2, 8, 8)
    bench.dump_outputs(str(tmp_path / "out"), {"latents": lat.bfloat16(), "exact": lat.double()})
    a = np.load(tmp_path / "out" / "latents.npy")
    b = np.load(tmp_path / "out" / "exact.npy")
    assert a.dtype == np.float32 and a.shape == (1, 4, 2, 8, 8)
    assert np.array_equal(a, lat.bfloat16().float().numpy())
    assert b.dtype == np.float64 and np.array_equal(b, lat.double().numpy())
    with pytest.raises(SystemExit, match="limit"):
        bench.dump_outputs(str(tmp_path / "big"), {"x": torch.empty(bench.DUMP_LIMIT_BYTES // 4 + 1)})
    assert not (tmp_path / "big").exists()


# ------------------------------------------------------------------ round-2 advisor findings
def test_mask_cache_never_aliases_recycled_addresses():
    """Two compositions with different masks of the SAME shape in one process: the token masks must follow the
    mask objects, not their addresses (the allocator hands a freed mask's address to the next one)."""
    from mvoc_b200 import pnp_utils

    cache = pnp_utils._MaskCache()
    for it in range(6):
        val = float(it % 2)
        mf = torch.full((1, 4, 2, 8, 8), val)
        mb = mf > 0.5
        tok = cache.tokens([(mf, mb)], 4, 4, soft=False)
        assert int(tok.sum()) == int(val) * tok.numel(), f"iteration {it}: stale token mask"
        soft = cache.tokens([(mf, mb)], 4, 4, soft=True)
        assert float(soft.sum()) == val * soft.numel()
        feat = cache.feature_planes([(mf, mb)])
        assert int(feat.sum()) == int(val) * feat.numel()
        del mf, mb, tok, soft, feat
    assert len(cache) <= cache.MAX_ENTRIES
    # the same objects hit the same entry; an in-place edit of a mask invalidates it
    mf = torch.zeros(1, 4, 2, 8, 8)
    mb = mf > 0.5
    h0 = cache.handle([(mf, mb)])
    assert cache.handle([(mf, mb)]) is h0
    mf.add_(1.0)
    assert cache.handle([(mf, mb)]) is not h0


def test_ops_refuse_tensors_of_another_device(monkeypatch):
    """The C-ABI launches on the current device: a tensor living elsewhere must raise, not launch."""
    from mvoc_b200 import ops

    class _T:
        is_cuda = True
        device = torch.device("cuda", 1)

    monkeypatch.setattr(torch.cuda, "current_device", lambda: 0)
    with pytest.raises(RuntimeError, match="current CUDA device"):
        ops._need_cuda(_T())


def test_scripts_fail_hard_on_missing_inputs(tmp_path):
    """composite.py / inverse.py: missing latents, masks, conditioning or weights are errors unless --synthetic."""
    from mvoc_b200 import composite, inverse

    cfg = SimpleNamespace(video_name="vid", get=lambda k, d=None: d)
    assert composite.conditioning_path("c/{video_name}.pt", cfg) == "c/vid.pt"
    assert composite.build_parser().parse_args([]).synthetic is False
    assert inverse.build_parser().parse_args(["--synthetic"]).synthetic is True
    assert inverse.inversion_complete(str(tmp_path / "nope"), 4) is False
    from mvoc_b200.pipeline import save_ddim_latents_at_t
    from mvoc_b200.scheduler import DDIMSchedule

    ts = DDIMSchedule(4, inverse=True).timesteps
    for t in ts[:-1]:
        save_ddim_latents_at_t(torch.zeros(1, 4, 2, 4, 4), t, str(tmp_path))
    assert inverse.inversion_complete(str(tmp_path), 4) is False          # a partial run is not "done"
    save_ddim_latents_at_t(torch.zeros(1, 4, 2, 4, 4), ts[-1], str(tmp_path))
    assert inverse.inversion_complete(str(tmp_path), 4) is True
    assert torch.load(os.path.join(str(tmp_path), f"ddim_latents_{int(ts[0])}.pt")).dtype == torch.float16
