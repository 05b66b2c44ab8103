"""CLIP image tower without a GPU: key layout and parameter count of the full-width model against transformers'
CLIPVisionModelWithProjection, the loader, the host model (kernels emulated in torch) against transformers in fp32,
the preprocessing, the argument checks of mvoc_attn_d80_fwd / mvoc_linear_gelu, and the scripts' CLIP paths."""
import os

import pytest
import torch
import torch.nn.functional as F

from tests import cpu_ops_emulation as emu

FULL_PARAMS = 632_076_800
FULL = dict(hidden_size=1280, intermediate_size=5120, num_hidden_layers=32, num_attention_heads=16, patch_size=14,
            image_size=224, projection_dim=1024)   # the reference checkpoint's image_encoder/config.json
# head_dim 80 like the checkpoint, widths multiples of 64 like the kernels need
SMALL = dict(hidden_size=320, intermediate_size=1280, num_hidden_layers=2, num_attention_heads=4, patch_size=14,
             image_size=224, projection_dim=128)


def _hf_model(**kw):
    transformers = pytest.importorskip("transformers")
    cfg = transformers.CLIPVisionConfig(hidden_act="gelu", layer_norm_eps=1e-5, **kw)
    cfg._attn_implementation = "eager"
    return transformers.CLIPVisionModelWithProjection(cfg).eval()


def _small_cfg():
    from mvoc_b200.clip import CLIPVisionConfig

    return CLIPVisionConfig(**SMALL)


def test_full_width_layout_and_parameter_count():
    from mvoc_b200.clip import CLIPVisionEncoder

    with torch.device("meta"):
        ours = CLIPVisionEncoder()
        ref = _hf_model(**FULL)
    mine = {k: tuple(v.shape) for k, v in ours.state_dict().items()}
    theirs = {k: tuple(v.shape) for k, v in ref.state_dict().items()}
    assert mine == theirs
    assert sum(v.numel() for v in ours.parameters()) == FULL_PARAMS
    assert "visual_projection.bias" not in mine and "vision_model.pre_layrnorm.weight" in mine


# ------------------------------------------------------------------ loader
@pytest.fixture()
def small_files(tmp_path):
    torch.manual_seed(0)
    sd = _hf_model(**SMALL).state_dict()
    from safetensors.torch import save_file

    pt, st = str(tmp_path / "clip.pt"), str(tmp_path / "clip.safetensors")
    torch.save(sd, pt)
    save_file({k: v.contiguous() for k, v in sd.items()}, st)
    return sd, pt, st


@pytest.mark.parametrize("fmt", ["pt", "safetensors"])
def test_loader_round_trip(small_files, fmt):
    from mvoc_b200.clip import load_clip_image_encoder

    sd, pt, st = small_files
    enc = load_clip_image_encoder(pt if fmt == "pt" else st, "cpu", torch.float32, cfg=_small_cfg())
    got = enc.state_dict()
    assert set(got) == set(sd) and all(torch.equal(got[k], sd[k]) for k in sd)
    assert all(k.startswith(("vision_model.", "visual_projection.")) for k in got)


def test_loader_accepts_text_tower_and_position_ids(small_files, tmp_path):
    from mvoc_b200.clip import load_clip_image_encoder

    sd, _, _ = small_files
    extra = dict(sd)
    extra["vision_model.embeddings.position_ids"] = torch.arange(257).view(1, -1)
    extra["text_projection.weight"] = torch.zeros(4, 4)
    extra["logit_scale"] = torch.tensor(1.0)
    p = str(tmp_path / "full.pt")
    torch.save(extra, p)
    load_clip_image_encoder(p, "cpu", torch.float32, cfg=_small_cfg())


def test_loader_names_the_bad_key(small_files, tmp_path):
    from mvoc_b200.clip import load_clip_image_encoder

    sd, _, _ = small_files
    key = "vision_model.encoder.layers.1.mlp.fc1.weight"
    missing = {k: v for k, v in sd.items() if k != key}
    torch.save(missing, tmp_path / "missing.pt")
    with pytest.raises(KeyError, match=key.replace(".", r"\.")):
        load_clip_image_encoder(str(tmp_path / "missing.pt"), "cpu", cfg=_small_cfg())
    bad = dict(sd)
    bad[key] = torch.zeros(7, 3)
    torch.save(bad, tmp_path / "shape.pt")
    with pytest.raises(ValueError, match=key.replace(".", r"\.")):
        load_clip_image_encoder(str(tmp_path / "shape.pt"), "cpu", cfg=_small_cfg())
    with pytest.raises(FileNotFoundError, match="CLIP image encoder"):
        load_clip_image_encoder(str(tmp_path / "absent.pt"), "cpu", cfg=_small_cfg())


# ------------------------------------------------------------------ host model with emulated kernels
def attention_d80(q, k, v, heads, scale=None, out=None):
    """The contract of mvoc_attn_d80_fwd: [B, N, H*80] views with a contiguous last dim and 16-byte strides."""
    for t in (q, k, v):
        assert t.dim() == 3 and t.shape[-1] == heads * 80 and t.stride(-1) == 1
        assert all(s % 8 == 0 for s in t.stride()[:-1])
    B, Nq, C = q.shape
    sp = lambda t: t.reshape(B, t.shape[1], heads, 80).transpose(1, 2)
    o = F.scaled_dot_product_attention(sp(q), sp(k), sp(v), scale=scale)
    return o.transpose(1, 2).reshape(B, Nq, C)


def linear_gelu(x, weight, bias=None, out=None, variant=None):
    n, k = weight.shape
    assert n % 64 == 0 and k % 64 == 0 and weight.is_contiguous() and x.stride(-1) == 1
    return F.gelu(F.linear(x, weight, bias))


@pytest.fixture()
def emulated_ops():
    from mvoc_b200 import ops

    saved = emu.install()
    extra = {n: getattr(ops, n) for n in ("attention_d80", "linear_gelu")}
    ops.attention_d80, ops.linear_gelu = attention_d80, linear_gelu
    yield
    for n, f in extra.items():
        setattr(ops, n, f)
    emu.uninstall(saved)


def _small_pair(seed=0):
    from mvoc_b200.clip import CLIPVisionEncoder

    torch.manual_seed(seed)
    ref = _hf_model(**SMALL)
    ours = CLIPVisionEncoder(_small_cfg()).eval()
    ours.load_state_dict(ref.state_dict(), strict=True)
    return ref, ours


def test_host_model_vs_transformers(emulated_ops):
    ref, ours = _small_pair()
    torch.manual_seed(1)
    x = torch.randn(3, 3, 224, 224)
    with torch.no_grad():
        want = ref(pixel_values=x).image_embeds
        got = ours(x)
    assert got.shape == want.shape == (3, 128)
    err = float((got - want).norm() / want.norm())
    assert err <= 1e-5, err


def test_encode_image_chunks_and_needs_an_encoder(emulated_ops):
    from mvoc_b200.pipeline import I2VGenXLPipeline

    with pytest.raises(RuntimeError, match="image encoder"):
        I2VGenXLPipeline(None, "cpu").encode_image(torch.zeros(1, 3, 224, 224))
    _, ours = _small_pair()
    pipe = I2VGenXLPipeline(None, "cpu", image_encoder=ours)
    x = torch.randn(5, 3, 224, 224)
    a, b = pipe.encode_image(x, encode_chunk_size=2), pipe.encode_image(x, encode_chunk_size=5)
    assert a.shape == (5, 1, 128)
    assert torch.allclose(a, b, rtol=1e-5, atol=1e-6)


# ------------------------------------------------------------------ preprocessing
def test_clip_image_input_known_answers():
    from PIL import Image

    from mvoc_b200.clip import CLIP_MEAN, CLIP_STD, clip_image_input

    # a 300 x 200 image whose centre (200 x 200 after the covering resize) is grey 128 and whose left and right
    # 50-pixel margins are white: the crop box must drop the margins exactly
    a = torch.full((200, 300, 3), 128, dtype=torch.uint8)
    a[:, :50] = 255
    a[:, 250:] = 255
    x = clip_image_input(Image.fromarray(a.numpy()), width=200)
    assert x.shape == (1, 3, 224, 224) and x.dtype == torch.float32
    for c in range(3):
        assert torch.allclose(x[0, c], torch.full((224, 224), (128 / 255 - CLIP_MEAN[c]) / CLIP_STD[c]), atol=1e-6)
    # mean / std: white and black
    for v in (0, 255):
        x = clip_image_input([Image.new("RGB", (64, 96), (v, v, v))] * 2, width=64)
        assert x.shape == (2, 3, 224, 224)
        want = torch.tensor([(v / 255 - m) / s for m, s in zip(CLIP_MEAN, CLIP_STD)])
        assert torch.allclose(x[:, :, 5, 7], want.expand(2, 3), atol=1e-6)


def test_first_frame_of_a_directory(tmp_path):
    from PIL import Image

    from mvoc_b200.clip import first_frame

    for i, v in enumerate((30, 10, 20)):
        Image.new("RGB", (8, 8), (v, v, v)).save(tmp_path / f"{[2, 0, 1][i]:03d}.png")
    assert first_frame(str(tmp_path)).getpixel((0, 0)) == (10, 10, 10)
    with pytest.raises(FileNotFoundError):
        first_frame(str(tmp_path / "nope.png"))


# ------------------------------------------------------------------ entry argument checks (no GPU touched)
def test_attn_d80_entry_rejects_bad_arguments():
    from mvoc_b200 import _cabi

    lib = _cabi.load()
    st = [257 * 240, 240, 80] * 4
    call = lambda p=16, D=80, dtype=0, strides=st: lib.mvoc_attn_d80_fwd(p, 16, 16, 16, 1, 3, 257, 257, D, *strides,
                                                                      80 ** -0.5, dtype, None)
    assert call(p=None) == -1 and b"null pointer" in lib.mvoc_last_error()
    assert call(D=64) == -2 and b"head_dim 64" in lib.mvoc_last_error()
    assert call(p=24) == -1 and b"16-byte aligned" in lib.mvoc_last_error()
    assert call(dtype=2) == -2 and b"dtype" in lib.mvoc_last_error()
    assert call(strides=[257 * 240, 244, 80] + st[3:]) == -2 and b"multiple of 8" in lib.mvoc_last_error()
    # mvoc_attn_fwd keeps its head_dim-64 contract
    rc = lib.mvoc_attn_fwd(16, 16, 16, 16, 1, 1, 128, 128, 80, *([0] * 12), 0.125, 0, 0, None)
    assert rc == -2 and b"head_dim" in lib.mvoc_last_error()


def test_linear_gelu_entry_rejects_bad_arguments():
    from mvoc_b200 import _cabi

    lib = _cabi.load()
    call = lambda x=16, w=16, b=None, o=16, M=128, K=640, N=1280, ldx=640, ldo=1280, dtype=0: lib.mvoc_linear_gelu(
        x, w, b, o, M, K, N, ldx, ldo, dtype, 0, None)
    assert call(x=None) == -1 and b"non-null" in lib.mvoc_last_error()
    assert call(o=None) == -1 and b"non-null" in lib.mvoc_last_error()
    assert call(K=588, ldx=588) == -2 and b"K=588" in lib.mvoc_last_error()
    assert call(N=1000, ldo=1000) == -2 and b"multiple of 64" in lib.mvoc_last_error()
    assert call(w=24) == -1 and b"16-byte aligned" in lib.mvoc_last_error()
    assert call(b=8) == -1 and b"16-byte aligned" in lib.mvoc_last_error()
    assert call(dtype=2) == -2 and b"dtype" in lib.mvoc_last_error()
    assert call(ldx=320) == -1 and b"leading dimensions" in lib.mvoc_last_error()
    assert call(M=0) == -1 and b"empty problem" in lib.mvoc_last_error()


def test_wrappers_need_cuda_tensors():
    from mvoc_b200 import ops

    x = torch.zeros(1, 4, 160)
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.attention_d80(x, x, x, 2)
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.linear_gelu(torch.zeros(4, 64), torch.zeros(64, 64))


# ------------------------------------------------------------------ the scripts' CLIP paths
def _composite_config(tmp_path, n_obj=2, T=3):
    from mvoc_b200.config import Config

    cfg = Config({"n_frames": T, "image_size": [96, 64],
                  "edited_contorl_frame_path_background": str(tmp_path / "bg"),
                  "edited_contorl_frame_path": [str(tmp_path / f"obj{j}.png") for j in range(n_obj)],
                  "edited_contorl_frame_path_main": str(tmp_path / "main.png")})
    return cfg


def _write_frames(tmp_path, n_obj=2):
    from PIL import Image

    g = torch.Generator().manual_seed(4)
    rnd = lambda: Image.fromarray(torch.randint(0, 256, (64, 96, 3), generator=g, dtype=torch.uint8).numpy())
    (tmp_path / "bg").mkdir()
    bg = rnd()
    bg.save(tmp_path / "bg" / "000.png")
    rnd().save(tmp_path / "bg" / "001.png")
    objs = [rnd() for _ in range(n_obj)]
    for j, im in enumerate(objs):
        im.save(tmp_path / f"obj{j}.png")
    main = rnd()
    main.save(tmp_path / "main.png")
    return [bg] + objs + [main]


def test_composite_embeddings_order_and_repeat(tmp_path, emulated_ops):
    """[bg, objs..., zeros, main], one embedding per branch repeated over T; the UNet's context reads [:, 0:1], so the
    repeat gives it exactly what per-frame embeddings of the same control frames give it."""
    from mvoc_b200.clip import clip_image_input
    from mvoc_b200.composite import branch_image_embeddings
    from mvoc_b200.pipeline import I2VGenXLPipeline

    images = _write_frames(tmp_path)
    cfg = _composite_config(tmp_path)
    _, ours = _small_pair()
    pipe = I2VGenXLPipeline(None, "cpu", image_encoder=ours)
    emb = branch_image_embeddings(pipe, cfg)
    assert emb.shape == (5, 3, 128)
    want = pipe.encode_image(clip_image_input(images, 96))[:, 0]                 # bg, obj0, obj1, main
    for i, j in ((0, 0), (1, 1), (2, 2), (4, 3)):
        assert torch.equal(emb[i], want[j].expand(3, -1))
    assert torch.equal(emb[3], torch.zeros(3, 128))
    # per-frame encoding of the same frames (the reference's T calls) and the repeat agree on what the UNet reads
    per_frame = torch.stack([pipe.encode_image(clip_image_input([im] * 3, 96))[:, 0] for im in images])
    assert torch.allclose(emb[[0, 1, 2, 4], 0:1], per_frame[:, 0:1], rtol=1e-5, atol=1e-6)


def test_composite_missing_control_frame_is_an_error(tmp_path, emulated_ops):
    from mvoc_b200.composite import branch_image_embeddings
    from mvoc_b200.pipeline import I2VGenXLPipeline

    _write_frames(tmp_path)
    os.remove(tmp_path / "obj1.png")
    cfg = _composite_config(tmp_path)
    _, ours = _small_pair()
    pipe = I2VGenXLPipeline(None, "cpu", image_encoder=ours)
    with pytest.raises(FileNotFoundError, match="obj1.png"):
        branch_image_embeddings(pipe, cfg)
    emb = branch_image_embeddings(pipe, cfg, allow_synthetic=True)                # --synthetic substitutes it
    assert emb.shape == (5, 3, 128) and torch.isfinite(emb).all()


def test_inverse_image_embeddings_entry(tmp_path, emulated_ops):
    from mvoc_b200.clip import clip_image_input, first_frame
    from mvoc_b200.config import Config
    from mvoc_b200.inverse import image_embeddings_entry
    from mvoc_b200.pipeline import I2VGenXLPipeline

    _, ours = _small_pair()
    pipe = I2VGenXLPipeline(None, "cpu", image_encoder=ours)
    cfg = Config({"video_dir": str(tmp_path), "video_name": "clip", "inverse_config": Config({"image_size": [96, 64]})})
    with pytest.raises(FileNotFoundError, match="clip"):
        image_embeddings_entry(pipe, cfg, 0, False)
    syn = image_embeddings_entry(pipe, cfg, 0, True)                              # --synthetic, no frames
    assert syn.shape == (1, 1, 128) and torch.isfinite(syn).all()
    _write_frames(tmp_path)
    os.rename(tmp_path / "bg", tmp_path / "clip")
    got = image_embeddings_entry(pipe, cfg, 0, False)
    want = pipe.encode_image(clip_image_input(first_frame(str(tmp_path / "clip")), 96))
    assert torch.equal(got, want)
