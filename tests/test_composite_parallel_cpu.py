"""composite.py frame-parallel over gloo ranks, and the composition's image latents computed from its control frames,
without a GPU: the 4-level model in fp32 on CPU with the kernels emulated (tests/cpu_ops_emulation.py)."""
import json
import os
import socket
import sys

import pytest
import torch
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOL = 1e-5
TEMPLATE = os.path.join(ROOT, "configs", "group_composite", "template.yaml")


def rel_l2(a, b):
    return float((a.float() - b.float()).norm() / b.float().norm())


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _entry(name, T, w_px, h_px, n_obj, **kw):
    e = {"active": True, "video_name": name, "edited_video_name": f"{name} edit", "image_size": [w_px, h_px],
         "n_frames": T, "n_steps": 3, "ddim_init_latents_t_idx": 0, "fusion_step": [0, 1], "random_noise_ratio": 0.0,
         "pnp_f_t": 0.4, "pnp_spatial_attn_t": 1.0, "pnp_temp_attn_t": 1.0,
         "obj_mask_path": [f"m{j}" for j in range(n_obj)], "obj_ddim_latents_path": [f"l{j}" for j in range(n_obj)]}
    e.update(kw)
    return e


def _group(path, data_dir, entries):
    path.write_text(json.dumps([dict(e, data_dir=str(data_dir)) for e in entries]))
    return str(path)


def _out_dir(data_dir, e):
    return os.path.join(str(data_dir), "Results", "MVOC-B200", "i2vgen-xl", e["video_name"], e["edited_video_name"])


# two active entries of different geometry: 4 x 16x16 latents with two objects, 8 x 8x16 with one (its 1x2 lowest
# level divides by no rank count above 2, so its temporal operators also run replicated)
ENTRIES = [_entry("a", 4, 128, 128, 2), _entry("b", 8, 128, 64, 1)]
VAE_WIDTHS = (32, 64, 128, 512)


def _small_decoder(path, device, dtype=torch.bfloat16):
    """A narrow AutoencoderKL decoder (the mid block stays 512 wide: the attention kernel is for D = 512 only),
    seeded, so every rank builds the same one."""
    from mvoc_b200.unet3d import prepare
    from mvoc_b200.vae import AutoencoderKLDecoder

    torch.manual_seed(11)
    return prepare(AutoencoderKLDecoder(VAE_WIDTHS, groups=8).eval().requires_grad_(False).to(device, torch.float32))


def _worker(rank, world, port, ret, cfg, decode):
    """composite.main on one gloo rank (world 1: the single-process path, no process group)."""
    import traceback

    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    torch.set_num_threads(max(1, (os.cpu_count() or 2) // world))
    try:
        from mvoc_b200 import composite, ops, unet3d, vae
        from tests import cpu_ops_emulation as emu
        from tests.test_vae_cpu import attention_d512

        emu.install()
        ops.attention_d512 = attention_d512
        unet3d.UNetConfig.full = staticmethod(unet3d.UNetConfig.tiny4)
        real_prepare = unet3d.prepare
        unet3d.prepare = lambda m: real_prepare(m.to(torch.float32))
        vae.load_vae_decoder = _small_decoder
        latents, saved = [], []
        real_run_entry, real_save = composite.run_entry, torch.save

        def run_entry(*a, **kw):
            latents.append(real_run_entry(*a, **kw))
            return latents[-1]

        def save(obj, path, *a, **kw):
            saved.append(str(path))
            return real_save(obj, path, *a, **kw)

        composite.run_entry, torch.save = run_entry, save
        torch.manual_seed(100 + rank)      # random-init UNet weights differ per rank until rank 0's are broadcast
        done = composite.main(TEMPLATE, cfg, device="cpu", synthetic_inputs=True,
                              vae_state_dict="decoder" if decode else None)
        ret[rank] = ("ok", done, [x.clone() for x in latents], saved)
    except Exception as e:
        ret[rank] = ("error", f"{type(e).__name__}: {e}", traceback.format_exc(), [])


def _spawn(world, cfg, decode=False):
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_worker, args=(world, _free_port(), ret, cfg, decode), nprocs=world, join=True)
    return [ret.get(r) for r in range(world)]


def _frames(d):
    import numpy as np
    from PIL import Image

    return {n: np.asarray(Image.open(os.path.join(d, n)), dtype=np.int16) for n in sorted(os.listdir(d))}


@pytest.mark.parametrize("world", [2, pytest.param(4, marks=pytest.mark.skipif(
    os.environ.get("MVOC_LONG_TESTS") != "1", reason="5 processes; ~1 min (world 2 runs by default)"))])
def test_composite_main_frame_parallel_matches_one_rank(tmp_path, world):
    """Two entries of different geometry, one after another over all ranks: every rank ends with the latents of a
    one-rank run (rel-L2 <= 1e-5, fp32), bit-identical across ranks; only rank 0 writes composite_latents; every
    rank decodes its own frames, and together they write the frames a one-rank run writes."""
    runs = {}
    for w in (1, world):
        data = tmp_path / f"w{w}"
        data.mkdir()
        runs[w] = (data, _spawn(w, _group(tmp_path / f"w{w}.json", data, ENTRIES), decode=True))
    (data1, (one,)), (dataN, ranks) = runs[1], runs[world]
    assert one[0] == "ok", one[2]
    for r, res in enumerate(ranks):
        assert res[0] == "ok", f"rank {r}: {res[1]}\n{res[2]}"
        assert res[1] == len(ENTRIES)
    for i, e in enumerate(ENTRIES):
        ref = one[2][i]
        assert ref.shape == (1, 4, e["n_frames"], e["image_size"][1] // 8, e["image_size"][0] // 8)
        for r, res in enumerate(ranks):
            assert torch.equal(res[2][i], ranks[0][2][i]), f"entry {i}: rank {r} differs from rank 0"
        err = rel_l2(ranks[0][2][i], ref)
        assert err <= TOL, f"entry {i}: {err:.3e}"
        out = os.path.join(_out_dir(dataN, e), "composite_latents.synthetic.pt")
        assert torch.equal(torch.load(out), ranks[0][2][i])
        frames_n = _frames(os.path.join(_out_dir(dataN, e), "composite_frames.synthetic"))
        frames_1 = _frames(os.path.join(_out_dir(data1, e), "composite_frames.synthetic"))
        assert sorted(frames_n) == sorted(frames_1) == [f"{t:03d}.png" for t in range(e["n_frames"])]
        for n in frames_1:
            assert abs(frames_n[n] - frames_1[n]).max() <= 1, n
    assert sorted(os.path.basename(p) for p in ranks[0][3]) == ["composite_latents.synthetic.pt"] * len(ENTRIES)
    for r in range(1, world):
        assert ranks[r][3] == [], f"rank {r} wrote {ranks[r][3]}"


def test_composite_main_refuses_a_frame_count_the_ranks_do_not_divide(tmp_path):
    """n_frames = 3 on 2 ranks: every rank raises before any collective (naming both numbers), and every process
    exits."""
    data = tmp_path / "odd"
    data.mkdir()
    cfg = _group(tmp_path / "odd.json", data, [ENTRIES[0], _entry("c", 3, 128, 128, 1)])
    for r, res in enumerate(_spawn(2, cfg)):
        assert res[0] == "error", f"rank {r} did not raise"
        assert res[1].startswith("ValueError") and "n_frames=3" in res[1] and "WORLD_SIZE=2" in res[1], res[1]
    assert not os.path.exists(os.path.join(str(data), "Results"))


def test_exchange_arena_rule(monkeypatch):
    """bench.py's sizing rule: ~60 first-level tensors of (n+3) x T x h x w x 320 bf16 split over the ranks,
    clamped to [4096, 32768] MiB; MVOC_EXCHANGE_ARENA_MB wins when set."""
    from mvoc_b200.parallel import exchange_arena_mb

    monkeypatch.delenv("MVOC_EXCHANGE_ARENA_MB", raising=False)
    assert exchange_arena_mb(5, 16, 64, 64, 2) == 6000          # config 2
    assert exchange_arena_mb(5, 16, 64, 64, 8) == 4096
    assert exchange_arena_mb(6, 32, 88, 160, 2) == 32768        # config 5
    assert exchange_arena_mb(6, 32, 88, 160, 8) == 12375
    monkeypatch.setenv("MVOC_EXCHANGE_ARENA_MB", "1234")
    assert exchange_arena_mb(5, 16, 64, 64, 2) == 1234


# ------------------------------------------------------------------ image latents from the control frames
def _golden_control_frames(tmp_path):
    """The golden composition fixture's first frames as control-frame PNGs; the background as a directory."""
    from tests.golden import spec

    fx = spec.loop_fixture("default")
    imgs = spec.loop_images(fx)
    (tmp_path / "bg").mkdir()
    imgs["bg"][0].save(tmp_path / "bg" / "000.png")
    imgs["bg"][1].save(tmp_path / "bg" / "001.png")
    for j, frames in enumerate(imgs["objs"]):
        frames[0].save(tmp_path / f"obj{j}.png")
    imgs["main"][0].save(tmp_path / "main.png")
    return fx


def _control_config(tmp_path, fx):
    from mvoc_b200.config import Config

    return Config({"n_frames": fx["T"], "image_size": [fx["W"] * 8, fx["H"] * 8], "seed": 6,
                   "obj_mask_path": [f"m{j}" for j in range(fx["n_obj"])],
                   "edited_contorl_frame_path_background": str(tmp_path / "bg"),
                   "edited_contorl_frame_path": [str(tmp_path / f"obj{j}.png") for j in range(fx["n_obj"])],
                   "edited_contorl_frame_path_main": str(tmp_path / "main.png")})


def _vae_double(images, generator=None, encode_chunk_size=4):
    # make_golden_loops.FakeVAE: average pooling, the channel mean as the fourth channel, x3; the double's
    # latent_dist.sample() returns that tensor, which the reference then scales
    import torch.nn.functional as F

    from mvoc_b200.vae import SCALING_FACTOR

    p = F.avg_pool2d(images.float(), 8)
    return torch.cat([p, p.mean(1, keepdim=True)], dim=1) * 3.0 * SCALING_FACTOR


def test_branch_image_latents_match_reference_golden(tmp_path):
    """The control frames through center_crop_wide -> pil_to_model_input -> prepare_image_latents, with the golden
    generator's VAE double in place of the encoder, give the reference's own image_latents_first and image_latents
    of the composition golden ([bg, objs, main, main])."""
    from mvoc_b200.composite import branch_image_latents
    from mvoc_b200.pipeline import I2VGenXLPipeline

    fx = _golden_control_frames(tmp_path)
    seam = torch.load(os.path.join(ROOT, "tests", "golden", "composition_loop_tiny4.pt"))["seam"]
    pipe = I2VGenXLPipeline(None, "cpu")
    pipe._vae_latents = _vae_double
    got = branch_image_latents(pipe, _control_config(tmp_path, fx))
    assert got.shape == seam["image_latents"].shape == (fx["n_obj"] + 3, 4, fx["T"], fx["H"], fx["W"])
    for key in ("image_latents_first", "image_latents"):
        assert float((got - seam[key].float()).abs().max()) <= 1e-6, key


def test_branch_image_latents_draw_one_seeded_posterior_sample(tmp_path):
    """prepare_image_latents of the n+2 distinct frames under torch.Generator().manual_seed(seed), main duplicated;
    a missing control frame is an error unless --synthetic substitutes a seeded one."""
    from mvoc_b200.composite import branch_image_latents, control_frames
    from mvoc_b200.pipeline import I2VGenXLPipeline
    from mvoc_b200.vae import pil_to_model_input

    fx = _golden_control_frames(tmp_path)
    cfg = _control_config(tmp_path, fx)
    seen = []

    def encoder(images, generator=None, encode_chunk_size=4):
        seen.append((images.clone(), generator.initial_seed()))
        noise = torch.randn(images.shape[0], 4, images.shape[2] // 8, images.shape[3] // 8, generator=generator)
        return _vae_double(images) + noise

    pipe = I2VGenXLPipeline(None, "cpu")
    pipe._vae_latents = encoder
    got = branch_image_latents(pipe, cfg)
    (images, seed), = seen
    assert seed == 6 and torch.equal(images, pil_to_model_input(control_frames(cfg)))
    want = pipe.prepare_image_latents(images, fx["T"], torch.Generator().manual_seed(6))
    assert torch.equal(got[:-1], want) and torch.equal(got[-1], want[-1])
    os.remove(tmp_path / "obj1.png")
    with pytest.raises(FileNotFoundError, match="obj1.png"):
        branch_image_latents(pipe, cfg)
    assert branch_image_latents(pipe, cfg, allow_synthetic=True).shape == got.shape


# ------------------------------------------------------------------ the script's flags
def test_encode_image_latents_needs_the_vae_file(tmp_path):
    from mvoc_b200 import composite

    with pytest.raises(ValueError, match="--encode_image_latents needs --vae_state_dict"):
        composite.main(TEMPLATE, str(tmp_path / "absent.json"), synthetic_inputs=True, device="cpu",
                       encode_image_latents=True)
    args = composite.build_parser().parse_args(["--encode_image_latents", "--vae_state_dict", "v.pt"])
    assert args.encode_image_latents is True
    assert composite.build_parser().parse_args([]).encode_image_latents is False


@pytest.fixture()
def stubbed_towers(monkeypatch, tmp_path):
    """composite.main on the 4-level model with every tower stubbed: the VAE encoder is the golden double, the CLIP
    towers return seeded constants, run_entry records its conditioning and decoding returns zeros."""
    from mvoc_b200 import composite, unet3d
    from mvoc_b200.pipeline import I2VGenXLPipeline

    monkeypatch.setattr(unet3d.UNetConfig, "full", staticmethod(unet3d.UNetConfig.tiny4))
    weights = str(tmp_path / "unet.pt")
    torch.save(unet3d.I2VGenXLUNet(unet3d.UNetConfig.tiny4()).state_dict(), weights)
    monkeypatch.setattr("mvoc_b200.vae.load_vae_decoder", lambda p, device: object())
    monkeypatch.setattr("mvoc_b200.vae.load_vae_encoder", lambda p, device: object())
    monkeypatch.setattr("mvoc_b200.clip.load_clip_image_encoder", lambda p, device: object())
    monkeypatch.setattr("mvoc_b200.clip_text.load_text_tower", lambda p, d, device: (object(), object()) if p else (None, None))
    monkeypatch.setattr(I2VGenXLPipeline, "_vae_latents", lambda self, images, generator=None: _vae_double(images))
    monkeypatch.setattr(I2VGenXLPipeline, "encode_image",
                        lambda self, x: torch.arange(x.shape[0] * 1024.0).view(-1, 1, 1024))
    monkeypatch.setattr(I2VGenXLPipeline, "encode_prompt", lambda self, p: torch.ones(len(p), 77, 1024))
    monkeypatch.setattr(I2VGenXLPipeline, "decode_latents",
                        lambda self, lat: torch.zeros(1, 3, lat.shape[2], 8 * lat.shape[3], 8 * lat.shape[4]))
    seen = []

    def run_entry(pipe, config, device, conditioning=None, allow_synthetic=False):
        seen.append((pipe, conditioning))
        T, h, w = composite.latent_geometry(config)
        return torch.zeros(1, 4, T, h, w)

    monkeypatch.setattr(composite, "run_entry", run_entry)
    return weights, seen


def test_composite_runs_without_conditioning_when_every_key_is_computed(tmp_path, stubbed_towers, caplog):
    """--encode_image_latents, --image_encoder_state_dict and the text flags together: no --conditioning file (nor
    --synthetic) is needed and the image latents reaching the loop are branch_image_latents of the control frames.
    With a conditioning file, computed keys replace the file's (logged) and the others are read from it; without
    the image tower the error names the key no flag computes."""
    import logging

    from mvoc_b200 import composite

    weights, seen = stubbed_towers
    fx = _golden_control_frames(tmp_path)
    entry = _entry("golden", fx["T"], fx["W"] * 8, fx["H"] * 8, fx["n_obj"],
                   edited_contorl_frame_path_background="bg",
                   edited_contorl_frame_path=[f"obj{j}.png" for j in range(fx["n_obj"])],
                   edited_contorl_frame_path_main="main.png")
    cfg = _group(tmp_path / "group.json", tmp_path, [entry])
    flags = dict(unet_state_dict=weights, device="cpu", vae_state_dict="vae", image_encoder_state_dict="clip",
                 text_encoder_state_dict="text", tokenizer_dir="tok", encode_image_latents=True)
    assert composite.main(TEMPLATE, cfg, **flags) == 1
    pipe, cond = seen[-1]
    want = composite.branch_image_latents(pipe, _control_config(tmp_path, fx))
    assert sorted(cond) == sorted(composite.CONDITIONING_KEYS)
    assert torch.equal(cond["image_latents_first"], want) and torch.equal(cond["image_latents"], want)
    assert torch.equal(cond["prompt_embeds"], torch.ones(fx["n_obj"] + 3, 77, 1024))
    frames = tmp_path / "Results" / "MVOC-B200" / "i2vgen-xl" / "golden" / "golden edit" / "composite_frames"
    assert sorted(os.listdir(frames)) == [f"{t:03d}.png" for t in range(fx["T"])]

    nb = fx["n_obj"] + 3
    file = {"prompt_embeds": torch.full((nb, 77, 1024), 2.0), "image_embeddings": torch.full((nb, fx["T"], 1024), 3.0),
            "image_latents_first": torch.zeros(nb, 4, fx["T"], fx["H"], fx["W"]),
            "image_latents": torch.zeros(nb, 4, fx["T"], fx["H"], fx["W"])}
    torch.save(file, tmp_path / "cond.pt")
    with caplog.at_level(logging.INFO, logger="mvoc_b200.composite"):
        composite.main(TEMPLATE, cfg, unet_state_dict=weights, device="cpu", vae_state_dict="vae",
                       encode_image_latents=True, conditioning=str(tmp_path / "cond.pt"))
    _, cond = seen[-1]
    assert torch.equal(cond["image_latents"], want) and torch.equal(cond["image_latents_first"], want)
    assert torch.equal(cond["prompt_embeds"], file["prompt_embeds"])
    assert torch.equal(cond["image_embeddings"], file["image_embeddings"])
    assert "image_latents of the conditioning file is not read (--encode_image_latents computes it)" in caplog.text

    with pytest.raises(FileNotFoundError, match="image_embeddings"):
        composite.main(TEMPLATE, cfg, **dict(flags, image_encoder_state_dict=None))
