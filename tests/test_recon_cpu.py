"""The plain sampling loop (I2VGenXLPipeline.sample) and inverse.py's recon_config without a GPU: the product's host
layer in fp32 on CPU with the kernels emulated (tests/cpu_ops_emulation.py), against the fp32 oracle loop
(oracle/sampling.py) on the 4-level golden model.  Nothing is bf16 here, so the bar is tight (1e-5)."""
import json
import os

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOL = 1e-5


def rel_l2(a, b):
    return float((a.float() - b.float()).norm() / b.float().norm())


@pytest.fixture()
def emulated_ops():
    from tests import cpu_ops_emulation as emu

    saved = emu.install()
    yield
    emu.uninstall(saved)


def _product_cpu(oracle_unet, kind):
    from mvoc_b200.unet3d import I2VGenXLUNet, UNetConfig, prepare

    m = I2VGenXLUNet(UNetConfig.named(kind)).eval().requires_grad_(False)
    m.load_state_dict(oracle_unet.state_dict(), strict=True)
    return prepare(m.to(torch.float32))


def seam_inputs():
    """Batch-1 conditioning of the inversion golden (the reference's own seam tensors) plus a seeded negative prompt."""
    from tests.golden import spec

    seam = torch.load(os.path.join(ROOT, "tests", "golden", "inversion_loop_tiny4.pt"), map_location="cpu")["seam"]
    return {"prompt_embeds": seam["encoder_hidden_states"], "negative_prompt_embeds": spec.text_embedding("blurry"),
            "image_embeddings": seam["image_embeddings"], "image_latents": seam["image_latents"], "fps": seam["fps"]}


def _pipe():
    from mvoc_b200.pipeline import I2VGenXLPipeline
    from tests.golden import spec

    ou = spec.build_tiny4(seed=0)
    return I2VGenXLPipeline(_product_cpu(ou, "tiny4"), "cpu"), ou


def _sample(pipe, inp, **kw):
    return pipe.sample(inp["prompt_embeds"], inp["negative_prompt_embeds"], inp["image_embeddings"],
                       inp["image_latents"], inp["fps"], **kw)


@pytest.mark.parametrize("cfg,steps,max_steps", [(9.0, 10, 3), (1.0, 10, 3), (9.0, 10, None), (1.0, 10, None)])
def test_sample_from_latents_vs_oracle(emulated_ops, cfg, steps, max_steps):
    from oracle.sampling import sample_loop

    pipe, ou = _pipe()
    inp = seam_inputs()
    x0 = torch.randn(1, 4, 4, 16, 16, generator=torch.Generator().manual_seed(5))
    ref_rec, rec = [], []
    ref = sample_loop(ou, inp, steps, cfg, x0, max_steps=max_steps, record=ref_rec)
    out = _sample(pipe, inp, num_inference_steps=steps, guidance_scale=cfg, latents=x0, max_steps=max_steps,
                  callback=lambda i, t, lat: rec.append(lat.clone()))
    assert out.dtype == torch.float32 and out.shape == x0.shape
    assert len(rec) == len(ref_rec) == (max_steps or steps)
    for i, (a, b) in enumerate(zip(rec, ref_rec)):
        assert rel_l2(a, b) <= TOL, f"step {i}: {rel_l2(a, b):.3e}"
    assert rel_l2(out, ref) <= TOL
    assert torch.equal(x0, torch.randn(1, 4, 4, 16, 16, generator=torch.Generator().manual_seed(5)))  # not modified


@pytest.mark.parametrize("cfg", [9.0, 1.0])
def test_sample_from_a_seeded_generator_vs_oracle(emulated_ops, cfg):
    """latents=None: torch.randn((1,4,T,h,w)) in fp32 on the generator's device (prepare_latents)."""
    from oracle.sampling import sample_loop

    pipe, ou = _pipe()
    inp = seam_inputs()
    ref = sample_loop(ou, inp, 10, cfg, torch.randn(1, 4, 4, 16, 16, generator=torch.Generator().manual_seed(3)),
                      max_steps=2)
    out = _sample(pipe, inp, num_inference_steps=10, guidance_scale=cfg, generator=torch.Generator().manual_seed(3),
                  max_steps=2)
    assert rel_l2(out, ref) <= TOL
    again = _sample(pipe, inp, num_inference_steps=10, guidance_scale=cfg, generator=torch.Generator().manual_seed(3),
                    max_steps=2)
    assert torch.equal(out, again)


@pytest.mark.parametrize("cfg", [9.0, 1.0, 0.5])
def test_sample_assembles_the_guidance_batch(emulated_ops, monkeypatch, cfg):
    """Under guidance the UNet batch is [uncond, cond]: prompt embeds [negative, prompt], image embeddings
    [zeros, emb], the image latents and fps twice; at guidance <= 1 it is the batch-1 conditioning of `invert`."""
    from mvoc_b200.pipeline import I2VGenXLPipeline

    pipe, _ = _pipe()
    inp = seam_inputs()
    seen = []
    real = I2VGenXLPipeline._unet_forward

    def spy(self, sample, t, cond):
        seen.append((sample.clone(), cond))
        return real(self, sample, t, cond)

    monkeypatch.setattr(I2VGenXLPipeline, "_unet_forward", spy)
    x0 = torch.randn(1, 4, 4, 16, 16, generator=torch.Generator().manual_seed(5))
    _sample(pipe, inp, num_inference_steps=10, guidance_scale=cfg, latents=x0, max_steps=2)
    assert len(seen) == 2
    sample, cond = seen[0]
    assert seen[1][1] is cond                                  # ONE Conditioning per run: caches / graphs built once
    if cfg > 1:
        assert sample.shape[0] == 2 and torch.equal(sample[0], x0[0]) and torch.equal(sample[1], x0[0])
        assert torch.equal(cond.prompt_embeds, torch.cat([inp["negative_prompt_embeds"], inp["prompt_embeds"]]))
        assert torch.equal(cond.image_embeddings, torch.cat([torch.zeros_like(inp["image_embeddings"]),
                                                             inp["image_embeddings"]]))
        assert torch.equal(cond.image_latents, torch.cat([inp["image_latents"]] * 2))
        assert torch.equal(cond.fps, torch.cat([inp["fps"]] * 2))
    else:
        assert sample.shape[0] == 1 and torch.equal(sample, x0)
        assert torch.equal(cond.prompt_embeds, inp["prompt_embeds"])
        assert torch.equal(cond.image_embeddings, inp["image_embeddings"])
        assert torch.equal(cond.image_latents, inp["image_latents"]) and torch.equal(cond.fps, inp["fps"])
    assert cond.image_latents_first is cond.image_latents


def test_sample_needs_a_negative_prompt_under_guidance(emulated_ops):
    pipe, _ = _pipe()
    inp = dict(seam_inputs(), negative_prompt_embeds=None)
    with pytest.raises(ValueError, match="negative_prompt_embeds"):
        _sample(pipe, inp, num_inference_steps=10, guidance_scale=9.0, max_steps=1)
    _sample(pipe, inp, num_inference_steps=10, guidance_scale=1.0, max_steps=1)     # not read without guidance


def test_sample_refuses_injection_hooks(emulated_ops):
    from types import SimpleNamespace

    from mvoc_b200.pipeline import init_pnp
    from mvoc_b200.scheduler import DDIMSchedule

    pipe, _ = _pipe()
    inp = seam_inputs()
    init_pnp(pipe, DDIMSchedule(50), SimpleNamespace(n_steps=50, pnp_f_t=0.1, pnp_spatial_attn_t=1.0,
                                                     pnp_temp_attn_t=1.0, inject_background=False))
    with pytest.raises(ValueError, match="injection hooks"):
        _sample(pipe, inp, num_inference_steps=10, guidance_scale=9.0, max_steps=1)
    # only the feature injection scheduled: still refused
    pipe2, _ = _pipe()
    init_pnp(pipe2, DDIMSchedule(50), SimpleNamespace(n_steps=50, pnp_f_t=0.1, pnp_spatial_attn_t=0.0,
                                                      pnp_temp_attn_t=0.0, inject_background=False))
    with pytest.raises(ValueError, match="injection hooks"):
        _sample(pipe2, inp, num_inference_steps=10, guidance_scale=1.0, max_steps=1)


# ------------------------------------------------------------------ inverse.py recon_config
T, PX = 2, 64           # 2 frames of 64 x 64 px -> 8 x 8 latents


def _write_inputs(path, negative=True):
    from tests.golden import spec

    g = torch.Generator().manual_seed(21)
    src = {"latents": torch.randn(1, 4, T, PX // 8, PX // 8, generator=g),
           "prompt_embeds": spec.text_embedding("a boat"),
           "image_embeddings": torch.randn(1, 1, 1024, generator=g),
           "image_latents": torch.randn(1, 4, T, PX // 8, PX // 8, generator=g) * 0.18}
    if negative:
        src["negative_prompt_embeds"] = spec.text_embedding("blurry")
    torch.save(src, path)
    return src


def _group(tmp_path, name, recon):
    entry = {"active": True, "force_recompute_latents": True, "video_name": "clip", "data_dir": str(tmp_path / name),
             "image_size": [PX, PX], "n_frames": T, "inverse_config": {"n_steps": 4}}
    if recon is not None:
        entry["recon_config"] = recon
    p = tmp_path / f"{name}.json"
    p.write_text(json.dumps([entry]))
    return str(p), tmp_path / name / "inversions" / "i2vgen-xl" / "clip"


def _template(tmp_path, with_recon_key=True):
    """The shipped template, with or without its recon_config key."""
    import yaml

    from mvoc_b200 import config as cfgmod

    t = cfgmod.load_template(os.path.join(ROOT, "configs", "group_inversion", "template.yaml"))
    if not with_recon_key:
        t.pop("recon_config")
    p = tmp_path / ("template.yaml" if with_recon_key else "template_no_recon.yaml")
    p.write_text(yaml.safe_dump(t))
    return str(p)


@pytest.fixture()
def tiny_script(monkeypatch, tmp_path, emulated_ops):
    """inverse.main on the 4-level model in fp32 on CPU: UNet weights file, --inputs file."""
    from mvoc_b200 import unet3d
    from tests.golden import spec

    monkeypatch.setattr(unet3d.UNetConfig, "full", staticmethod(unet3d.UNetConfig.tiny4))
    real_prepare = unet3d.prepare
    monkeypatch.setattr(unet3d, "prepare", lambda m: real_prepare(m.to(torch.float32)))
    weights = str(tmp_path / "unet.pt")
    torch.save(spec.build_tiny4(seed=0).state_dict(), weights)
    return weights


def test_inverse_recon_writes_the_sample_of_the_noisiest_latents(tmp_path, tiny_script, monkeypatch):
    from mvoc_b200 import inverse
    from mvoc_b200.pipeline import I2VGenXLPipeline
    from mvoc_b200.utils import load_ddim_latents_at_T

    inputs = str(tmp_path / "inputs.pt")
    src = _write_inputs(inputs)
    seen = {}
    real = I2VGenXLPipeline.sample

    def spy(self, *args, **kw):
        seen.update(pipe=self, args=args, kw=kw)
        return real(self, *args, **kw)

    monkeypatch.setattr(I2VGenXLPipeline, "sample", spy)
    cfg, out = _group(tmp_path, "recon", {"enable_recon": True, "n_steps": 3, "cfg": 9.0})
    assert inverse.main(_template(tmp_path), cfg, tiny_script, inputs=inputs, device="cpu") == 1
    lat_dir = out / "ddim_latents"
    assert sorted(os.listdir(lat_dir)) == [f"ddim_latents_{t}.pt" for t in (1, 251, 501, 751)]
    got = torch.load(out / "recon" / "recon_latents.pt")
    x_T = load_ddim_latents_at_T(str(lat_dir))
    assert x_T.dtype == torch.float16
    pipe = seen["pipe"]
    prompt, negative, emb, il, fps = seen["args"]
    assert torch.equal(prompt, src["prompt_embeds"]) and torch.equal(negative, src["negative_prompt_embeds"])
    assert torch.equal(emb, src["image_embeddings"]) and torch.equal(il, src["image_latents"])
    assert seen["kw"]["num_inference_steps"] == 3 and seen["kw"]["guidance_scale"] == 9.0
    want = pipe.sample(prompt, negative, emb, il, fps, num_inference_steps=3, guidance_scale=9.0,
                       latents=x_T.float())
    assert got.dtype == torch.float32 and got.shape == (1, 4, T, PX // 8, PX // 8)
    assert torch.equal(got, want)
    # a complete inversion is skipped, the reconstruction still runs (and gives the same latents)
    os.remove(out / "recon" / "recon_latents.pt")
    cfg2, _ = _group(tmp_path, "recon", {"enable_recon": True, "n_steps": 3, "cfg": 9.0})
    data = json.loads(open(cfg2).read())
    data[0]["force_recompute_latents"] = False
    open(cfg2, "w").write(json.dumps(data))
    assert inverse.main(_template(tmp_path), cfg2, tiny_script, inputs=inputs, device="cpu") == 0
    assert torch.equal(torch.load(out / "recon" / "recon_latents.pt"), want)


def test_inverse_without_recon_is_unchanged(tmp_path, tiny_script):
    """enable_recon false (the template's value) writes the same ddim_latents files as a template without the
    recon_config key, and no reconstruction output."""
    from mvoc_b200 import inverse

    inputs = str(tmp_path / "inputs.pt")
    _write_inputs(inputs, negative=False)
    cfg_a, out_a = _group(tmp_path, "off", None)
    cfg_b, out_b = _group(tmp_path, "absent", None)
    assert inverse.main(_template(tmp_path), cfg_a, tiny_script, inputs=inputs, device="cpu") == 1
    assert inverse.main(_template(tmp_path, with_recon_key=False), cfg_b, tiny_script, inputs=inputs,
                        device="cpu") == 1
    names = sorted(os.listdir(out_a / "ddim_latents"))
    assert names == sorted(os.listdir(out_b / "ddim_latents")) and len(names) == 4
    for n in names:
        assert (out_a / "ddim_latents" / n).read_bytes() == (out_b / "ddim_latents" / n).read_bytes()
    assert sorted(os.listdir(out_a)) == sorted(os.listdir(out_b)) == ["ddim_latents"]


def test_inverse_recon_names_the_missing_negative_prompt(tmp_path, tiny_script):
    from mvoc_b200 import inverse

    inputs = str(tmp_path / "inputs.pt")
    _write_inputs(inputs, negative=False)
    cfg, out = _group(tmp_path, "noneg", {"enable_recon": True, "n_steps": 2, "cfg": 9.0})
    with pytest.raises(KeyError, match="negative_prompt_embeds"):
        inverse.main(_template(tmp_path), cfg, tiny_script, inputs=inputs, device="cpu")
    # without guidance the key is not needed
    cfg, out = _group(tmp_path, "cfg1", {"enable_recon": True, "n_steps": 2, "cfg": 1.0})
    assert inverse.main(_template(tmp_path), cfg, tiny_script, inputs=inputs, device="cpu") == 1
    assert (out / "recon" / "recon_latents.pt").exists()


def test_template_recon_keys():
    from mvoc_b200 import config as cfgmod

    (c,) = list(cfgmod.iter_configs(os.path.join(ROOT, "configs", "group_inversion", "template.yaml"),
                                    os.path.join(ROOT, "configs", "group_inversion", "group_config.json")))
    r = c.recon_config
    assert r.enable_recon is False and r.n_steps == 50 and r.cfg == 9.0
    assert r.output_dir == f"{c.output_dir}/recon" and r.ddim_latents_path == c.inverse_config.output_dir
    # an entry's values win over the template's
    merged = cfgmod.merge(cfgmod.load_template(os.path.join(ROOT, "configs", "group_inversion", "template.yaml")),
                          {"video_name": "v", "recon_config": {"enable_recon": True, "n_steps": 25, "cfg": 7.5}})
    assert merged.recon_config.enable_recon is True and merged.recon_config.n_steps == 25
    assert merged.recon_config.cfg == 7.5 and merged.recon_config.output_dir.endswith("/v/recon")
