"""The plain sampling loop (I2VGenXLPipeline.sample) on the B200 kernels against the fp32 oracle loop
(oracle/sampling.py), and inverse.py's recon_config end to end on one GPU.

Bars (bf16 kernels vs the fp32 oracle) are ~2x what a B200 measured, stated beside each."""
import json
import os

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

BAR_TINY4_10 = 4.5e-2      # tiny4, 10 guided steps, final latents: measured 2.22e-2
BAR_FULL_STEP = 2.5e-3      # config 2's full-width model (2 of its 16 frames), one guided step: measured 1.23e-3
ROUND_TRIP_FACTOR = 2.0     # product round-trip distance to x0 over the oracle's own: measured 0.2209 / 0.2208


def rel_l2(a, b):
    a, b = a.float().cpu(), b.float().cpu()
    return float((a - b).norm() / b.norm())


def _tiny4(device):
    from mvoc_b200.unet3d import I2VGenXLUNet, UNetConfig, prepare
    from tests.golden import spec

    m = I2VGenXLUNet(UNetConfig.tiny4()).eval().requires_grad_(False)
    m.load_state_dict(spec.build_tiny4(seed=0).state_dict(), strict=True)
    return prepare(m.to(device, torch.bfloat16))


def _sample(pipe, inp, device, **kw):
    bf = lambda x: None if x is None else x.to(device, torch.bfloat16)  # noqa: E731
    return pipe.sample(bf(inp["prompt_embeds"]), bf(inp.get("negative_prompt_embeds")), bf(inp["image_embeddings"]),
                       bf(inp["image_latents"]), inp["fps"].to(device), **kw)


def test_sample_tiny4_10_guided_steps_vs_oracle(cuda_device):
    """The reference-golden seam conditioning of inversion_loop_tiny4.pt plus a seeded negative prompt, all 10 steps
    at guidance 9, CUDA graphs on."""
    from mvoc_b200.pipeline import I2VGenXLPipeline
    from oracle.sampling import sample_loop
    from tests.golden import spec
    from tests.test_recon_cpu import seam_inputs

    inp = seam_inputs()
    x0 = torch.randn(1, 4, 4, 16, 16, generator=torch.Generator().manual_seed(5))
    ref_rec, rec = [], []
    ref = sample_loop(spec.build_tiny4(seed=0), inp, 10, 9.0, x0, record=ref_rec)
    pipe = I2VGenXLPipeline(_tiny4(cuda_device), cuda_device, use_cuda_graphs=True)
    out = _sample(pipe, inp, cuda_device, num_inference_steps=10, guidance_scale=9.0, latents=x0,
                  callback=lambda i, t, lat: rec.append(lat.float().cpu()))
    torch.cuda.synchronize()
    errs = [rel_l2(a, b) for a, b in zip(rec, ref_rec)]
    print(f"[sample tiny4, cfg 9, 10 steps] rel L2 per step {[f'{e:.2e}' for e in errs]} (bar {BAR_TINY4_10:.0e})")
    assert len(rec) == 10 and torch.isfinite(out).all()
    assert rel_l2(out, ref) <= BAR_TINY4_10


def test_sample_full_model_one_guided_step_vs_oracle(cuda_device):
    """UNetConfig.full() (1.42 B parameters) at config 2's 64x64 latents with 2 of its 16 frames, one step at
    guidance 9 (batch 2)."""
    from mvoc_b200 import synthetic
    from mvoc_b200.pipeline import I2VGenXLPipeline
    from oracle import pipeline as opipe
    from oracle.sampling import sample_loop
    from tests.test_pipeline_gpu import _product_from

    wl = synthetic.WORKLOADS["config2_t2"]
    inp = synthetic.make_inversion_inputs(wl)
    x0 = torch.randn(1, 4, wl.n_frames, wl.latent_h, wl.latent_w, generator=torch.Generator().manual_seed(12))
    ou = opipe.build_unet(wl.unet, seed=0)
    ref = sample_loop(ou, inp, 50, 9.0, x0, max_steps=1)
    pipe = I2VGenXLPipeline(_product_from(ou, wl, cuda_device), cuda_device)
    del ou
    out = _sample(pipe, inp, cuda_device, num_inference_steps=50, guidance_scale=9.0, latents=x0, max_steps=1)
    torch.cuda.synchronize()
    err = rel_l2(out, ref)
    print(f"[sample full model 2x64x64, cfg 9, one step] latents rel L2 {err:.4e} (bar {BAR_FULL_STEP:.0e})")
    assert err <= BAR_FULL_STEP


def test_sample_graphs_and_generator_are_deterministic(cuda_device):
    """Eager and CUDA-graph runs give the same bits; two runs from the same seed give the same bits."""
    from mvoc_b200.pipeline import I2VGenXLPipeline
    from tests.test_recon_cpu import seam_inputs

    inp = seam_inputs()
    unet = _tiny4(cuda_device)
    runs = {}
    for graphs in (False, True):
        pipe = I2VGenXLPipeline(unet, cuda_device, use_cuda_graphs=graphs)
        for rep in range(2):
            g = torch.Generator(device=cuda_device).manual_seed(9)
            runs[(graphs, rep)] = _sample(pipe, inp, cuda_device, num_inference_steps=10, guidance_scale=9.0,
                                          generator=g, max_steps=4).clone()
    torch.cuda.synchronize()
    base = runs[(False, 0)]
    assert base.device.type == "cuda" and torch.isfinite(base).all()
    for k, v in runs.items():
        assert torch.equal(v, base), k


@pytest.mark.parametrize("K", [10])
def test_invert_then_sample_round_trip(cuda_device, K):
    """invert with K steps, then sample K steps from its last latents at guidance 1 under the same conditioning: both
    loops use DDIMSchedule(K), so the sampling grid starts where the inversion ended.  The product's distance to x0
    stays within 2x of the oracle's own round trip: the two GPU loops are each other's inverse."""
    from mvoc_b200.pipeline import I2VGenXLPipeline
    from oracle import pipeline as opipe
    from oracle.sampling import sample_loop
    from tests.golden import spec
    from tests.test_recon_cpu import seam_inputs

    inp = seam_inputs()
    x0 = spec.inversion_init_latents(spec.inversion_fixture())
    ou = spec.build_tiny4(seed=0)
    inv_in = dict(inp, latents=x0)
    o_saved = opipe.invert_loop(ou, None, inv_in, n_steps=K)
    o_back = sample_loop(ou, inp, K, 1.0, o_saved[max(o_saved)])
    d_oracle = rel_l2(o_back, x0)
    bf = lambda x: x.to(cuda_device, torch.bfloat16)  # noqa: E731
    pipe = I2VGenXLPipeline(_tiny4(cuda_device), cuda_device, use_cuda_graphs=True)
    saved = pipe.invert(x0.to(cuda_device).clone(), bf(inp["prompt_embeds"]), bf(inp["image_embeddings"]),
                        bf(inp["image_latents"]), inp["fps"].to(cuda_device), num_inference_steps=K)
    assert len(saved) == K
    back = _sample(pipe, inp, cuda_device, num_inference_steps=K, guidance_scale=1.0, latents=saved[max(saved)])
    torch.cuda.synchronize()
    d_prod = rel_l2(back, x0)
    print(f"[round trip K={K}] product |x0' - x0| / |x0| = {d_prod:.4e}, oracle {d_oracle:.4e}, "
          f"x_T product vs oracle {rel_l2(saved[max(saved)], o_saved[max(o_saved)]):.3e}")
    assert d_prod <= ROUND_TRIP_FACTOR * d_oracle


def _write_vae(path):
    """A random-init full-width AutoencoderKL file: encoder and decoder under diffusers' names."""
    from oracle import vae as ovae
    from oracle import vae_encoder as oenc
    from tests.test_vae_cpu import diffusers_state_dict
    from tests.test_vae_encode_cpu import diffusers_encoder_state_dict

    sd = diffusers_encoder_state_dict(oenc.build_encoder(narrow=False, seed=1).state_dict())
    sd.update(diffusers_state_dict(ovae.build_decoder(narrow=False, seed=2).state_dict()))
    torch.save(sd, path)


def test_inverse_script_reconstructs(cuda_device, tmp_path):
    """--synthetic --vae_state_dict FILE with enable_recon: T PNGs of 8h x 8w and recon_latents.synthetic.pt; without
    enable_recon the outputs are byte-identical to a template without the recon_config key."""
    import yaml
    from PIL import Image

    from mvoc_b200 import config as cfgmod
    from mvoc_b200 import inverse

    vae_path = str(tmp_path / "vae.pt")
    _write_vae(vae_path)
    T, w_px, h_px = 2, 128, 64
    template = os.path.join(ROOT, "configs", "group_inversion", "template.yaml")
    t = cfgmod.load_template(template)
    t.pop("recon_config")
    no_recon_template = tmp_path / "template_no_recon.yaml"
    no_recon_template.write_text(yaml.safe_dump(t))

    def entry(run, recon=None):
        data = tmp_path / run
        data.mkdir()
        e = {"active": True, "force_recompute_latents": True, "video_name": "clip", "data_dir": str(data),
             "image_size": [w_px, h_px], "n_frames": T}
        if recon is not None:
            e["recon_config"] = recon
        cfg = data / "group.json"
        cfg.write_text(json.dumps([e]))
        return data / "inversions" / "i2vgen-xl" / "clip", str(cfg)

    out, cfg = entry("recon", {"enable_recon": True, "n_steps": 25})
    assert inverse.main(template, cfg, synthetic_inputs=True, vae_state_dict=vae_path, max_steps=2) == 1
    lat = torch.load(out / "recon" / "recon_latents.synthetic.pt")
    assert lat.shape == (1, 4, T, h_px // 8, w_px // 8) and lat.dtype == torch.float32 and torch.isfinite(lat).all()
    frames = sorted(os.listdir(out / "recon" / "recon_frames.synthetic"))
    assert frames == [f"{i:03d}.png" for i in range(T)]
    for f in frames:
        assert Image.open(out / "recon" / "recon_frames.synthetic" / f).size == (w_px, h_px)
    assert not (out / "recon" / "recon_latents.pt").exists()

    out_a, cfg_a = entry("off")
    out_b, cfg_b = entry("absent")
    torch.manual_seed(0)                                        # --synthetic: random-init UNet weights
    assert inverse.main(template, cfg_a, synthetic_inputs=True, vae_state_dict=vae_path, max_steps=2) == 1
    torch.manual_seed(0)
    assert inverse.main(str(no_recon_template), cfg_b, synthetic_inputs=True, vae_state_dict=vae_path,
                        max_steps=2) == 1
    assert sorted(os.listdir(out_a)) == sorted(os.listdir(out_b)) == ["ddim_latents"]
    names = sorted(os.listdir(out_a / "ddim_latents"))
    assert names == sorted(os.listdir(out_b / "ddim_latents")) and len(names) == 2
    for n in names:
        assert (out_a / "ddim_latents" / n).read_bytes() == (out_b / "ddim_latents" / n).read_bytes()
