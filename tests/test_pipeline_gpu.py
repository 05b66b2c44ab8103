"""GPU parity of the whole path: product UNet / composition loop / inversion loop (bf16, sm_100a kernels)
against the fp32 CPU oracle on the same weights and synthetic inputs.

Tolerance (SURVEY §8d): the error any bf16 implementation incurs is measured first by running the
oracle's own module tree in bf16 on the GPU (torch SDPA / ATen GroupNorm); the product must stay within
1.5x of that envelope (plus a small absolute floor).
"""
import copy
import os
from types import SimpleNamespace

import pytest
import torch

pytestmark = pytest.mark.gpu


def rel_l2(a, b):
    a, b = a.float().cpu(), b.float().cpu()
    return float((a - b).norm() / b.norm())


def _setup(wl_name):
    from mvoc_b200 import synthetic
    from mvoc_b200.scheduler import DDIMSchedule
    from oracle import pipeline as opipe

    wl = synthetic.WORKLOADS[wl_name]
    sched = DDIMSchedule(wl.n_steps)
    inputs = synthetic.make_inputs(wl, sched.timesteps, sched.alphas_cumprod)
    oracle_unet = opipe.build_unet(wl.unet, seed=0)
    return wl, sched, inputs, oracle_unet


def _product_from(oracle_unet, wl, device):
    from mvoc_b200.unet3d import I2VGenXLUNet, UNetConfig

    m = I2VGenXLUNet(UNetConfig.named(wl.unet)).eval().requires_grad_(False)
    m.load_state_dict(oracle_unet.state_dict(), strict=True)
    from mvoc_b200.unet3d import prepare

    return prepare(m.to(device=device, dtype=torch.bfloat16))


def _cond(inputs, device):
    from mvoc_b200.pipeline import Conditioning

    bf = lambda x: x.to(device=device, dtype=torch.bfloat16)
    return Conditioning(bf(inputs["prompt_embeds"]), bf(inputs["image_embeddings"]),
                        bf(inputs["image_latents_first"]), bf(inputs["image_latents"]),
                        inputs["fps"].to(device))


def _run_product_composite(wl, sched, inputs, unet, device, max_steps, host_io=False, graphs=False):
    from mvoc_b200.pipeline import I2VGenXLPipeline, LatentBank, init_pnp

    pipe = I2VGenXLPipeline(unet, device, use_cuda_graphs=graphs)
    init_pnp(pipe, sched, wl)
    banks = [LatentBank(src, device, pin_host=host_io) for src in inputs["source_latents"]]
    masks = [(mf.to(device), mb.to(device)) for mf, mb in inputs["masks"]]
    lat = inputs["init_latents"].to(device).clone()
    out = pipe.sample_with_pnp_pipeline_with_edit_prompt_extraction_with_attn_injection(
        _cond(inputs, device), lat, banks[0], banks[1:], masks, num_inference_steps=wl.n_steps,
        guidance_scale=wl.cfg, ddim_init_latents_t_idx=wl.ddim_init_latents_t_idx,
        fusion_steps=tuple(wl.fusion_step), random_noise_ratio=wl.random_noise_ratio,
        obj_random_noise_fusion=wl.obj_random_noise_fusion, max_steps=max_steps, host_io=host_io)
    torch.cuda.synchronize()
    return out


@pytest.mark.parametrize("wl_name", ["config1", "reduced2"])
def test_unet_forward_vs_oracle(cuda_device, wl_name):
    """One UNet forward with every hook firing (t = first timestep)."""
    from mvoc_b200.pipeline import I2VGenXLPipeline, init_pnp
    from mvoc_b200 import pnp_utils
    from oracle import hooks as ohooks
    from oracle import pipeline as opipe

    wl, sched, inputs, ou = _setup(wl_name)
    t = sched.timesteps[0]
    torch.manual_seed(11)
    sample = torch.randn(wl.n_branches, 4, wl.n_frames, wl.latent_h, wl.latent_w)
    ou16 = copy.deepcopy(ou).to(cuda_device, torch.bfloat16)  # before the hooks capture `ou` in closures
    # oracle fp32
    opipe_ns = SimpleNamespace(unet=ou)
    opipe.init_pnp(opipe_ns, torch.tensor(sched.timesteps), wl)
    ohooks.register_time_all(opipe_ns, t, inputs["masks"])
    ref = opipe.unet_extension_forward(ou, sample, t, inputs["fps"], inputs["image_latents_first"],
                                       inputs["image_latents"], inputs["image_embeddings"], inputs["prompt_embeds"])
    # envelope: the oracle's own tree in bf16 on the GPU
    ns16 = SimpleNamespace(unet=ou16)
    opipe.init_pnp(ns16, torch.tensor(sched.timesteps), wl)
    masks_d = [(mf.to(cuda_device), mb.to(cuda_device)) for mf, mb in inputs["masks"]]
    ohooks.register_time_all(ns16, t, masks_d)
    bf = lambda x: x.to(cuda_device, torch.bfloat16)
    env = opipe.unet_extension_forward(ou16, bf(sample), t, inputs["fps"].to(cuda_device), bf(inputs["image_latents_first"]),
                                       bf(inputs["image_latents"]), bf(inputs["image_embeddings"]),
                                       bf(inputs["prompt_embeds"]))
    env_err = rel_l2(env, ref)
    # product
    pu = _product_from(ou, wl, cuda_device)
    pipe = I2VGenXLPipeline(pu, cuda_device)
    init_pnp(pipe, sched, wl)
    pnp_utils.register_time_all(pipe, t, masks_d)
    out = pipe._gather_prediction(pipe._unet_forward(bf(sample), t, _cond(inputs, cuda_device)))
    torch.cuda.synchronize()
    err = rel_l2(out, ref)
    print(f"[{wl_name}] product rel L2 {err:.4e}; torch-bf16 envelope {env_err:.4e}")
    assert torch.isfinite(out.float()).all()
    assert err <= 1.5 * env_err + 2e-3, f"product {err:.3e} vs envelope {env_err:.3e}"


def test_composite_step_config1(cuda_device):
    """BASELINE config 1: reduced UNet, 8 x 32x32, bg + 1 object, one composite DDIM step."""
    from oracle import pipeline as opipe

    wl, sched, inputs, ou = _setup("config1")
    ref = opipe.composite_loop(copy.deepcopy(ou), wl, inputs, max_steps=1)
    out = _run_product_composite(wl, sched, inputs, _product_from(ou, wl, cuda_device), cuda_device, 1)
    err = rel_l2(out, ref)
    print(f"[config1, 1 step] latents rel L2 {err:.4e}")
    assert err <= 2e-2


def test_composite_multi_step_reduced2(cuda_device):
    """Two objects, 4 steps: fusion on step 0, conv injection on steps 0-4, attention injection throughout;
    device-resident and host-IO loops agree bit for bit."""
    from oracle import pipeline as opipe

    wl, sched, inputs, ou = _setup("reduced2")
    rec = []
    opipe.composite_loop(copy.deepcopy(ou), wl, inputs, max_steps=4, record=rec)
    pu = _product_from(ou, wl, cuda_device)
    out = _run_product_composite(wl, sched, inputs, pu, cuda_device, 4)
    err = rel_l2(out, rec[-1])
    print(f"[reduced2, 4 steps] latents rel L2 {err:.4e}")
    assert err <= 5e-2
    out_h = _run_product_composite(wl, sched, inputs, _product_from(ou, wl, cuda_device), cuda_device, 4, host_io=True)
    assert torch.equal(out.cpu(), out_h.cpu())
    # CUDA-graph replay of the UNet forward (one graph per hook configuration) == eager launches.
    # 7 steps: step 0 fuses, steps 0-4 inject features, steps 5-6 only inject attention => 2 graphs, replayed
    wl7 = wl
    eager7 = _run_product_composite(wl7, sched, inputs, _product_from(ou, wl, cuda_device), cuda_device, 7)
    graph7 = _run_product_composite(wl7, sched, inputs, _product_from(ou, wl, cuda_device), cuda_device, 7, graphs=True)
    assert torch.equal(eager7.cpu(), graph7.cpu())


def test_invert_reduced(cuda_device, tmp_path):
    """Inversion loop (3 of 500 steps) + ddim_latents_{t}.pt wire format."""
    from mvoc_b200 import synthetic
    from mvoc_b200.pipeline import I2VGenXLPipeline, load_ddim_latents_at_t
    from oracle import pipeline as opipe

    wl = synthetic.WORKLOADS["config1"]
    inv = synthetic.make_inversion_inputs(wl)
    ou = opipe.build_unet(wl.unet, seed=0)
    ref = opipe.invert_loop(ou, wl, inv, max_steps=3)
    pu = _product_from(ou, wl, cuda_device)
    pipe = I2VGenXLPipeline(pu, cuda_device)
    bf = lambda x: x.to(cuda_device, torch.bfloat16)
    saved = pipe.invert(inv["latents"].to(cuda_device).clone(), bf(inv["prompt_embeds"]), bf(inv["image_embeddings"]),
                        bf(inv["image_latents"]), inv["fps"].to(cuda_device), num_inference_steps=wl.inversion_steps,
                        output_dir=str(tmp_path), max_steps=3)
    torch.cuda.synchronize()
    assert sorted(saved) == sorted(ref) == [1, 3, 5]
    for t in saved:
        err = rel_l2(saved[t], ref[t])
        assert err <= 2e-2, f"t={t}: {err:.3e}"
        disk = load_ddim_latents_at_t(t, str(tmp_path))
        assert disk.shape == (1, 4, wl.n_frames, wl.latent_h, wl.latent_w)
        assert disk.dtype == torch.float16                  # the reference's wire dtype (pipeline_i2vgen_xl.py:1990)
        assert torch.equal(disk, saved[t].cpu().half())


@pytest.mark.parametrize("case_name", ["all_hooks_t981", "attn_only_t481", "inject_bg_t481", "no_hooks_t21"])
def test_unet_forward_vs_reference_golden(cuda_device, case_name):
    """Product (bf16 kernels) against the output of the REFERENCE'S OWN code on the 4-level golden model
    (tests/golden/unet_extension_forward_tiny4.pt, produced by tests/golden/make_golden.py)."""
    import os

    from mvoc_b200 import pnp_utils
    from mvoc_b200.pipeline import Conditioning, I2VGenXLPipeline, init_pnp
    from mvoc_b200.scheduler import DDIMSchedule
    from mvoc_b200.unet3d import I2VGenXLUNet, UNetConfig
    from tests.golden import spec

    gold = torch.load(os.path.join(os.path.dirname(__file__), "golden", "unet_extension_forward_tiny4.pt"),
                      map_location="cpu")
    case = next(c for c in spec.CASES if c["name"] == case_name)
    ou = spec.build_tiny4(seed=0)
    pu = I2VGenXLUNet(UNetConfig.tiny4()).eval().requires_grad_(False)
    pu.load_state_dict(ou.state_dict(), strict=True)
    from mvoc_b200.unet3d import prepare

    pu = prepare(pu.to(cuda_device, torch.bfloat16))
    pipe = I2VGenXLPipeline(pu, cuda_device)
    cfg = SimpleNamespace(n_steps=50, pnp_f_t=case["pnp_f_t"], pnp_spatial_attn_t=case["pnp_spatial_attn_t"],
                          pnp_temp_attn_t=case["pnp_temp_attn_t"], inject_background=case["inject_background"])
    init_pnp(pipe, DDIMSchedule(50), cfg)
    inp = spec.make_inputs(case)
    masks = [(mf.to(cuda_device), mb.to(cuda_device)) for mf, mb in inp["masks"]]
    pnp_utils.register_time_all(pipe, case["t"], masks)
    out = pipe._gather_prediction(pipe._unet_forward(inp["sample"].to(cuda_device, torch.bfloat16), case["t"],
                                                     _cond(inp, cuda_device)))
    torch.cuda.synchronize()
    ref = gold[case_name]
    err = rel_l2(out, ref)
    comp = rel_l2(out[3:], ref[3:])
    print(f"[golden {case_name}] rel L2 all {err:.4e}, composite branches {comp:.4e}")
    assert err <= 3e-2 and comp <= 3e-2


def test_bench_steps_and_dump_outputs(cuda_device, tmp_path, monkeypatch, capsys):
    """bench.py --steps K times exactly K steps: past the end of the schedule (47 steps here, it starts at index 3)
    it starts again from the initial latents, so 48 steps end where 1 step does.  --dump-outputs writes those
    latents after the JSON line."""
    import dataclasses
    import json
    import sys

    import numpy as np

    import bench
    from mvoc_b200 import synthetic

    wl = dataclasses.replace(synthetic.WORKLOADS["config1"], name="config1_from_idx3", ddim_init_latents_t_idx=3)
    monkeypatch.setitem(synthetic.WORKLOADS, wl.name, wl)
    monkeypatch.setattr(torch.backends.cudnn, "benchmark", torch.backends.cudnn.benchmark)   # restored afterwards
    out = {}
    for k in (1, 48):
        d = tmp_path / f"k{k}"
        monkeypatch.setattr(sys, "argv", ["bench.py", "--workload", wl.name, "--steps", str(k), "--warmup", "1",
                                          "--no-cpu-baseline", "--dump-outputs", str(d)])
        bench.main()
        line = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
        assert line["steps"] == k
        assert sorted(os.listdir(d)) == ["latents.npy"]
        out[k] = np.load(d / "latents.npy")
    assert out[1].dtype == np.float32 and out[1].shape == (1, 4, wl.n_frames, wl.latent_h, wl.latent_w)
    assert rel_l2(torch.from_numpy(out[48]), torch.from_numpy(out[1])) <= 1e-3
