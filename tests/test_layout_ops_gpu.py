"""The up blocks' skip-connection concat (mvoc_concat_lastdim) and the once-per-forward SiLU of the time embedding:
both change where the work runs, not what it computes, so the UNet's outputs are bit-identical to the torch ops they
replace."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("shape_a,cb", [((2, 8, 8, 320), 320), ((3, 5, 7, 640), 1280), ((1, 1, 1, 8), 16),
                                        ((4, 11, 20, 1280), 640), ((0, 4, 4, 64), 64)])
def test_concat_lastdim_equals_torch_cat(cuda_device, dtype, shape_a, cb):
    from mvoc_b200 import ops

    g = torch.Generator(device=cuda_device).manual_seed(1)
    a = torch.randn(shape_a, generator=g, device=cuda_device).to(dtype)
    b = torch.randn(shape_a[:-1] + (cb,), generator=g, device=cuda_device).to(dtype)
    assert torch.equal(ops.concat_lastdim(a, b), torch.cat([a, b], dim=-1))


def test_concat_lastdim_rejects_what_it_cannot_do(cuda_device):
    from mvoc_b200 import ops

    a = torch.zeros(2, 4, 4, 12, dtype=torch.bfloat16, device=cuda_device)
    with pytest.raises(RuntimeError, match="multiples of 8"):
        ops.concat_lastdim(a, a)
    a = torch.zeros(2, 4, 4, 16, device=cuda_device)
    with pytest.raises(RuntimeError, match="dtype"):
        ops.concat_lastdim(a, a)
    b = torch.zeros(2, 4, 16, 16, dtype=torch.bfloat16, device=cuda_device)
    with pytest.raises(ValueError, match="contiguous"):
        ops.concat_lastdim(b.transpose(1, 2), b)
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.concat_lastdim(b.cpu(), b.cpu())


def test_composition_step_bit_identical_to_torch_layout_ops(cuda_device, monkeypatch):
    """One composition step (every hook firing) and one plain guided sampling step give the same bits with the library
    concat + shared SiLU as with torch.cat + a SiLU per resnet."""
    from mvoc_b200 import synthetic, unet3d
    from mvoc_b200.pipeline import I2VGenXLPipeline
    from mvoc_b200.scheduler import DDIMSchedule
    from oracle import pipeline as opipe
    from tests.test_pipeline_gpu import _product_from, _run_product_composite

    wl = synthetic.WORKLOADS["reduced2"]
    sched = DDIMSchedule(wl.n_steps)
    inputs = synthetic.make_inputs(wl, sched.timesteps, sched.alphas_cumprod)
    ou = opipe.build_unet(wl.unet, seed=0)
    inv = synthetic.make_inversion_inputs(wl)
    bf = lambda x: x.to(cuda_device, torch.bfloat16)  # noqa: E731

    def run():
        comp = _run_product_composite(wl, sched, inputs, _product_from(ou, wl, cuda_device), cuda_device, 2)
        pipe = I2VGenXLPipeline(_product_from(ou, wl, cuda_device), cuda_device)
        plain = pipe.sample(bf(inv["prompt_embeds"]), bf(inv["negative_prompt_embeds"]), bf(inv["image_embeddings"]),
                            bf(inv["image_latents"]), inv["fps"].to(cuda_device), num_inference_steps=50,
                            latents=inv["latents"], max_steps=2)
        torch.cuda.synchronize()
        return comp.clone(), plain.clone()

    calls = {"cat": 0, "silu": 0}
    real_cat = unet3d.cat_channels
    monkeypatch.setattr(unet3d, "cat_channels", lambda a, b: calls.__setitem__("cat", calls["cat"] + 1) or real_cat(a, b))
    mine = run()
    assert calls["cat"] > 0
    monkeypatch.setattr(unet3d, "cat_channels", lambda a, b: torch.cat([a, b], dim=-1))
    monkeypatch.setattr(unet3d, "_temb_act", lambda ctx, temb: F.silu(temb))
    torch_ops = run()
    for x, y in zip(mine, torch_ops):
        assert torch.isfinite(x).all() and torch.equal(x, y)
