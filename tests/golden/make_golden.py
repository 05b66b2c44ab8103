"""Generates tests/golden/*.pt by executing the REFERENCE'S OWN code (run in the build container only).

    python tests/golden/make_golden.py            # needs /root/reference; writes tests/golden/*.pt

What is executed from /root/reference (unmodified, loaded from where it lies):
  * i2vgen-xl/pnp_utils.py   — modify_diffuser_attention_forward, register_spatial_attention_pnp,
                               register_temp_attention_pnp, register_resnet_injection,
                               register_temp_conv_injection, register_out_conv_injection, register_time_all
  * i2vgen-xl/composite.py   — init_pnp
  * i2vgen-xl/pipelines/pipeline_i2vgen_xl.py — I2VGenXLUnetExtension.forward
  * i2vgen-xl/utils.py       — load_ddim_latents_at_t (wire format round trip)

Their third-party imports (diffusers 0.27.2, omegaconf, transformers CLIP, torchvision.io.read_video) are
not installed here, so they are stubbed: the ``diffusers`` classes the reference isinstance-checks /
subclasses are bound to the restated modules of ``oracle/unet.py`` (same attribute names), everything
else is an inert placeholder.  The module tree those functions then run over is therefore the oracle's
restatement of diffusers — what these vectors pin is the MVOC layer (hooks, processors, UNet driver,
injection schedule), which IS in the reference tree; diffusers internals stay unpinned (see oracle/unet.py).

The reference hard-codes the 4-level layout (up_blocks[1..3], three layers each) and `// 5` (two objects),
so the golden model is a narrow 4-level UNet ("tiny4": block_out_channels 64/128/256/256, head_dim 64)
with background + 2 objects.
"""
from __future__ import annotations

import importlib.util
import logging
import os
import shutil
import sys
import types
from types import SimpleNamespace

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
REF = "/root/reference/i2vgen-xl"

from oracle import unet as ou  # noqa: E402
from tests.golden import spec  # noqa: E402


class _Anything:
    """Inert placeholder: callable, subclassable, attribute-able."""

    def __init__(self, *a, **k):
        pass

    def __call__(self, *a, **k):
        return self

    def __getattr__(self, name):
        return _Anything()


class _StubModule(types.ModuleType):
    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)
        cls = type(name, (_Anything,), {})
        setattr(self, name, cls)
        return cls


def _stub(name: str, **attrs) -> types.ModuleType:
    m = _StubModule(name)
    m.__path__ = []  # behave like a package
    for k, v in attrs.items():
        setattr(m, k, v)
    sys.modules[name] = m
    return m


class _Out:
    def __init__(self, sample=None, **k):
        self.sample = sample


def install_stubs():
    identity_decorator = lambda *a, **k: (lambda f: f)
    _stub("diffusers", DiffusionPipeline=type("DiffusionPipeline", (), {}))
    _stub("diffusers.models", AutoencoderKL=_Anything)
    _stub("diffusers.models.attention_processor", AttnProcessor2_0=ou.AttnProcessor2_0, Attention=ou.Attention)
    _stub("diffusers.models.attention", BasicTransformerBlock=ou.BasicTransformerBlock,
          _chunked_feed_forward=lambda *a, **k: (_ for _ in ()).throw(RuntimeError("unused")))
    _stub("diffusers.models.transformers")
    _stub("diffusers.models.transformers.transformer_2d", Transformer2DModel=ou.Transformer2DModel,
          Transformer2DModelOutput=_Out)
    _stub("diffusers.models.transformers.transformer_temporal", TransformerTemporalModel=ou.TransformerTemporalModel,
          TransformerTemporalModelOutput=_Out, TransformerSpatioTemporalModel=type("TSTM", (), {}))
    _stub("diffusers.models.upsampling", Upsample2D=ou.Upsample2D)
    _stub("diffusers.models.downsampling", Downsample2D=ou.Downsample2D)
    _stub("diffusers.models.lora")
    _stub("diffusers.models.unets")
    _stub("diffusers.models.unets.unet_i2vgen_xl", I2VGenXLUNet=ou.I2VGenXLUNet, UNet3DConditionOutput=_Out)
    _stub("diffusers.image_processor")
    _stub("diffusers.loaders", LoraLoaderMixin=type("LoraLoaderMixin", (), {}))
    _stub("diffusers.schedulers")
    _stub("diffusers.utils", USE_PEFT_BACKEND=True, is_torch_version=lambda *a: True,
          BaseOutput=type("BaseOutput", (), {}), replace_example_docstring=identity_decorator,
          logging=SimpleNamespace(get_logger=logging.getLogger), load_image=_Anything(),
          export_to_video=_Anything(), export_to_gif=_Anything())
    _stub("diffusers.utils.torch_utils")
    _stub("omegaconf")
    _stub("transformers")
    import torchvision.io as tvio

    for n in ("read_video", "write_video"):
        if not hasattr(tvio, n):
            setattr(tvio, n, _Anything())


def load_ref(modname: str, relpath: str):
    spec_ = importlib.util.spec_from_file_location(modname, os.path.join(REF, relpath))
    mod = importlib.util.module_from_spec(spec_)
    sys.modules[modname] = mod
    spec_.loader.exec_module(mod)
    return mod


def main():
    assert os.path.isdir(REF), "run in the build container (needs /root/reference)"
    install_stubs()
    sys.path.insert(0, REF)
    sys.path.insert(0, os.path.dirname(REF))  # `common`
    ref_utils = load_ref("utils", "utils.py")
    ref_pnp = load_ref("pnp_utils", "pnp_utils.py")
    ref_pipe = load_ref("ref_pipeline_i2vgen_xl", "pipelines/pipeline_i2vgen_xl.py")
    ref_comp = load_ref("ref_composite", "composite.py")
    torch.set_grad_enabled(False)

    out = {}
    for case in spec.CASES:
        unet = spec.build_tiny4(seed=0)
        pipe = SimpleNamespace(unet=unet)
        sched = SimpleNamespace(timesteps=torch.tensor(spec.timesteps_50()))
        cfg = SimpleNamespace(n_steps=50, pnp_f_t=case["pnp_f_t"], pnp_spatial_attn_t=case["pnp_spatial_attn_t"],
                              pnp_temp_attn_t=case["pnp_temp_attn_t"], pnp_cross_attn_t=0.0,
                              inject_background=case["inject_background"])
        ref_comp.init_pnp(pipe, sched, cfg)                                   # composite.py:38-69 (real)
        inp = spec.make_inputs(case)
        masks = list(zip([m for m, _ in inp["masks"]], [b for _, b in inp["masks"]]))
        ref_pnp.register_time_all(pipe, case["t"], masks)                     # pnp_utils.py:48-166 (real)
        y = ref_pipe.I2VGenXLUnetExtension.forward(                            # pipeline:109-362 (real)
            unet, inp["sample"], torch.tensor(case["t"]), inp["fps"], inp["image_latents_first"],
            inp["image_latents"], inp["image_embeddings"], inp["prompt_embeds"], multi_frame_guidance=False,
            return_dict=False)[0]
        out[case["name"]] = y.clone()
        print(case["name"], tuple(y.shape), float(y.std()))
    torch.save(out, os.path.join(HERE, "unet_extension_forward_tiny4.pt"))

    # mask_preprocess (utils.py:92-154) on small synthetic PNG masks committed under tests/golden/masks
    from PIL import Image, ImageDraw, ImageFilter

    mdir = os.path.join(HERE, "masks")
    os.makedirs(os.path.join(mdir, "dynamic"), exist_ok=True)
    for i in range(5):  # 5 files: the reference truncates to `frames` (= 4) after a numeric sort
        im = Image.new("L", (128, 96), 0)
        ImageDraw.Draw(im).ellipse([20 + 6 * i, 24, 70 + 6 * i, 70], fill=255)
        im = im.filter(ImageFilter.GaussianBlur(2.5))
        if i == 2:
            im = im.convert("RGB")  # the demo folders mix modes (P / L / RGB)
        im.save(os.path.join(mdir, "dynamic", ["000.png", "001.png", "002.png", "003.png", "010.png"][i]))
    im = Image.new("L", (128, 96), 0)
    ImageDraw.Draw(im).rectangle([30, 10, 90, 60], fill=200)
    im.filter(ImageFilter.GaussianBlur(1.5)).save(os.path.join(mdir, "static.png"))
    mg = {}
    for name, path in (("dynamic", os.path.join(mdir, "dynamic")), ("static", os.path.join(mdir, "static.png"))):
        mf, mb = ref_utils.mask_preprocess(path, "cpu", torch.float32, 1, 4, 4, downscale=8)   # real reference code
        mg[name] = (mf.clone(), mb.clone())
        print("mask", name, tuple(mf.shape), float(mb.float().mean()))
    torch.save(mg, os.path.join(HERE, "mask_preprocess.pt"))

    # wire format: what the reference's loader reads back from a file written like pipeline:1990-1993
    lat = torch.randn(1, 4, 4, 8, 8, generator=torch.Generator().manual_seed(5)).half()
    d = os.path.join(HERE, "ddim_latents_fixture")
    os.makedirs(d, exist_ok=True)
    torch.save(lat.detach().clone(), os.path.join(d, f"ddim_latents_{torch.tensor(981)}.pt"))
    back = ref_utils.load_ddim_latents_at_t(torch.tensor(981), d)
    assert torch.equal(back, lat)

    # the reference's own config files, byte for byte (a few KB): the config loader is tested on them
    for sub in ("group_composite", "group_inversion"):
        os.makedirs(os.path.join(HERE, "reference_configs", sub), exist_ok=True)
        for name in ("template.yaml", "group_config.json"):
            shutil.copyfile(os.path.join(REF, "configs", sub, name), os.path.join(HERE, "reference_configs", sub, name))
    print("wrote goldens")


if __name__ == "__main__":
    main()
