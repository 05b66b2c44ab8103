"""composite.py frame-parallel under torchrun on two GPUs against one GPU, and a composition whose image latents are
encoded from its control frames (--encode_image_latents)."""
import json
import os
import signal
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TEMPLATE = os.path.join(ROOT, "configs", "group_composite", "template.yaml")
PARITY_BAR = 5e-3          # bench.py's multi-rank bar (bf16, only the merge order of GroupNorm statistics differs)

pytestmark = pytest.mark.gpu


def rel_l2(a, b):
    return float((a.float() - b.float()).norm() / b.float().norm())


def _entry(data_dir, **kw):
    e = {"active": True, "video_name": "fp", "edited_video_name": "fp edit", "data_dir": str(data_dir),
         "image_size": [512, 512], "n_frames": 16, "n_steps": 4, "ddim_init_latents_t_idx": 0, "fusion_step": [0, 1],
         "random_noise_ratio": 0.0, "pnp_f_t": 0.5, "pnp_spatial_attn_t": 1.0, "pnp_temp_attn_t": 1.0,
         "obj_mask_path": ["m0", "m1"], "obj_ddim_latents_path": ["l0", "l1"]}
    e.update(kw)
    return e


def _out_dir(data_dir, e):
    return os.path.join(str(data_dir), "Results", "MVOC-B200", "i2vgen-xl", e["video_name"], e["edited_video_name"])


def _vae_file(path, encoder=False):
    """A full-width random-init AutoencoderKL state dict: the decoder side, and with encoder=True the encoder side."""
    from oracle import vae as ovae
    from tests.test_vae_cpu import diffusers_state_dict

    sd = diffusers_state_dict(ovae.build_decoder(narrow=False, seed=1).state_dict())
    if encoder:
        from oracle import vae_encoder as oenc
        from tests.test_vae_encode_cpu import diffusers_encoder_state_dict

        sd.update(diffusers_encoder_state_dict(oenc.build_encoder(narrow=False, seed=1).state_dict()))
    torch.save(sd, path)


def _frames(d):
    from PIL import Image

    return {n: np.asarray(Image.open(os.path.join(d, n)), dtype=np.int16) for n in sorted(os.listdir(d))}


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 visible GPUs")
def test_composite_torchrun_two_gpus_matches_one_gpu(cuda_device, tmp_path):
    """`torch.distributed.run --nproc-per-node 2 -m mvoc_b200.composite --synthetic --vae_state_dict FILE` on a
    16-frame 512 x 512 entry with two objects: its latents are within the multi-rank bar of the same entry on one GPU,
    and each of its 16 frames (half written by each rank) is within 1 uint8 level of the one-GPU frame at >= 99.9 %
    of the pixels.  The UNet weights come from one file (random-init weights differ between processes)."""
    from mvoc_b200 import composite
    from mvoc_b200.unet3d import I2VGenXLUNet, UNetConfig

    vae_path = str(tmp_path / "vae.pt")
    _vae_file(vae_path)
    unet_path = str(tmp_path / "unet.pt")
    torch.manual_seed(0)
    with torch.device(cuda_device):
        unet = I2VGenXLUNet(UNetConfig.full())
    torch.save({k: v.to("cpu", torch.bfloat16) for k, v in unet.state_dict().items()}, unet_path)
    del unet
    torch.cuda.empty_cache()

    runs = {}
    for name in ("two", "one"):
        data = tmp_path / name
        data.mkdir()
        e = _entry(data)
        cfg = data / "group.json"
        cfg.write_text(json.dumps([e]))
        runs[name] = (data, e)
        args = ["--template_config", TEMPLATE, "--configs_json", str(cfg), "--synthetic", "--vae_state_dict",
                vae_path, "--unet_state_dict", unet_path]
        if name == "one":
            assert composite.main(TEMPLATE, str(cfg), unet_path, synthetic_inputs=True, vae_state_dict=vae_path) == 1
            continue
        env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""))
        env.pop("MVOC_EXCHANGE_ARENA_MB", None)
        cmd = [sys.executable, "-m", "torch.distributed.run", "--standalone", "--nproc-per-node", "2",
               "-m", "mvoc_b200.composite"] + args
        p = subprocess.Popen(cmd, cwd=ROOT, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True,
                             start_new_session=True)
        try:
            out, _ = p.communicate(timeout=900)
        except subprocess.TimeoutExpired:
            os.killpg(p.pid, signal.SIGKILL)           # torchrun and both ranks: nothing is left behind
            out, _ = p.communicate()
            pytest.fail("torchrun composite did not finish in 900 s:\n" + out[-4000:])
        assert p.returncode == 0, out[-4000:]

    (d2, e2), (d1, e1) = runs["two"], runs["one"]
    lat2 = torch.load(os.path.join(_out_dir(d2, e2), "composite_latents.synthetic.pt"))
    lat1 = torch.load(os.path.join(_out_dir(d1, e1), "composite_latents.synthetic.pt"))
    assert lat2.shape == lat1.shape == (1, 4, 16, 64, 64)
    err = rel_l2(lat2, lat1)
    print(f"two GPUs vs one: rel-L2 {err:.3e}")
    assert err <= PARITY_BAR, f"{err:.3e}"
    f2 = _frames(os.path.join(_out_dir(d2, e2), "composite_frames.synthetic"))
    f1 = _frames(os.path.join(_out_dir(d1, e1), "composite_frames.synthetic"))
    assert sorted(f2) == sorted(f1) == [f"{t:03d}.png" for t in range(16)]
    for n in f1:
        assert f2[n].shape == (512, 512, 3)
        close = float((np.abs(f2[n] - f1[n]) <= 1).mean())
        assert close >= 0.999, f"{n}: {close:.5f} of the pixels within 1 level"


def test_composite_encodes_image_latents_from_control_frames(cuda_device, tmp_path, monkeypatch):
    """--encode_image_latents with a full-width AutoencoderKL file: the image latents reaching the loop are
    prepare_image_latents of the first control frames ([bg, objs, main, main], one seeded draw), the loop runs, and
    the frames are written."""
    from PIL import Image

    from mvoc_b200 import composite
    from mvoc_b200.vae import center_crop_wide, pil_to_model_input

    vae_path = str(tmp_path / "vae.pt")
    _vae_file(vae_path, encoder=True)
    T, w_px, h_px = 2, 128, 64
    g = torch.Generator().manual_seed(5)
    rnd = lambda: Image.fromarray(torch.randint(0, 256, (80, 160, 3), generator=g, dtype=torch.uint8).numpy())
    images = [rnd() for _ in range(4)]                                          # bg, obj0, obj1, main
    (tmp_path / "bg").mkdir()
    images[0].save(tmp_path / "bg" / "000.png")
    for j in range(2):
        images[1 + j].save(tmp_path / f"obj{j}.png")
    images[3].save(tmp_path / "main.png")
    e = _entry(tmp_path, image_size=[w_px, h_px], n_frames=T, n_steps=2, seed=6,
               edited_contorl_frame_path_background="bg", edited_contorl_frame_path=["obj0.png", "obj1.png"],
               edited_contorl_frame_path_main="main.png")
    cfg = tmp_path / "group.json"
    cfg.write_text(json.dumps([e]))
    seen = {}
    real = composite.run_entry

    def run_entry(pipe, config, device, conditioning=None, allow_synthetic=False):
        seen.update(pipe=pipe, cond=conditioning)
        return real(pipe, config, device, conditioning, allow_synthetic)

    monkeypatch.setattr(composite, "run_entry", run_entry)
    torch.manual_seed(0)
    assert composite.main(TEMPLATE, str(cfg), synthetic_inputs=True, vae_state_dict=vae_path,
                          encode_image_latents=True) == 1
    pipe, cond = seen["pipe"], seen["cond"]
    x = pil_to_model_input([center_crop_wide(im, (w_px, h_px)) for im in images]).to(cuda_device)
    want = pipe.prepare_image_latents(x, T, torch.Generator().manual_seed(6))
    want = torch.cat([want, want[-1:]])
    assert cond["image_latents"].shape == (5, 4, T, h_px // 8, w_px // 8)
    assert torch.equal(cond["image_latents"], want) and torch.equal(cond["image_latents_first"], want)
    out = _out_dir(tmp_path, e)
    lat = torch.load(os.path.join(out, "composite_latents.synthetic.pt"))
    assert lat.shape == (1, 4, T, h_px // 8, w_px // 8) and torch.isfinite(lat).all()
    assert sorted(os.listdir(os.path.join(out, "composite_frames.synthetic"))) == [f"{t:03d}.png" for t in range(T)]
