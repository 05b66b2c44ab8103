"""`inverse.py` of the reference (i2vgen-xl/inverse.py) over the B200 path.

    python -m mvoc_b200.inverse --template_config configs/group_inversion/template.yaml \\
                                --configs_json configs/group_inversion/group_config.json

Same flags and config contract (inverse.py:230-255, :136-150).  Per active entry it runs the DDIM inversion
loop (pipelines/pipeline_i2vgen_xl.py:1940-2000; `inverse_config.n_steps`, cfg 1.0 => batch 1) and writes one
`ddim_latents_{t}.pt` per timestep into `inverse_config.output_dir` (:1988-1993) — the wire format
`composite.py` reads.  Like the reference it skips entries that were already inverted unless
`force_recompute_latents` (inverse.py:181-183) — "already inverted" means that EVERY expected
`ddim_latents_{t}.pt` is present (the reference only tests for the directory, so a crashed or `--max_steps` run is
never completed and composite.py later asserts on the missing timesteps).

The clean video latents / prompt / CLIP tensors are read from `--inputs file.pt` (dict: latents [1,4,T,h,w],
prompt_embeds [1,77,1024], image_embeddings [1,1,1024], image_latents [1,4,T,h,w]; `{video_name}` in the path
selects one file per entry).  A missing file is an error; `--synthetic` substitutes seeded synthetic tensors and
random UNet weights.

With `--vae_state_dict FILE` (a diffusers AutoencoderKL state dict) the video latents and the first-frame image
latents are computed here, as inverse.py:143-153 and :49-55 do: the first `n_frames` .png / .jpg files of
`<video_dir>/<video_name>/` are centre-cropped to `image_size` and encoded with one
`torch.Generator().manual_seed(seed)` per entry, first the video (`encode_vae_video`), then the first frame
(`prepare_image_latents`).  `--inputs` then only needs prompt_embeds and image_embeddings (unless the CLIP flags
below compute them; the reference's mp4 fallback, :154-165, stays out of scope).  With `--synthetic` and no frame
directory, seeded synthetic frames are encoded; the encoder weights always come from FILE.

With `--image_encoder_state_dict FILE` (a transformers CLIPVisionModelWithProjection state dict) `image_embeddings`
[1,1,1024] is computed here from the first frame of the same directory: centre-cropped to (width, width), resized to
224 x 224 and CLIP-normalised (mvoc_b200.clip.clip_image_input), then encoded on the library's kernels.  It works with
or without `--vae_state_dict`; with both, `--inputs` only needs prompt_embeds.  `--synthetic` without a frame
directory encodes the first seeded synthetic frame.

With `--text_encoder_state_dict FILE` (a transformers CLIPTextModel state dict) and `--tokenizer_dir DIR` (the
checkpoint's tokenizer/ folder) `prompt_embeds` [1,77,1024] is `encode_prompt(inverse_config.prompt)` (batch 1: the
inversion runs at cfg 1.0).  The two flags go together; `--synthetic` never invents text weights or a vocabulary.
With the VAE, image and text flags all given, every input is computed here and `--inputs` is not needed.

With `recon_config.enable_recon: true` an entry is also reconstructed after its inversion (also when the inversion was
skipped as complete), the reference's sanity check (inverse.py:192-227): the noisiest stored latents of
`recon_config.ddim_latents_path` (utils.load_ddim_latents_at_T) are sampled back with the plain I2VGenXL loop
(`I2VGenXLPipeline.sample`, `recon_config.n_steps` steps, guidance `recon_config.cfg`) under the entry's own
conditioning, and the result is written to `<recon_config.output_dir>/recon_latents.pt`.  Under guidance the negative
prompt is `encode_prompt(inverse_config.negative_prompt)` with the text flags, else `negative_prompt_embeds` of
`--inputs` (seeded under `--synthetic`).  With `--vae_state_dict` the result is also decoded to `recon_frames/NNN.png`
(the decoder is read from the same file as the encoder).  `--synthetic` writes `.synthetic` names, and `--max_steps`
caps the sampling loop as it caps the inversion.

Independent videos are the unit of multi-GPU work here: with torchrun, entry i goes to rank i % world_size
(replicas, no collective).
"""
from __future__ import annotations

import argparse
import logging
import os

import torch

from . import config as cfgmod
from . import synthetic

logger = logging.getLogger(__name__)

# recon_config defaults when the merged entry lacks the keys: diffusers' I2VGenXLPipeline.__call__ defaults (the
# reference's own values could not be read); the template states them and an entry overrides them
RECON_STEPS = 50
RECON_CFG = 9.0


def inversion_complete(out_dir: str, n_steps: int) -> bool:
    """True when every ddim_latents_{t}.pt of an n_steps inversion exists in out_dir."""
    from .pipeline import ddim_latents_filename
    from .scheduler import DDIMSchedule

    if not os.path.isdir(out_dir):
        return False
    return all(os.path.exists(os.path.join(out_dir, ddim_latents_filename(t)))
               for t in DDIMSchedule(n_steps, inverse=True).timesteps)


def synthetic_frames(n_frames: int, height: int, width: int, seed: int) -> torch.Tensor:
    """Seeded uint8 noise frames as model input: [n_frames, 3, height, width] fp32 in [-1, 1]."""
    g = torch.Generator().manual_seed(seed)
    return torch.randint(0, 256, (n_frames, 3, height, width), generator=g, dtype=torch.uint8).float() / 127.5 - 1.0


def encode_entry(pipe, config, idx: int, synthetic_inputs: bool, device):
    """(video latents [1,4,T,h,w], first-frame image latents [1,4,T,h,w]) of one entry, fp32 on `device`."""
    from .vae import load_frames

    inv = config.inverse_config
    w_px, h_px = inv.image_size
    n_frames = int(inv.n_frames)
    frame_dir = os.path.join(str(config.get("video_dir", ".")), str(config.video_name))
    if os.path.isdir(frame_dir) or not synthetic_inputs:
        frames = load_frames(frame_dir, n_frames, (int(w_px), int(h_px)))
    else:
        logger.info("%s not found: encoding seeded synthetic frames (--synthetic)", frame_dir)
        frames = synthetic_frames(n_frames, int(h_px), int(w_px), 9000 + idx)
    frames = frames.to(device)
    generator = torch.Generator().manual_seed(int(config.get("seed", 0)))
    latents = pipe.encode_vae_video(frames, generator)                         # inverse.py:49-55
    image_latents = pipe.prepare_image_latents(frames[:1], n_frames, generator)   # inside invert (:860-890)
    return latents, image_latents


def image_embeddings_entry(pipe, config, idx: int, synthetic_inputs: bool) -> torch.Tensor:
    """CLIP image_embeddings [1,1,1024] of one entry's first frame (the frame directory of encode_entry)."""
    from PIL import Image

    from .clip import clip_image_input, first_frame

    inv = config.inverse_config
    w_px, h_px = (int(v) for v in inv.image_size)
    frame_dir = os.path.join(str(config.get("video_dir", ".")), str(config.video_name))
    if os.path.isdir(frame_dir) or not synthetic_inputs:
        image = first_frame(frame_dir)
    else:
        logger.info("%s not found: encoding the first seeded synthetic frame (--synthetic)", frame_dir)
        f0 = synthetic_frames(1, h_px, w_px, 9000 + idx)[0]
        image = Image.fromarray(((f0 + 1.0) * 127.5).round().to(torch.uint8).permute(1, 2, 0).numpy())
    return pipe.encode_image(clip_image_input(image, w_px))


def main(template_config: str, configs_json: str, unet_state_dict: str = None, inputs: str = None,
         device: str = None, max_steps: int = None, synthetic_inputs: bool = False, vae_state_dict: str = None,
         image_encoder_state_dict: str = None, text_encoder_state_dict: str = None, tokenizer_dir: str = None):
    from .clip_text import check_text_flags, load_text_tower
    from .pipeline import I2VGenXLPipeline
    from .unet3d import I2VGenXLUNet, UNetConfig, prepare

    check_text_flags(text_encoder_state_dict, tokenizer_dir)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    template = cfgmod.load_template(template_config)
    device = torch.device(device or (f"cuda:{local}" if world > 1 else template.get("device", "cuda:0")))
    if device.type == "cuda":
        torch.cuda.set_device(device)      # the C-ABI launches on the current device (mvoc_b200.ops._need_cuda)
    torch.set_grad_enabled(False)
    unet = I2VGenXLUNet(UNetConfig.full()).eval().requires_grad_(False)
    if unet_state_dict:
        unet.load_state_dict(torch.load(unet_state_dict, map_location="cpu"), strict=True)
    elif not synthetic_inputs:
        raise FileNotFoundError("--unet_state_dict is required (pass --synthetic to run on random-init weights)")
    unet = prepare(unet.to(device=device, dtype=torch.bfloat16))
    vae_encoder = None
    if vae_state_dict:
        from .vae import load_vae_encoder

        vae_encoder = load_vae_encoder(vae_state_dict, device)
    image_encoder = None
    if image_encoder_state_dict:
        from .clip import load_clip_image_encoder

        image_encoder = load_clip_image_encoder(image_encoder_state_dict, device)
    text_encoder, tokenizer = load_text_tower(text_encoder_state_dict, tokenizer_dir, device)
    pipe = I2VGenXLPipeline(unet, device, use_cuda_graphs=device.type == "cuda", vae_encoder=vae_encoder,
                            image_encoder=image_encoder, text_encoder=text_encoder, tokenizer=tokenizer)
    computes_all = vae_encoder is not None and image_encoder is not None and text_encoder is not None
    done = 0
    for idx, config in enumerate(cfgmod.iter_configs(template_config, configs_json)):
        if idx % world != rank:
            continue                                                            # one video per GPU
        inv = config.inverse_config
        out_dir = inv.output_dir
        recon = config.get("recon_config") or {}
        do_recon = bool(recon.get("enable_recon", False))
        skip = inversion_complete(out_dir, int(inv.n_steps)) and not config.get("force_recompute_latents", False)
        if skip:
            logger.info("%s is complete: skipping (force_recompute_latents is false)", out_dir)   # inverse.py:181-183
            if not do_recon:
                continue
        w_px, h_px = inv.image_size
        wl = synthetic.Workload(config.video_name, "full", int(inv.n_frames), int(h_px) // 8, int(w_px) // 8, 0,
                                inversion_steps=int(inv.n_steps))
        if inputs:
            ipath = inputs.format(video_name=config.video_name)
            if not os.path.exists(ipath):
                raise FileNotFoundError(f"inversion inputs {ipath!r} not found")
            src = torch.load(ipath, map_location="cpu")
        elif computes_all:
            src = {}                                                            # every input is computed below
        elif synthetic_inputs:
            src = synthetic.make_inversion_inputs(wl, idx)
        else:
            raise FileNotFoundError("no --inputs file (VAE / CLIP outputs are inputs of this script unless "
                                    "--vae_state_dict, --image_encoder_state_dict and --text_encoder_state_dict with "
                                    "--tokenizer_dir compute them all); pass --synthetic for seeded synthetic tensors")
        if vae_encoder is not None:
            if inputs and any(k in src for k in ("latents", "image_latents")):
                logger.info("%s: latents / image_latents of the inputs file are not read (--vae_state_dict encodes "
                            "the frames)", config.video_name)
            latents, image_latents = encode_entry(pipe, config, idx, synthetic_inputs, device)
        else:
            latents, image_latents = src["latents"].to(device).float().clone(), src["image_latents"]
        if image_encoder is not None:
            if inputs and "image_embeddings" in src:
                logger.info("%s: image_embeddings of the inputs file is not read (--image_encoder_state_dict encodes "
                            "the first frame)", config.video_name)
            image_embeddings = image_embeddings_entry(pipe, config, idx, synthetic_inputs)
        else:
            image_embeddings = src["image_embeddings"]
        if text_encoder is not None:
            if inputs and "prompt_embeds" in src:
                logger.info("%s: prompt_embeds of the inputs file is not read (--text_encoder_state_dict encodes "
                            "inverse_config.prompt)", config.video_name)
            prompt_embeds = pipe.encode_prompt([inv.get("prompt", "")])           # [1, 77, 1024]
        else:
            prompt_embeds = src["prompt_embeds"]
        dt = unet.dtype
        prompt_embeds, image_embeddings = prompt_embeds.to(device, dt), image_embeddings.to(device, dt)
        image_latents = image_latents.to(device, dt)
        fps = torch.full((1,), int(inv.get("target_fps", 8)), dtype=torch.int64, device=device)
        negative = None
        if do_recon and float(recon.get("cfg", RECON_CFG)) > 1.0:    # checked before the inversion is spent
            if text_encoder is not None:
                negative = pipe.encode_prompt([inv.get("negative_prompt", "")])
            elif "negative_prompt_embeds" in src:
                negative = src["negative_prompt_embeds"].to(device, dt)
            else:
                raise KeyError(f"{config.video_name}: recon_config.cfg > 1 (classifier-free guidance) needs "
                               "negative_prompt_embeds in the --inputs file, or --text_encoder_state_dict with "
                               "--tokenizer_dir to encode inverse_config.negative_prompt")
        if not skip:
            pipe.invert(latents, prompt_embeds, image_embeddings, image_latents, fps,
                        num_inference_steps=int(inv.n_steps), guidance_scale=float(inv.cfg), output_dir=out_dir,
                        max_steps=max_steps, keep=False)
            done += 1
        if do_recon:
            reconstruct(pipe, recon, prompt_embeds, negative, image_embeddings, image_latents, fps, device,
                        vae_state_dict, synthetic_inputs, max_steps)
    return done


def reconstruct(pipe, recon, prompt_embeds, negative_prompt_embeds, image_embeddings, image_latents, fps, device,
                vae_state_dict: str = None, synthetic_inputs: bool = False, max_steps: int = None) -> torch.Tensor:
    """The reconstruction check of one entry (the reference's inverse.py:192-227): plain sampling (pipe.sample) from
    the noisiest stored latents of `recon.ddim_latents_path` with `recon.n_steps` and guidance `recon.cfg`; writes
    `<recon.output_dir>/recon_latents.pt` and, with a VAE file, the decoded frames to `recon_frames/` (`.synthetic`
    names under --synthetic, as composite.py does).  Returns the final latents."""
    from .utils import load_ddim_latents_at_T

    x_T = load_ddim_latents_at_T(recon.ddim_latents_path).float()              # utils.py:39-45, fp16 on disk
    latents = pipe.sample(prompt_embeds, negative_prompt_embeds, image_embeddings, image_latents, fps,
                          num_inference_steps=int(recon.get("n_steps", RECON_STEPS)),
                          guidance_scale=float(recon.get("cfg", RECON_CFG)), latents=x_T, max_steps=max_steps)
    out_dir = recon.get("output_dir") or os.path.join(os.path.dirname(os.path.normpath(recon.ddim_latents_path)),
                                                      "recon")
    os.makedirs(out_dir, exist_ok=True)
    out = os.path.join(out_dir, "recon_latents.synthetic.pt" if synthetic_inputs else "recon_latents.pt")
    torch.save(latents.detach().cpu(), out)
    logger.info("saved %s", out)
    if vae_state_dict:
        from .vae import load_vae_decoder, save_frames

        if pipe.vae is None:
            pipe.vae = load_vae_decoder(vae_state_dict, device)                 # the same file as the encoder's
        frames_dir = os.path.join(out_dir, "recon_frames.synthetic" if synthetic_inputs else "recon_frames")
        save_frames(pipe.decode_latents(latents)[0], frames_dir)
        logger.info("saved %s", frames_dir)
    return latents


def build_parser() -> argparse.ArgumentParser:
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--template_config", type=str, default="./configs/group_inversion/template.yaml")
    ap.add_argument("--configs_json", type=str, default="./configs/group_inversion/group_config.json")
    ap.add_argument("--unet_state_dict", type=str, default=None)
    ap.add_argument("--inputs", type=str, default=None)
    ap.add_argument("--device", type=str, default=None)
    ap.add_argument("--max_steps", type=int, default=None)
    ap.add_argument("--synthetic", action="store_true",
                    help="substitute seeded synthetic tensors for the inputs and random-init weights")
    ap.add_argument("--vae_state_dict", type=str, default=None,
                    help="AutoencoderKL state dict (.safetensors or torch file): encode <video_dir>/<video_name>/ "
                         "frames to the video and first-frame latents instead of reading them from --inputs")
    ap.add_argument("--image_encoder_state_dict", type=str, default=None,
                    help="CLIPVisionModelWithProjection state dict (.safetensors or torch file): encode the first "
                         "frame of <video_dir>/<video_name>/ to image_embeddings instead of reading it from --inputs")
    ap.add_argument("--text_encoder_state_dict", type=str, default=None,
                    help="CLIPTextModel state dict (.safetensors or torch file): encode inverse_config.prompt to "
                         "prompt_embeds instead of reading it from --inputs (needs --tokenizer_dir)")
    ap.add_argument("--tokenizer_dir", type=str, default=None,
                    help="the checkpoint's tokenizer/ folder (vocab.json, merges.txt, tokenizer_config.json / "
                         "special_tokens_map.json) for --text_encoder_state_dict")
    return ap


if __name__ == "__main__":
    args = build_parser().parse_args()
    logging.basicConfig(level=logging.INFO)
    assert os.path.exists(args.template_config) and os.path.exists(args.configs_json)   # inverse.py:134
    main(args.template_config, args.configs_json, args.unet_state_dict, args.inputs, args.device, args.max_steps,
         args.synthetic, args.vae_state_dict, args.image_encoder_state_dict, args.text_encoder_state_dict,
         args.tokenizer_dir)
