"""`composite.py` of the reference (i2vgen-xl/composite.py) over the B200 path.

    python -m mvoc_b200.composite --template_config configs/group_composite/template.yaml \\
                                  --configs_json configs/group_composite/group_config.json

Same flags, same template-YAML + group-JSON contract (composite.py:227-255, :87-106).  Per active entry it
resolves the paths exactly like composite.py:97-106, builds the injection schedules with `init_pnp`
(:38-69 / :157), loads the inverted source latents (`ddim_latents_{t}.pt`, utils.py:31-36) and the object
masks (utils.mask_preprocess) and runs the 50-step composition loop
(pipelines/pipeline_i2vgen_xl.py:1636-1734) on the GPU.  The final latents are written to
`<output_dir>/composite_latents.pt`.

Out of scope here (SURVEY §2 #9, #10): CLIP / VAE encode.  The tensors those stages produce are read from
`--conditioning file.pt` (a dict with prompt_embeds [n+3,77,1024], image_embeddings [n+3,T,1024],
image_latents_first / image_latents [n+3,4,T,h,w]); the path may contain `{video_name}` / `{edited_video_name}`
so that every config entry gets its own file.  Missing inverted latents, masks or conditioning are ERRORS, like
the reference's asserts (utils.py:34, composite.py:246).  Only with `--synthetic` are seeded synthetic tensors
of the right shape substituted (mvoc_b200.synthetic) — the offline end-to-end exercise of the config → hooks →
loop path; the output is then written as `composite_latents.synthetic.pt`.  UNet weights come from
`--unet_state_dict` (a diffusers I2VGenXLUNet state dict) or, with `--synthetic`, are random-initialised.

With `--vae_state_dict` (a diffusers AutoencoderKL state dict, .safetensors or a torch file) the final latents are
also decoded (decode_latents, pipelines/pipeline_i2vgen_xl.py:771-791) and written as one PNG per frame to
`<output_dir>/composite_frames/` (`composite_frames.synthetic/` under `--synthetic`).  `--synthetic` never invents
decoder weights: without the flag nothing is decoded.

With `--image_encoder_state_dict FILE` (a transformers CLIPVisionModelWithProjection state dict) `image_embeddings`
[n+3,T,1024] is computed here in the branch order [bg, objs..., zeros, main] (pipelines/pipeline_i2vgen_xl.py:766-767)
from `edited_contorl_frame_path_background`, `edited_contorl_frame_path[j]` and `edited_contorl_frame_path_main` (the
first frame when a path is a directory), each centre-cropped to (width, width), resized to 224 x 224 and
CLIP-normalised.  Every other conditioning key still comes from `--conditioning`.  A missing control frame is an
error; only `--synthetic` substitutes a seeded synthetic frame for it.

With `--text_encoder_state_dict FILE` (a transformers CLIPTextModel state dict) and `--tokenizer_dir DIR` (the
checkpoint's tokenizer/ folder) `prompt_embeds` [n+3,77,1024] is computed here from the entry's `prompt`,
`negative_prompt` and `ddim_inv_prompt` in the branch order [inv x (n+1), negative, prompt] (SURVEY Appendix B #9),
each distinct string encoded once.  The two flags go together; `--synthetic` never invents text weights or a
vocabulary.  `image_latents_first` / `image_latents` still come from `--conditioning`.
"""
from __future__ import annotations

import argparse
import logging
import os
from typing import List

import torch

from . import config as cfgmod
from . import synthetic

logger = logging.getLogger(__name__)


def resolve_paths(config):
    """composite.py:97-106 — the same os.path.join calls on the merged entry."""
    j = os.path.join
    config.video_path = j(config.video_dir, config.video_name + ".mp4")
    config.video_frames_path = j(config.video_dir, config.video_name)
    config.edited_first_frame_path = j(config.data_dir, config.edited_first_frame_path)
    config.obj_mask_path = [j(config.data_dir, p) for p in _as_list(config.obj_mask_path)]
    config.obj_ddim_latents_path = [j(config.data_dir, p) for p in _as_list(config.obj_ddim_latents_path)]
    config.bg_ddim_latents_path = j(config.data_dir, config.bg_ddim_latents_path)
    config.edited_contorl_frame_path_main = j(config.data_dir, config.edited_contorl_frame_path_main)
    config.edited_contorl_frame_path_background = j(config.data_dir, config.edited_contorl_frame_path_background)
    config.edited_contorl_frame_path = [j(config.data_dir, p) for p in _as_list(config.edited_contorl_frame_path)]
    return config


def _as_list(x) -> List:
    if x is None or x == "":
        return []
    return list(x) if isinstance(x, (list, tuple)) else [x]


def latent_geometry(config):
    """(T, h, w) of the latents: image_size is (width, height) in pixels, VAE factor 8."""
    w_px, h_px = config.image_size
    return int(config.n_frames), int(h_px) // 8, int(w_px) // 8


def conditioning_path(template: str, config) -> str:
    """`--conditioning` may name one file per entry through {video_name} / {edited_video_name}."""
    return template.format(video_name=config.video_name,
                           edited_video_name=config.get("edited_video_name", config.video_name))


def run_entry(pipe, config, device, conditioning=None, allow_synthetic: bool = False):
    """One config entry -> final composite latents [1,4,T,h,w] (fp32, on `device`).  Missing inputs raise
    FileNotFoundError unless allow_synthetic."""
    from .pipeline import Conditioning, LatentBank, init_pnp
    from .scheduler import DDIMSchedule
    from .utils import mask_preprocess, seed_everything

    seed_everything(int(config.seed))
    T, h, w = latent_geometry(config)
    n_obj = len(config.obj_mask_path)
    sched = DDIMSchedule(int(config.n_steps))
    init_pnp(pipe, sched, config)                                              # composite.py:157
    wl = synthetic.Workload(config.video_name, "full", T, h, w, n_obj, n_steps=int(config.n_steps))
    synth = synthetic.make_inputs(wl, sched.timesteps, sched.alphas_cumprod)
    dt = pipe.unet.dtype

    def bank(path, fallback):
        if path and os.path.isdir(path):
            return LatentBank.from_dir(path, sched.timesteps, device)
        if not allow_synthetic:
            raise FileNotFoundError(f"inverted latents directory {path!r} not found (run inverse.py first, or pass "
                                    "--synthetic for an offline exercise with seeded synthetic latents)")
        logger.warning("inverted latents %s not found: using synthetic source latents (--synthetic)", path)
        return LatentBank(fallback, device)

    bg = bank(config.bg_ddim_latents_path, synth["source_latents"][0])
    objs = [bank(p, synth["source_latents"][j + 1]) for j, p in enumerate(config.obj_ddim_latents_path)]
    masks = []
    for j, p in enumerate(config.obj_mask_path):
        if os.path.exists(p):
            mf, mb = mask_preprocess(p, device, torch.float32, 1, 4, T, downscale=8)   # pipeline :1594
            if tuple(mf.shape[-2:]) != (h, w):
                raise ValueError(f"mask {p} is {tuple(mf.shape[-2:])} after /8, latents are {(h, w)}")
        else:
            if not allow_synthetic:
                raise FileNotFoundError(f"object mask {p!r} not found (pass --synthetic for a synthetic mask)")
            logger.warning("mask %s not found: using a synthetic mask (--synthetic)", p)
            mf, mb = (t.to(device) for t in synth["masks"][j])
        masks.append((mf, mb))
    if conditioning is None and not allow_synthetic:
        raise FileNotFoundError("no --conditioning file for this entry (CLIP / VAE outputs are inputs of this "
                                "script); pass --synthetic for seeded synthetic conditioning")
    src = conditioning if conditioning is not None else synth
    cond = Conditioning(src["prompt_embeds"].to(device, dt), src["image_embeddings"].to(device, dt),
                        src["image_latents_first"].to(device, dt), src["image_latents"].to(device, dt),
                        torch.full((n_obj + 3,), int(config.target_fps), dtype=torch.int64, device=device))
    latents = synth["init_latents"].to(device).clone()                          # prepare_latents, :1570-1580
    return pipe.sample_with_pnp_pipeline_with_edit_prompt_extraction_with_attn_injection(
        cond, latents, bg, objs, masks, num_inference_steps=int(config.n_steps), guidance_scale=float(config.cfg),
        ddim_init_latents_t_idx=int(config.ddim_init_latents_t_idx), fusion_steps=tuple(config.fusion_step),
        random_noise_ratio=float(config.random_noise_ratio),
        obj_random_noise_fusion=bool(config.obj_random_noise_fusion),
        obj_ddim_latents_idx_offset=list(config.obj_ddim_latents_idx_offset)[:n_obj] or None)


def branch_image_embeddings(pipe, config, allow_synthetic: bool = False) -> torch.Tensor:
    """image_embeddings [n+3, T, 1024] of one entry in the branch order [bg, objs..., zeros, main] (SURVEY Appendix B
    #9; pipelines/pipeline_i2vgen_xl.py:766-767).  The reference encodes every frame of every branch, T x (n+2) CLIP
    calls, but the UNet reads only image_embeddings[:, 0:1] (mvoc_b200/unet3d.py, I2VGenXLUNet.context), so ONE
    embedding per branch from its control frame, repeated over T, gives the UNet the same input with n+2 calls."""
    from PIL import Image

    from .clip import clip_image_input, first_frame

    T = int(config.n_frames)
    w_px, h_px = (int(v) for v in config.image_size)
    paths = ([config.edited_contorl_frame_path_background] + list(config.edited_contorl_frame_path)
             + [config.edited_contorl_frame_path_main])
    images = []
    for i, p in enumerate(paths):
        if os.path.exists(p):
            images.append(first_frame(p))
            continue
        if not allow_synthetic:
            raise FileNotFoundError(f"control frame {p!r} not found (pass --synthetic for a synthetic frame)")
        logger.warning("control frame %s not found: using a seeded synthetic frame (--synthetic)", p)
        g = torch.Generator().manual_seed(7000 + i)
        images.append(Image.fromarray(torch.randint(0, 256, (h_px, w_px, 3), generator=g, dtype=torch.uint8).numpy()))
    emb = pipe.encode_image(clip_image_input(images, w_px))                      # [n+2, 1, 1024]
    emb = torch.cat([emb[:-1], torch.zeros_like(emb[:1]), emb[-1:]])           # [bg, objs, zeros, main]
    return emb.expand(-1, T, -1).contiguous()


def branch_prompt_embeds(pipe, config) -> torch.Tensor:
    """prompt_embeds [n+3, 77, 1024] of one entry: encode_prompt of [ddim_inv_prompt x (n+1), negative_prompt,
    prompt], each distinct string encoded once."""
    from .clip_text import composition_prompt_embeds

    return composition_prompt_embeds(pipe.encode_prompt, len(config.obj_mask_path), config.get("prompt", ""),
                                     config.get("negative_prompt", ""), config.get("ddim_inv_prompt", ""))


def main(template_config: str, configs_json: str, unet_state_dict: str = None, conditioning: str = None,
         device: str = None, max_entries: int = None, synthetic_inputs: bool = False, vae_state_dict: str = None,
         image_encoder_state_dict: str = None, text_encoder_state_dict: str = None, tokenizer_dir: str = None):
    from .clip_text import check_text_flags, load_text_tower
    from .pipeline import I2VGenXLPipeline
    from .unet3d import I2VGenXLUNet, UNetConfig, prepare
    from .vae import load_vae_decoder, save_frames

    check_text_flags(text_encoder_state_dict, tokenizer_dir)

    template = cfgmod.load_template(template_config)
    device = torch.device(device or template.get("device", "cuda:0"))
    if device.type == "cuda":
        torch.cuda.set_device(device)      # the C-ABI launches on the current device (mvoc_b200.ops._need_cuda)
    torch.set_grad_enabled(False)                                               # composite.py:253
    unet = I2VGenXLUNet(UNetConfig.full()).eval().requires_grad_(False)
    if unet_state_dict:
        unet.load_state_dict(torch.load(unet_state_dict, map_location="cpu"), strict=True)
    elif not synthetic_inputs:
        raise FileNotFoundError("--unet_state_dict is required (pass --synthetic to run on random-init weights)")
    unet = prepare(unet.to(device=device, dtype=torch.bfloat16))
    vae = load_vae_decoder(vae_state_dict, device) if vae_state_dict else None
    image_encoder = None
    if image_encoder_state_dict:
        from .clip import load_clip_image_encoder

        image_encoder = load_clip_image_encoder(image_encoder_state_dict, device)
    text_encoder, tokenizer = load_text_tower(text_encoder_state_dict, tokenizer_dir, device)
    pipe = I2VGenXLPipeline(unet, device, use_cuda_graphs=True, vae=vae, image_encoder=image_encoder,
                            text_encoder=text_encoder, tokenizer=tokenizer)
    done = 0
    for config in cfgmod.iter_configs(template_config, configs_json):
        config = resolve_paths(config)
        logger.info("Processing %s / %s", config.video_name, config.edited_video_name)
        cond = None
        if conditioning:
            cpath = conditioning_path(conditioning, config)
            if not os.path.exists(cpath):
                raise FileNotFoundError(f"conditioning file {cpath!r} not found")
            cond = torch.load(cpath, map_location="cpu")
        if image_encoder is not None or text_encoder is not None:
            for key, flag, enc in (("image_embeddings", "--image_encoder_state_dict", image_encoder),
                                   ("prompt_embeds", "--text_encoder_state_dict", text_encoder)):
                if enc is not None and cond is not None and key in cond:
                    logger.info("%s: %s of the conditioning file is not read (%s computes it)", config.video_name,
                                key, flag)
            if cond is None and synthetic_inputs:   # the other keys stay synthetic
                T, h, w = latent_geometry(config)
                cond = synthetic.make_inputs(synthetic.Workload(config.video_name, "full", T, h, w,
                                                                len(config.obj_mask_path)), [], None)
            if cond is not None and image_encoder is not None:
                cond = dict(cond, image_embeddings=branch_image_embeddings(pipe, config, synthetic_inputs))
            if cond is not None and text_encoder is not None:
                cond = dict(cond, prompt_embeds=branch_prompt_embeds(pipe, config))
        latents = run_entry(pipe, config, device, cond, allow_synthetic=synthetic_inputs)
        os.makedirs(config.output_dir, exist_ok=True)
        out = os.path.join(config.output_dir,
                           "composite_latents.synthetic.pt" if synthetic_inputs else "composite_latents.pt")
        torch.save(latents.detach().cpu(), out)
        logger.info("saved %s", out)
        if vae is not None:
            frames_dir = os.path.join(config.output_dir,
                                      "composite_frames.synthetic" if synthetic_inputs else "composite_frames")
            save_frames(pipe.decode_latents(latents)[0], frames_dir)
            logger.info("saved %s", frames_dir)
        done += 1
        if max_entries is not None and done >= max_entries:
            break
    return done


def build_parser() -> argparse.ArgumentParser:
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--template_config", type=str, default="./configs/group_composite/template.yaml")
    ap.add_argument("--configs_json", type=str, default="./configs/group_composite/group_config.json")
    ap.add_argument("--unet_state_dict", type=str, default=None)
    ap.add_argument("--conditioning", type=str, default=None)
    ap.add_argument("--vae_state_dict", type=str, default=None,
                    help="diffusers AutoencoderKL state dict: also decode the latents and write PNG frames")
    ap.add_argument("--image_encoder_state_dict", type=str, default=None,
                    help="CLIPVisionModelWithProjection state dict: encode the control frames to image_embeddings "
                         "instead of reading them from --conditioning")
    ap.add_argument("--text_encoder_state_dict", type=str, default=None,
                    help="CLIPTextModel state dict: encode the entry's prompt, negative_prompt and ddim_inv_prompt to "
                         "prompt_embeds instead of reading them from --conditioning (needs --tokenizer_dir)")
    ap.add_argument("--tokenizer_dir", type=str, default=None,
                    help="the checkpoint's tokenizer/ folder (vocab.json, merges.txt, tokenizer_config.json / "
                         "special_tokens_map.json) for --text_encoder_state_dict")
    ap.add_argument("--device", type=str, default=None)
    ap.add_argument("--max_entries", type=int, default=None)
    ap.add_argument("--synthetic", action="store_true",
                    help="substitute seeded synthetic tensors for missing latents / masks / conditioning / weights")
    return ap


if __name__ == "__main__":
    args = build_parser().parse_args()
    logging.basicConfig(level=logging.INFO)
    assert os.path.exists(args.template_config) and os.path.exists(args.configs_json)   # composite.py:246
    main(args.template_config, args.configs_json, args.unet_state_dict, args.conditioning, args.device,
         args.max_entries, args.synthetic, args.vae_state_dict, args.image_encoder_state_dict,
         args.text_encoder_state_dict, args.tokenizer_dir)
