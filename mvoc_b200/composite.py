"""`composite.py` of the reference (i2vgen-xl/composite.py) over the B200 path.

    python -m mvoc_b200.composite --template_config configs/group_composite/template.yaml \\
                                  --configs_json configs/group_composite/group_config.json

Same flags, same template-YAML + group-JSON contract (composite.py:227-255, :87-106).  Per active entry it
resolves the paths exactly like composite.py:97-106, builds the injection schedules with `init_pnp`
(:38-69 / :157), loads the inverted source latents (`ddim_latents_{t}.pt`, utils.py:31-36) and the object
masks (utils.mask_preprocess) and runs the 50-step composition loop
(pipelines/pipeline_i2vgen_xl.py:1636-1734) on the GPU.  The final latents are written to
`<output_dir>/composite_latents.pt`.

The conditioning tensors not computed by the flags below are read from `--conditioning file.pt` (a dict with
prompt_embeds [n+3,77,1024], image_embeddings [n+3,T,1024], image_latents_first / image_latents [n+3,4,T,h,w]); the
path may contain `{video_name}` / `{edited_video_name}` so that every config entry gets its own file.  Missing inverted latents, masks or conditioning are ERRORS, like
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
CLIP-normalised.  A missing control frame is an error; only `--synthetic` substitutes a seeded synthetic frame for
it.

With `--text_encoder_state_dict FILE` (a transformers CLIPTextModel state dict) and `--tokenizer_dir DIR` (the
checkpoint's tokenizer/ folder) `prompt_embeds` [n+3,77,1024] is computed here from the entry's `prompt`,
`negative_prompt` and `ddim_inv_prompt` in the branch order [inv x (n+1), negative, prompt] (SURVEY Appendix B #9),
each distinct string encoded once.  The two flags go together; `--synthetic` never invents text weights or a
vocabulary.

With `--encode_image_latents` (needs `--vae_state_dict`, whose encoder half is then loaded too) `image_latents_first`
= `image_latents` [n+3,4,T,h,w] are computed here in the branch order [bg, objs..., main, main] from the first frame of
the same control-frame paths: each centre-cropped to image_size, encoded together by prepare_image_latents under one
`torch.Generator().manual_seed(seed)`.  The flag is opt-in: `--vae_state_dict` alone only decodes.  A key computed
here replaces the conditioning file's (logged).  With `--encode_image_latents`, `--image_encoder_state_dict` and the
text flags together every conditioning key is computed and `--conditioning` is not needed (fps comes from the
config's target_fps); otherwise a missing key is an error that names it.

Frame-parallel over the GPUs of one node, every active entry in turn over all ranks:

    python -m torch.distributed.run --nproc-per-node N -m mvoc_b200.composite --template_config ... --configs_json ...

Every rank owns n_frames / N frames of all n+3 branches (mvoc_b200.parallel.FrameParallel, the NVLink peer exchange
around the temporal operators); n_frames must divide by N, which is checked on every rank before any collective.
Every rank reads the same inputs and computes the same conditioning; under `--synthetic` rank 0's random-init UNet
weights are broadcast to the others.  The prediction is all-gathered before each DDIM update, so every rank ends with
the full latents; rank 0 writes composite_latents.pt, and with `--vae_state_dict` every rank decodes and writes its own
frames under their global numbers.  The peer-exchange arena is sized for the largest entry
(parallel.exchange_arena_mb; MVOC_EXCHANGE_ARENA_MB overrides it).  Without torchrun (or with N = 1) nothing of this
runs.
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


def control_frames(config, allow_synthetic: bool = False) -> list:
    """The first frame (PIL, RGB) of each branch's control frames in the order [bg, objs..., main]:
    `edited_contorl_frame_path_background`, `edited_contorl_frame_path[j]` and `edited_contorl_frame_path_main`, each a
    file or a directory of frames.  A missing one raises FileNotFoundError unless allow_synthetic, which substitutes a
    seeded uint8 noise frame of `image_size`."""
    from PIL import Image

    from .clip import first_frame

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
    return images


def branch_image_embeddings(pipe, config, allow_synthetic: bool = False) -> torch.Tensor:
    """image_embeddings [n+3, T, 1024] of one entry in the branch order [bg, objs..., zeros, main] (SURVEY Appendix B
    #9; pipelines/pipeline_i2vgen_xl.py:766-767).  The reference encodes every frame of every branch, T x (n+2) CLIP
    calls, but the UNet reads only image_embeddings[:, 0:1] (mvoc_b200/unet3d.py, I2VGenXLUNet.context), so ONE
    embedding per branch from its control frame, repeated over T, gives the UNet the same input with n+2 calls."""
    from .clip import clip_image_input

    T = int(config.n_frames)
    w_px = int(config.image_size[0])
    images = control_frames(config, allow_synthetic)
    emb = pipe.encode_image(clip_image_input(images, w_px))                      # [n+2, 1, 1024]
    emb = torch.cat([emb[:-1], torch.zeros_like(emb[:1]), emb[-1:]])           # [bg, objs, zeros, main]
    return emb.expand(-1, T, -1).contiguous()


def branch_image_latents(pipe, config, allow_synthetic: bool = False) -> torch.Tensor:
    """image_latents [n+3, 4, T, h, w] fp32 of one entry in the branch order [bg, objs..., main, main] (SURVEY
    Appendix B #9; the CFG doubling duplicates main; the composition uses the same tensor as image_latents_first).
    Each branch's first control frame is centre-cropped to image_size (center_crop_wide) and the n+2 distinct frames
    go through prepare_image_latents together, under one torch.Generator().manual_seed(seed): one posterior noise
    draw over the n+2 images in branch order."""
    from .vae import center_crop_wide, pil_to_model_input

    T = int(config.n_frames)
    size = tuple(int(v) for v in config.image_size)
    images = [center_crop_wide(im, size) for im in control_frames(config, allow_synthetic)]
    x = pil_to_model_input(images).to(pipe.device)
    lat = pipe.prepare_image_latents(x, T, torch.Generator().manual_seed(int(config.seed)))   # [n+2, 4, T, h, w]
    return torch.cat([lat, lat[-1:]])


def branch_prompt_embeds(pipe, config) -> torch.Tensor:
    """prompt_embeds [n+3, 77, 1024] of one entry: encode_prompt of [ddim_inv_prompt x (n+1), negative_prompt,
    prompt], each distinct string encoded once."""
    from .clip_text import composition_prompt_embeds

    return composition_prompt_embeds(pipe.encode_prompt, len(config.obj_mask_path), config.get("prompt", ""),
                                     config.get("negative_prompt", ""), config.get("ddim_inv_prompt", ""))


CONDITIONING_KEYS = ("prompt_embeds", "image_embeddings", "image_latents_first", "image_latents")


def check_frame_split(configs, world: int) -> None:
    """Frame-parallel composition gives every rank n_frames / world frames of an entry: an entry whose n_frames the
    rank count does not divide is an error, raised on every rank (they all read the same configs) before any
    collective, so that no rank waits for another."""
    for config in configs:
        T = int(config.n_frames)
        if T % world != 0:
            raise ValueError(f"{config.video_name}: n_frames={T} is not divisible by WORLD_SIZE={world} (every rank "
                             "composes n_frames / WORLD_SIZE frames)")


def main(template_config: str, configs_json: str, unet_state_dict: str = None, conditioning: str = None,
         device: str = None, max_entries: int = None, synthetic_inputs: bool = False, vae_state_dict: str = None,
         image_encoder_state_dict: str = None, text_encoder_state_dict: str = None, tokenizer_dir: str = None,
         encode_image_latents: bool = False):
    from .clip_text import check_text_flags
    from .parallel import FrameParallel, exchange_arena_mb

    check_text_flags(text_encoder_state_dict, tokenizer_dir)
    if encode_image_latents and not vae_state_dict:
        raise ValueError("--encode_image_latents needs --vae_state_dict: the VAE encoder is read from that file")

    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    template = cfgmod.load_template(template_config)
    device = torch.device(device or (f"cuda:{local}" if world > 1 else template.get("device", "cuda:0")))
    configs = [resolve_paths(c) for c in cfgmod.iter_configs(template_config, configs_json)]
    if max_entries is not None:
        configs = configs[:max_entries]
    if device.type == "cuda":
        torch.cuda.set_device(device)      # the C-ABI launches on the current device (mvoc_b200.ops._need_cuda)
    arena_mb = None
    if world > 1:
        check_frame_split(configs, world)
        arena_mb = max((exchange_arena_mb(len(c.obj_mask_path) + 3, *latent_geometry(c), world) for c in configs),
                       default=None)
    par = FrameParallel.from_env(device, arena_mb=arena_mb)            # world_size 1 => no process group
    try:
        return _run(configs, par, device, unet_state_dict, conditioning, synthetic_inputs, vae_state_dict,
                    image_encoder_state_dict, text_encoder_state_dict, tokenizer_dir, encode_image_latents)
    finally:
        par.shutdown()                     # no process group or IPC mapping outlives the run


def _run(configs, par, device, unet_state_dict, conditioning, synthetic_inputs, vae_state_dict,
         image_encoder_state_dict, text_encoder_state_dict, tokenizer_dir, encode_image_latents) -> int:
    from .clip_text import load_text_tower
    from .pipeline import I2VGenXLPipeline
    from .unet3d import I2VGenXLUNet, UNetConfig, prepare
    from .vae import load_vae_decoder, save_frames

    torch.set_grad_enabled(False)                                               # composite.py:253
    unet = I2VGenXLUNet(UNetConfig.full()).eval().requires_grad_(False)
    if unet_state_dict:
        unet.load_state_dict(torch.load(unet_state_dict, map_location="cpu"), strict=True)
    elif not synthetic_inputs:
        raise FileNotFoundError("--unet_state_dict is required (pass --synthetic to run on random-init weights)")
    unet = unet.to(device=device, dtype=torch.bfloat16)
    if not unet_state_dict:
        par.broadcast_module(unet)         # random-init weights: rank 0's on every rank
    unet = prepare(unet)
    vae = load_vae_decoder(vae_state_dict, device) if vae_state_dict else None
    vae_encoder = None
    if encode_image_latents:
        from .vae import load_vae_encoder

        vae_encoder = load_vae_encoder(vae_state_dict, device)
    image_encoder = None
    if image_encoder_state_dict:
        from .clip import load_clip_image_encoder

        image_encoder = load_clip_image_encoder(image_encoder_state_dict, device)
    text_encoder, tokenizer = load_text_tower(text_encoder_state_dict, tokenizer_dir, device)
    pipe = I2VGenXLPipeline(unet, device, parallel=par, use_cuda_graphs=device.type == "cuda", vae=vae,
                            vae_encoder=vae_encoder, image_encoder=image_encoder, text_encoder=text_encoder,
                            tokenizer=tokenizer)
    computes = {}                          # conditioning key -> the flag that computes it
    if image_encoder is not None:
        computes["image_embeddings"] = "--image_encoder_state_dict"
    if text_encoder is not None:
        computes["prompt_embeds"] = "--text_encoder_state_dict"
    if vae_encoder is not None:
        computes.update(image_latents_first="--encode_image_latents", image_latents="--encode_image_latents")
    done = 0
    for config in configs:
        logger.info("Processing %s / %s", config.video_name, config.edited_video_name)
        cond = None
        if conditioning:
            cpath = conditioning_path(conditioning, config)
            if not os.path.exists(cpath):
                raise FileNotFoundError(f"conditioning file {cpath!r} not found")
            cond = torch.load(cpath, map_location="cpu")
        if computes:
            for key, flag in computes.items():
                if cond is not None and key in cond:
                    logger.info("%s: %s of the conditioning file is not read (%s computes it)", config.video_name,
                                key, flag)
            if cond is None:
                if synthetic_inputs:       # the keys not computed stay synthetic
                    T, h, w = latent_geometry(config)
                    cond = synthetic.make_inputs(synthetic.Workload(config.video_name, "full", T, h, w,
                                                                    len(config.obj_mask_path)), [], None)
                elif len(computes) == len(CONDITIONING_KEYS):
                    cond = {}              # every key is computed below; fps comes from the config
                else:
                    missing = [k for k in CONDITIONING_KEYS if k not in computes]
                    raise FileNotFoundError(f"no --conditioning file for {config.video_name}, and no flag computes "
                                            f"{', '.join(missing)} (image_embeddings: --image_encoder_state_dict; "
                                            "prompt_embeds: --text_encoder_state_dict with --tokenizer_dir; "
                                            "image_latents_first / image_latents: --encode_image_latents)")
            if image_encoder is not None:
                cond = dict(cond, image_embeddings=branch_image_embeddings(pipe, config, synthetic_inputs))
            if text_encoder is not None:
                cond = dict(cond, prompt_embeds=branch_prompt_embeds(pipe, config))
            if vae_encoder is not None:
                il = branch_image_latents(pipe, config, synthetic_inputs)
                cond = dict(cond, image_latents_first=il, image_latents=il)
        latents = run_entry(pipe, config, device, cond, allow_synthetic=synthetic_inputs)
        if par.rank == 0:
            os.makedirs(config.output_dir, exist_ok=True)
            out = os.path.join(config.output_dir,
                               "composite_latents.synthetic.pt" if synthetic_inputs else "composite_latents.pt")
            torch.save(latents.detach().cpu(), out)
            logger.info("saved %s", out)
        if vae is not None:
            # every rank decodes and writes its own frames, under their global numbers
            frames_dir = os.path.join(config.output_dir,
                                      "composite_frames.synthetic" if synthetic_inputs else "composite_frames")
            f0, f1 = par.frame_range(latents.shape[2])
            save_frames(pipe.decode_latents(latents[:, :, f0:f1])[0], frames_dir, first_index=f0)
            logger.info("saved %s", frames_dir)
        done += 1
    par.barrier()                          # every rank's frames are on disk when the command returns
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
    ap.add_argument("--encode_image_latents", action="store_true",
                    help="encode each branch's first control frame with the VAE encoder of --vae_state_dict to "
                         "image_latents_first / image_latents instead of reading them from --conditioning")
    ap.add_argument("--device", type=str, default=None)
    ap.add_argument("--max_entries", type=int, default=None)
    ap.add_argument("--synthetic", action="store_true",
                    help="substitute seeded synthetic tensors for missing latents / masks / conditioning / weights")
    return ap


if __name__ == "__main__":
    args = build_parser().parse_args()
    # under torchrun only rank 0 logs progress; the other ranks report errors only
    logging.basicConfig(level=logging.INFO if int(os.environ.get("RANK", "0")) == 0 else logging.ERROR)
    assert os.path.exists(args.template_config) and os.path.exists(args.configs_json)   # composite.py:246
    main(args.template_config, args.configs_json, args.unet_state_dict, args.conditioning, args.device,
         args.max_entries, args.synthetic, args.vae_state_dict, args.image_encoder_state_dict,
         args.text_encoder_state_dict, args.tokenizer_dir, args.encode_image_latents)
