"""ORACLE — test infrastructure only (never imported by the product path).

fp32 CPU restatement of the plain I2VGenXL sampling loop, the reference of ``I2VGenXLPipeline.sample``:
  * ``sample_loop`` — diffusers 0.27.2 ``I2VGenXLPipeline.__call__`` steps 3-7, which the reference's own
    ``__call__`` (pipelines/pipeline_i2vgen_xl.py:980-1216) derives from.
RECALLED, not read: that method cannot be read in this tree, so this restates the published diffusers 0.27.2
source, as oracle/scheduler.py and oracle/unet.py do.  It runs the oracle UNet's stock forward (the one
``invert_loop`` calls) and the oracle ``DDIMScheduler``.  Kept beside oracle/pipeline.py, whose loops are restated
from the reference tree line by line.
"""
from __future__ import annotations

from typing import Optional

import torch

from .scheduler import DDIMScheduler


@torch.no_grad()
def sample_loop(unet, inputs: dict, n_steps: int, guidance_scale: float, latents: torch.Tensor,
                max_steps: Optional[int] = None, record: Optional[list] = None) -> torch.Tensor:
    """`inputs` holds batch-1 prompt_embeds, negative_prompt_embeds (read only under guidance), image_embeddings
    [1,1,C], image_latents [1,4,T,h,w] and fps [1]; `latents` [1,4,T,h,w] is the start.  Returns the final latents;
    with `record` also the latents after every step."""
    do_cfg = guidance_scale > 1                                                         # do_classifier_free_guidance
    prompt_embeds, image_embeddings = inputs["prompt_embeds"], inputs["image_embeddings"]
    image_latents, fps = inputs["image_latents"], inputs["fps"]
    if do_cfg:
        prompt_embeds = torch.cat([inputs["negative_prompt_embeds"], prompt_embeds])    # 3. encode_prompt
        image_embeddings = torch.cat([torch.zeros_like(image_embeddings), image_embeddings])  # 3.2 _encode_image
        image_latents = torch.cat([image_latents] * 2)                                  # 3.3 prepare_image_latents
        fps = torch.cat([fps] * 2)                                                      # 3.4 fps_tensor
    sched = DDIMScheduler()
    sched.set_timesteps(n_steps)                                                        # 4. prepare timesteps
    latents = latents.clone() * sched.init_noise_sigma                                  # 5. prepare_latents
    for i, t in enumerate(sched.timesteps):                                             # 7. denoising loop
        if max_steps is not None and i >= max_steps:
            break
        t = int(t)
        latent_model_input = torch.cat([latents] * 2) if do_cfg else latents
        latent_model_input = sched.scale_model_input(latent_model_input, t)
        noise_pred = unet(latent_model_input, t, fps, image_latents, image_embeddings, prompt_embeds,
                          return_dict=False)[0]
        if do_cfg:
            noise_pred_uncond, noise_pred_text = noise_pred.chunk(2)
            noise_pred = noise_pred_uncond + guidance_scale * (noise_pred_text - noise_pred_uncond)
        b, c, f, hh, ww = latents.shape                                                 # reshape for the scheduler
        lat = latents.permute(0, 2, 1, 3, 4).reshape(b * f, c, hh, ww)
        noise = noise_pred.permute(0, 2, 1, 3, 4).reshape(b * f, c, hh, ww)
        lat = sched.step(noise, t, lat)
        latents = lat[None, :].reshape(b, f, c, hh, ww).permute(0, 2, 1, 3, 4)
        if record is not None:
            record.append(latents.clone())
    return latents
