"""Synthetic workloads (SURVEY §8d): there is no network, checkpoint, VAE or CLIP here, so the
bench, the smoke test and the parity tests all run on seeded synthetic tensors of the right shape.

Pure data generation on the CPU (torch RNG); no arithmetic of the hot path lives here.
Shapes follow pipelines/pipeline_i2vgen_xl.py: UNet batch = [bg, obj_1..obj_n, uncond, cond]
(:1675-1677); prompt embeds [n+3, 77, 1024] (:1380-1389); CLIP image embeds [n+3, T, 1024] with the
uncond row zero (:766-767, :1540-1541); first-frame image latents [n+3, 4, T, h, w] whose frames
1..T-1 are the constant position channels i/(T-1) (:876-882).
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import Dict, List, Tuple

import torch


@dataclass
class Workload:
    name: str
    unet: str                  # "full" | "reduced"
    n_frames: int
    latent_h: int
    latent_w: int
    n_obj: int
    n_steps: int = 50
    inversion_steps: int = 500
    cfg: float = 9.0
    target_fps: int = 8
    ddim_init_latents_t_idx: int = 0
    pnp_f_t: float = 0.1
    pnp_spatial_attn_t: float = 1.0
    pnp_temp_attn_t: float = 1.0
    inject_background: bool = False
    random_noise_ratio: float = 0.0
    fusion_step: Tuple[int, int] = (0, 1)
    obj_random_noise_fusion: bool = False
    seed: int = 6
    n_videos: int = 1          # inversion workloads: independent source videos (replicas across GPUs)

    @property
    def n_branches(self) -> int:
        return self.n_obj + 3


WORKLOADS: Dict[str, Workload] = {
    # BASELINE.json configs[0]: reduced UNet, 8 x 32x32, bg + 1 object
    "config1": Workload("config1", "reduced", 8, 32, 32, 1),
    # configs[1] / [3]: full UNet, 16 x 64x64 (512x512 px), bg + 2 objects, boat_surf knobs
    "config2": Workload("config2", "full", 16, 64, 64, 2),
    # configs[2]: group DDIM inversion of 3 source videos (16 x 64x64 latents, 500 steps, cfg 1.0 => batch 1),
    # one video per GPU (replicas, no collective; configs/group_inversion/group_config.json shape)
    "config3": Workload("config3", "full", 16, 64, 64, 0, n_videos=3),
    # configs[4]: 32 x 88x160 (704x1280 px), bg + 3 objects
    "config5": Workload("config5", "full", 32, 88, 160, 3),
    # the benchmarked model and latent size with 2 of the 16 frames: full-architecture GPU parity against the
    # fp32 CPU oracle at a cost the oracle can pay (one step ~10 s on 16 host cores)
    "config2_t2": Workload("config2_t2", "full", 2, 64, 64, 2),
    # small full-architecture case for GPU parity tests
    "full_small": Workload("full_small", "full", 8, 32, 32, 2),
    "reduced2": Workload("reduced2", "reduced", 8, 32, 32, 2),
}


def make_masks(n_obj: int, T: int, h: int, w: int, seed: int = 0):
    """Per object: a moving ellipse with a ~2-latent-pixel linear soft edge, float in [0,1] with 255
    levels and bool = float > 10/255 (cv.threshold at utils.py:131), both shaped [1, 4, T, h, w]
    like utils.mask_preprocess (utils.py:92-154).  Centres of different objects are disjoint; with three objects neighbouring ellipses may
    overlap a little, which exercises the 'later object wins' rule (pnp_utils.py:643-662)."""
    g = torch.Generator().manual_seed(1234 + seed)
    ys = torch.arange(h).view(1, h, 1).float()
    xs = torch.arange(w).view(1, 1, w).float()
    out = []
    for j in range(n_obj):
        cy = h * (0.35 + 0.3 * torch.rand(1, generator=g)) + torch.linspace(0, h * 0.08, T).view(T, 1, 1)
        cx = w * (0.18 + 0.64 * (j + 0.5) / n_obj) + torch.linspace(0, w * 0.06, T).view(T, 1, 1)
        ry = h * (0.10 + 0.06 * torch.rand(1, generator=g))
        rx = w * (0.08 + 0.06 * torch.rand(1, generator=g))
        d = torch.sqrt(((ys - cy) / ry) ** 2 + ((xs - cx) / rx) ** 2)
        edge = 2.0 / float(min(ry, rx))
        mf = ((1.0 + edge - d) / edge).clamp(0, 1)
        mf = (mf * 255).round() / 255
        mb = mf > (10.0 / 255.0)
        out.append((mf[None, None].expand(1, 4, T, h, w).contiguous(),
                    mb[None, None].expand(1, 4, T, h, w).contiguous()))
    return out


def _randn(shape, seed: int) -> torch.Tensor:
    return torch.randn(shape, generator=torch.Generator().manual_seed(seed))


def _image_latents(nb: int, T: int, h: int, w: int, seed: int) -> torch.Tensor:
    """[nb, 4, T, h, w]: frame 0 = N(0,1)*0.18215, frames i>=1 = i/(T-1); composite rows share `main`."""
    rows = []
    for b in range(nb - 1):  # bg, objects, main
        f0 = _randn((4, 1, h, w), seed * 100 + b) * 0.18215
        pos = torch.stack([torch.full((4, h, w), (i + 1) / (T - 1)) for i in range(T - 1)], dim=1)
        rows.append(torch.cat([f0, pos], dim=1))
    rows.append(rows[-1].clone())  # CFG doubling of the main branch (:887-888)
    return torch.stack(rows)


def make_inputs(wl: Workload, timesteps: List[int], alphas_cumprod) -> dict:
    """Everything the composition loop consumes, fp32 on the CPU.

    source latents stand in for the inversion output files ``ddim_latents_{t}.pt``
    (utils.py:31-36): sqrt(a_t) x0 + sqrt(1-a_t) eps with x0, eps ~ N(0,1), seeds 1000 + branch.
    """
    T, h, w, n = wl.n_frames, wl.latent_h, wl.latent_w, wl.n_obj
    nb = wl.n_branches
    shape = (1, 4, T, h, w)
    sources = []
    for br in range(n + 1):
        x0 = _randn(shape, 1000 + br)
        eps = _randn(shape, 2000 + br)
        per_t = {}
        for t in timesteps:
            a = float(alphas_cumprod[t])
            per_t[int(t)] = (a ** 0.5) * x0 + ((1 - a) ** 0.5) * eps
        sources.append(per_t)
    clip = _randn((nb, T, 1024), 8)
    clip[n + 1] = 0.0  # negative image embeddings are zeros (:766)
    return {
        "source_latents": sources,                      # [bg, obj_1..obj_n] -> {t: [1,4,T,h,w]}
        "init_latents": _randn(shape, wl.seed),
        "prompt_embeds": _randn((nb, 77, 1024), 7),
        "image_embeddings": clip,
        "image_latents_first": _image_latents(nb, T, h, w, 9),
        "image_latents": _image_latents(nb, T, h, w, 10),
        "fps": torch.full((nb,), wl.target_fps, dtype=torch.int64),
        "masks": make_masks(n, T, h, w, seed=wl.seed),
    }


def make_inversion_inputs(wl: Workload, video_index: int = 0) -> dict:
    """Inputs of pipe.invert for one synthetic source video (inverse.py:48-76): clean latents x0,
    empty-prompt embeds, one CLIP embedding, first-frame image latents; batch 1 (cfg 1.0 => no CFG).  The negative
    prompt embeds are read only by the guided reconstruction (recon_config)."""
    T, h, w = wl.n_frames, wl.latent_h, wl.latent_w
    return {
        "latents": _randn((1, 4, T, h, w), 3000 + video_index) * 0.18215 * 4.0,
        "prompt_embeds": _randn((1, 77, 1024), 3100 + video_index),
        "image_embeddings": _randn((1, 1, 1024), 3200 + video_index),
        "image_latents": _image_latents(2, T, h, w, 33 + video_index)[:1],
        "fps": torch.full((1,), wl.target_fps, dtype=torch.int64),
        "negative_prompt_embeds": _randn((1, 77, 1024), 3300 + video_index),
    }
