"""Step loops of the MVOC pipeline over the B200 kernels.

Mirrors ``I2VGenXLPipeline`` of i2vgen-xl/pipelines/pipeline_i2vgen_xl.py for the two loops on the
hot path:
  * ``sample_with_pnp_pipeline_with_edit_prompt_extraction_with_attn_injection``  (:1220-1748,
    loop :1636-1734) — 50-step DDIM composition with source-branch feature injection;
  * ``invert``  (:1752-2018, loop :1940-2000) — DDIM inversion writing ``ddim_latents_{t}.pt``.
CLIP / PIL work around the loops (:1356-1541, :1739-1748) is out of scope (SURVEY §2 #9): the loops take
the tensors those stages produce (prompt embeds, CLIP image embeds, first-frame image latents, masks,
inverted latents).  The VAE runs here when the pipeline is given one: ``decode_latents`` (decoder),
``encode_vae_video`` and ``prepare_image_latents`` (encoder); so does the CLIP image tower (``encode_image``).
INTEGRATION.md shows the seam.

Per step the reference launches ~6 elementwise kernels per object for the fusion, a torch.cat, the
CFG combine and ~10 scheduler kernels, reloads the source latents from disk and syncs twice
(`t.item()`, f-string of a device tensor).  Here a step is: one ``mvoc_latent_composite`` launch
(fusion + concat + bf16 cast), the UNet, one ``mvoc_cfg_ddim_step`` launch; timesteps are Python ints,
conditioning that does not depend on t is computed once, and the latent store is resident in HBM.
"""
from __future__ import annotations

import os
from dataclasses import dataclass
from typing import Callable, Dict, List, Optional, Sequence, Tuple

import torch

from . import ops, pnp_utils
from .scheduler import DDIMSchedule


# --------------------------------------------------------------------------
# latent store: ddim_latents_{t}.pt wire format (utils.py:31-45, pipeline_i2vgen_xl.py:1988-1993)
# --------------------------------------------------------------------------
def ddim_latents_filename(t: int) -> str:
    return f"ddim_latents_{int(t)}.pt"


def save_ddim_latents_at_t(latents: torch.Tensor, t: int, path: str, dtype=torch.float16) -> None:
    """One `ddim_latents_{t}.pt` in the reference's wire dtype: it saves its fp16 pipeline latents
    (pipeline_i2vgen_xl.py:1990-1993) and reads them back with `.to(device)`, which keeps the dtype — an fp32
    file would meet fp16 weights there.  `dtype=None` keeps the tensor's own dtype (our packed store stays fp32)."""
    os.makedirs(path, exist_ok=True)
    x = latents.detach().clone().cpu()
    if dtype is not None:
        x = x.to(dtype)
    torch.save(x, os.path.join(path, ddim_latents_filename(t)))


def load_ddim_latents_at_t(t, ddim_latents_path: str) -> torch.Tensor:
    """utils.py:31-36."""
    p = os.path.join(ddim_latents_path, ddim_latents_filename(int(t)))
    assert os.path.exists(p), f"Missing latents at t {t} path {p}"
    return torch.load(p, map_location="cpu")


class LatentBank:
    """All timesteps of one source video resident on the device: [n_t, 4, T, h, w] fp32 + index by t.
    Replaces the per-step torch.load(...).to(device) at pipeline_i2vgen_xl.py:1637, :1648-1650, :1670."""

    def __init__(self, per_t: Dict[int, torch.Tensor], device, pin_host: bool = False):
        self.index = {int(t): i for i, t in enumerate(sorted(per_t))}
        stack = torch.stack([per_t[t].reshape(per_t[t].shape[-4:]).float() for t in sorted(per_t)])
        self.host = stack.pin_memory() if pin_host else None
        self.data = stack.to(device)

    @classmethod
    def from_dir(cls, path: str, timesteps: Sequence[int], device, pin_host: bool = False):
        return cls({int(t): load_ddim_latents_at_t(t, path) for t in timesteps}, device, pin_host)

    # packed single-file form of one video's latent store (SURVEY §8f-3): the per-timestep files stay the
    # interchange format with the reference, this is the fast path between our own inverse and composite runs
    def save_packed(self, path: str) -> None:
        os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
        ts = sorted(self.index, key=self.index.get)
        torch.save({"timesteps": ts, "latents": self.data.detach().cpu()}, path)

    @classmethod
    def load_packed(cls, path: str, device, pin_host: bool = False) -> "LatentBank":
        blob = torch.load(path, map_location="cpu")
        return cls({int(t): blob["latents"][i] for i, t in enumerate(blob["timesteps"])}, device, pin_host)

    def at(self, t: int) -> torch.Tensor:
        return self.data[self.index[int(t)]]

    def host_at(self, t: int) -> torch.Tensor:
        return self.host[self.index[int(t)]]


@dataclass
class Conditioning:
    """Tensors produced by the (out-of-scope) CLIP/VAE stages for the n_obj+3 branches, on the device in
    the UNet dtype: prompt embeds [nb,77,1024] (:1380-1389), CLIP image embeds [nb,T,1024] (:1540-1541),
    first-frame image latents [nb,4,T,h,w] twice (:1476-1478, :1499-1500), fps [nb] (:1545-1549)."""
    prompt_embeds: torch.Tensor
    image_embeddings: torch.Tensor
    image_latents_first: torch.Tensor
    image_latents: torch.Tensor
    fps: torch.Tensor


class I2VGenXLPipeline:
    def __init__(self, unet, device="cuda", parallel=None, use_cuda_graphs: bool = False, vae=None,
                 vae_encoder=None, image_encoder=None, text_encoder=None, tokenizer=None):
        from .parallel import FrameParallel

        self.unet = unet
        self.vae = vae             # mvoc_b200.vae.AutoencoderKLDecoder for decode_latents, or None
        self.vae_encoder = vae_encoder   # mvoc_b200.vae.AutoencoderKLEncoder for encode_vae_video, or None
        self.image_encoder = image_encoder   # mvoc_b200.clip.CLIPVisionEncoder for encode_image, or None
        self.text_encoder = text_encoder     # mvoc_b200.clip_text.CLIPTextEncoder for encode_prompt, or None
        self.tokenizer = tokenizer           # mvoc_b200.clip_text.CLIPTokenizer for encode_prompt, or None
        self.device = torch.device(device)
        self.parallel = parallel or FrameParallel.single(self.device)
        # A UNet forward is ~2700 launches; enqueuing them from Python takes about as long as the GPU needs
        # to run them (tools/step_probe.py), and with P GPUs the device work shrinks P-fold while the host
        # work does not.  With use_cuda_graphs the forward is captured once per hook configuration (which
        # hooks fire is host-side control flow) and replayed.
        self.use_cuda_graphs = use_cuda_graphs
        self._graphs = {}
        self._graph_pool = None
        self._t_dev = None
        self._static_in = {}
        self.scheduler: Optional[DDIMSchedule] = None
        self._cond_caches = {}     # id(cond) -> {"key": cond (strong ref), "ctx", "il", "fps_emb"}; a few conditionings
        self._plain_in = {}        # latent shape -> 4-slot input buffer of `sample`

    @torch.no_grad()
    def decode_latents(self, latents: torch.Tensor, decode_chunk_size: int = 4) -> torch.Tensor:
        """pipelines/pipeline_i2vgen_xl.py:771-791: latents [b, 4, T, h, w] -> video [b, 3, T, 8h, 8w] fp32, the
        frames decoded `decode_chunk_size` at a time (which bounds the decoder's activation memory)."""
        from .vae import SCALING_FACTOR

        if self.vae is None:
            raise RuntimeError("decode_latents: this pipeline was built without a VAE decoder (vae=None)")
        if decode_chunk_size < 1:
            raise ValueError(f"decode_latents: decode_chunk_size={decode_chunk_size} must be >= 1")
        latents = 1 / SCALING_FACTOR * latents.float()
        b, c, f, h, w = latents.shape
        flat = latents.permute(0, 2, 1, 3, 4).reshape(b * f, c, h, w)
        frames = [self.vae(flat[i:i + decode_chunk_size]) for i in range(0, flat.shape[0], decode_chunk_size)]
        image = torch.cat(frames, dim=0)
        return image.reshape((b, f) + image.shape[1:]).permute(0, 2, 1, 3, 4).float()

    @torch.no_grad()
    def _vae_latents(self, images: torch.Tensor, generator: Optional[torch.Generator] = None,
                     encode_chunk_size: int = 4) -> torch.Tensor:
        """images [n, 3, H, W] in [-1, 1] -> scaled latents [n, 4, H/8, W/8] fp32: vae.encode(x).latent_dist.sample()
        x scaling_factor.  The frames are encoded `encode_chunk_size` at a time (which bounds the encoder's activation
        memory); the noise of the sample is ONE torch.randn((n, 4, h, w)) in fp32 on the generator's device, so the
        chunk size changes nothing else.  Both encode_vae_video and prepare_image_latents go through here."""
        from .vae import SCALING_FACTOR, DiagonalGaussian

        if self.vae_encoder is None:
            raise RuntimeError("encoding frames: this pipeline was built without a VAE encoder (vae_encoder=None)")
        if encode_chunk_size < 1:
            raise ValueError(f"encode_chunk_size={encode_chunk_size} must be >= 1")
        moments = torch.cat([self.vae_encoder(images[i:i + encode_chunk_size])
                             for i in range(0, images.shape[0], encode_chunk_size)])
        post = DiagonalGaussian(moments)
        noise = torch.randn(tuple(post.mean.shape), generator=generator, dtype=torch.float32,
                            device=generator.device if generator is not None else post.mean.device)
        return post.sample(noise.to(post.mean.device)) * SCALING_FACTOR

    def encode_vae_video(self, frames: torch.Tensor, generator: Optional[torch.Generator] = None,
                         encode_chunk_size: int = 4) -> torch.Tensor:
        """pipelines/pipeline_i2vgen_xl.py:893-920: frames [T, 3, H, W] in [-1, 1] -> latents [1, 4, T, H/8, W/8]
        fp32, a sample of the posterior (not its mode) times the scaling factor.  Sample or mode could not be read
        off the reference here; the sample is what its prepare_image_latents takes (diffusers 0.27.2), and this
        method follows it."""
        lat = self._vae_latents(frames, generator, encode_chunk_size)
        return lat.permute(1, 0, 2, 3).unsqueeze(0).contiguous()

    def prepare_image_latents(self, image: torch.Tensor, num_frames: int,
                              generator: Optional[torch.Generator] = None) -> torch.Tensor:
        """pipelines/pipeline_i2vgen_xl.py:860-890 (diffusers 0.27.2) at one video per prompt and guidance 1: images
        [n, 3, H, W] -> [n, 4, T, H/8, W/8] fp32, one row per image (inversion passes one image, a composition the
        first control frame of each branch).  Frame 0 is the encoded, scaled image; frames 1..T-1 are constant
        planes i / (T - 1), the position mask of the later frames.  The posterior noise is one draw over the n
        images (see _vae_latents)."""
        lat = self._vae_latents(image, generator).unsqueeze(2)
        if num_frames > 1:
            pos = torch.arange(1, num_frames, dtype=torch.float32, device=lat.device) / (num_frames - 1)
            pos = pos.view(1, 1, -1, 1, 1).expand(lat.shape[0], lat.shape[1], -1, lat.shape[3], lat.shape[4])
            lat = torch.cat([lat, pos], dim=2)
        return lat

    @torch.no_grad()
    def encode_image(self, frames: torch.Tensor, encode_chunk_size: int = 64) -> torch.Tensor:
        """I2VGenXLPipeline._encode_image (diffusers 0.27.2, called from pipelines/pipeline_i2vgen_xl.py:1391-1541):
        CLIP-normalised images [B, 3, 224, 224] (mvoc_b200.clip.clip_image_input) -> image_embeds.unsqueeze(1)
        [B, 1, 1024] in the encoder's dtype, `encode_chunk_size` images at a time (which bounds the activation
        memory).  Every kernel of the tower computes an image's rows from that image alone and the GEMM's K order
        does not depend on its tile plan, so the result is bit-identical for every chunk size (tested on the GPU)."""
        if self.image_encoder is None:
            raise RuntimeError("encode_image: this pipeline was built without a CLIP image encoder (image_encoder=None)")
        if encode_chunk_size < 1:
            raise ValueError(f"encode_image: encode_chunk_size={encode_chunk_size} must be >= 1")
        frames = frames.to(self.device)
        emb = torch.cat([self.image_encoder(frames[i:i + encode_chunk_size])
                         for i in range(0, frames.shape[0], encode_chunk_size)])
        return emb.unsqueeze(1)

    @torch.no_grad()
    def encode_prompt(self, prompts, encode_chunk_size: int = 64) -> torch.Tensor:
        """I2VGenXLPipeline.encode_prompt (diffusers 0.27.2) for one prompt list, clip_skip None: each prompt (None
        becomes "") is tokenized to 77 ids (padding "max_length", truncation) and encoded by the text tower without an
        attention mask -> last_hidden_state [n, 77, 1024] in the encoder's dtype, `encode_chunk_size` prompts at a time.
        As in encode_image, every kernel computes a prompt's rows from that prompt alone, so the result is
        bit-identical for every chunk size (tested on the GPU)."""
        if self.text_encoder is None or self.tokenizer is None:
            raise RuntimeError("encode_prompt: this pipeline was built without a CLIP text encoder and tokenizer "
                               "(text_encoder=None or tokenizer=None)")
        if encode_chunk_size < 1:
            raise ValueError(f"encode_prompt: encode_chunk_size={encode_chunk_size} must be >= 1")
        prompts = [prompts] if prompts is None or isinstance(prompts, str) else list(prompts)
        ids = self.tokenizer(["" if p is None else p for p in prompts]).to(self.device)
        return torch.cat([self.text_encoder(ids[i:i + encode_chunk_size])
                          for i in range(0, ids.shape[0], encode_chunk_size)])

    def drop_graphs(self) -> None:
        """Forget every captured graph.  The private pool goes with them: torch asserts when a capture re-uses a
        pool handle whose graphs have all been destroyed."""
        self._graphs.clear()
        self._graph_pool = None

    def static_input(self, shape, device) -> torch.Tensor:
        """Persistent UNet input buffer [n_branches, 4, T, h, w] (captured graphs read from it)."""
        key = tuple(shape)
        buf = self._static_in.get(key)
        if buf is None:
            buf = torch.empty(key, dtype=self.unet.dtype, device=device)
            self._static_in[key] = buf
        return buf

    def step_kinds(self, timesteps, masks) -> list:
        """Indices of the first step of every distinct hook configuration in `timesteps` (host-side only)."""
        seen, firsts = set(), []
        for i, t in enumerate(timesteps):
            pnp_utils.register_time_all(self, t, masks)
            sig = pnp_utils.hook_signature(self.unet)
            if sig not in seen:
                seen.add(sig)
                firsts.append(i)
        return firsts

    # ------------------------------------------------------------------ UNet driver
    def _unet_forward(self, sample, t: int, cond: Conditioning):
        """I2VGenXLUnetExtension.forward (pipeline_i2vgen_xl.py:109-362) -> noise prediction of THIS rank's
        frames, [b, t_local, 4, h, w].  The context tokens and the image-latent stem input do not depend on
        t, so they are computed on the first step only (the reference recomputes them every step, T times).
        With world_size > 1 every rank runs all branches on its T/P frames (frame-parallel)."""
        unet = self.unet
        par = self.parallel
        unet.ctx.parallel = par if par.world > 1 else None
        b, c, T, h, w = sample.shape
        f0, f1 = par.frame_range(T) if par.world > 1 else (0, T)
        tl = f1 - f0
        cache = self._cond_caches.get(id(cond))
        if cache is None or cache["key"] is not cond:
            ctx = unet.context(cond.prompt_embeds, cond.image_latents, cond.image_embeddings)
            ctx = ctx.repeat_interleave(tl, dim=0)                              # one context per frame (:255-260)
            il = unet.stem_condition(cond.image_latents_first)                 # [(b T), c, h, w]
            il = il.view(b, T, c, h, w)[:, f0:f1].reshape(b * tl, c, h, w).contiguous()
            fps_emb = unet.fps_embedding(unet.time_proj(cond.fps).to(unet.dtype))
            cache = {"key": cond, "ctx": ctx, "il": il, "fps_emb": fps_emb}
            if len(self._cond_caches) >= 8:      # graphs captured for an evicted conditioning point at freed tensors
                self._cond_caches.clear()
                self.drop_graphs()
            self._cond_caches[id(cond)] = cache
        if self._t_dev is None:
            self._t_dev = torch.zeros(1, dtype=torch.int64, device=sample.device)
        self._t_dev.fill_(int(t))        # device-side timestep: the captured graph reads it at replay time
        if not self.use_cuda_graphs:
            return self._unet_body(sample, cond, cache, (f0, f1))
        static = self.static_input(sample.shape, sample.device)
        if sample.data_ptr() != static.data_ptr():
            static.copy_(sample)
        sample = static
        # the capture bakes in control flow (which hooks fire) and addresses (input buffer, conditioning cache,
        # token masks): all of them are part of the key
        mask = getattr(unet.conv_out, "mask", None)
        mask_handle = pnp_utils._MASKS.handle(mask) if mask else None
        key = (pnp_utils.hook_signature(unet), tuple(sample.shape), id(cond), par.world,
               mask_handle.serial if mask_handle is not None else 0, unet.__dict__.get("derived_epoch", 0))
        entry = self._graphs.get(key)
        if entry is None:
            # eager warm-up on a side stream (lazy weight fusions, cuDNN autotune, mask caches), then capture
            side = torch.cuda.Stream(device=sample.device)
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                self._unet_body(sample, cond, cache, (f0, f1))
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            if self._graph_pool is None:
                self._graph_pool = torch.cuda.graph_pool_handle()
            graph = torch.cuda.CUDAGraph()
            timer = ops._timer
            ops.set_timer(None)          # per-launch events cannot be recorded inside a capture
            try:
                with torch.cuda.graph(graph, pool=self._graph_pool):
                    out = self._unet_body(sample, cond, cache, (f0, f1))
            finally:
                ops.set_timer(timer)
            entry = (graph, out, mask_handle, cond)   # the handle / cond keep the captured addresses alive
            self._graphs[key] = entry
        entry[0].replay()
        return entry[1]

    def _unet_body(self, sample, cond, cache, frames):
        unet = self.unet
        self.parallel.begin_forward()      # peer-memory exchange: same arena offsets / sites in every forward
        b, c, T, h, w = sample.shape
        f0, f1 = frames
        tl = f1 - f0
        ts = self._t_dev.expand(b)
        t_emb = unet.time_embedding(unet.time_proj(ts).to(unet.dtype))
        emb = (t_emb + cache["fps_emb"]).repeat_interleave(tl, dim=0)            # :196-197
        frm = sample[:, :, f0:f1].permute(0, 2, 1, 3, 4).reshape(b * tl, c, h, w)     # :283
        x = unet.stem(frm, cache["il"], T)                                      # :282-290
        fwd_up = any(s % (2 ** unet.num_upsamplers) != 0 for s in (h, w))
        out = unet.body(x, emb, cache["ctx"], T, fwd_up)                        # [(b t_local), 4, h, w]
        return out.view(b, tl, *out.shape[1:])

    def _gather_prediction(self, pred_local: torch.Tensor) -> torch.Tensor:
        """[k, t_local, 4, h, w] -> [k, 4, T, h, w] contiguous (the latents' layout)."""
        if self.parallel.world > 1:
            pred_local = self.parallel.gather_frames(pred_local)
        return pred_local.permute(0, 2, 1, 3, 4).contiguous()

    # ------------------------------------------------------------------ composition
    @torch.no_grad()
    def sample_with_pnp_pipeline_with_edit_prompt_extraction_with_attn_injection(
        self,
        cond: Conditioning,
        latents: torch.Tensor,
        bg_bank: LatentBank,
        obj_banks: Sequence[LatentBank],
        obj_mask: Sequence[Tuple[torch.Tensor, torch.Tensor]],
        num_inference_steps: int = 50,
        guidance_scale: float = 9.0,
        ddim_init_latents_t_idx: int = 0,
        fusion_steps: Tuple[int, int] = (0, 1),
        random_noise_ratio: float = 0.0,
        obj_random_noise_fusion: bool = False,
        obj_ddim_latents_idx_offset: Optional[Sequence[int]] = None,
        max_steps: Optional[int] = None,
        start_step: int = 0,
        host_io: bool = False,
        callback: Optional[Callable] = None,
    ) -> torch.Tensor:
        """Composition loop, pipeline_i2vgen_xl.py:1552-1734.  `latents` [1,4,T,h,w] fp32 (device) is
        updated in place and returned.  With host_io the step's source latents come from pinned host
        memory and the updated latents are read back every step (what the reference's per-step
        torch.load / progress reporting does)."""
        n_obj = len(obj_banks)
        nb = n_obj + 3
        sched = self.scheduler or DDIMSchedule(num_inference_steps)
        timesteps_full = sched.timesteps
        timesteps = timesteps_full[ddim_init_latents_t_idx:]                    # :1554
        offs = list(obj_ddim_latents_idx_offset or [0] * n_obj)
        obj_fusion_timesteps = [[timesteps_full[offs[i]:][j] for j in range(*fusion_steps)]
                                for i in range(n_obj)]                          # :1560-1566
        fusion_counter = 0                                                      # never incremented (:1634)
        E = latents.numel()
        T = latents.shape[2]
        mask_f = torch.stack([m[0][0, 0].reshape(-1).float() for m in obj_mask]).contiguous()  # [n_obj, T*h*w]
        masks = list(obj_mask)
        unet_in = self.static_input((nb,) + tuple(latents.shape[1:]), latents.device)
        objs = torch.empty((n_obj,) + tuple(latents.shape[1:]), dtype=torch.float32, device=latents.device)
        bg = torch.empty(tuple(latents.shape[1:]), dtype=torch.float32, device=latents.device)
        host_out = self._pinned_out(latents) if host_io else None
        for i, t in enumerate(timesteps):
            if i < start_step:
                continue
            if max_steps is not None and i >= start_step + max_steps:
                break
            do_fusion = fusion_steps[0] <= i < fusion_steps[1]                  # :1639
            obj_ts = [obj_fusion_timesteps[j][fusion_counter] if do_fusion else t for j in range(n_obj)]
            if host_io:
                bg.copy_(bg_bank.host_at(t), non_blocking=True)                # :1637
                for j in range(n_obj):
                    objs[j].copy_(obj_banks[j].host_at(obj_ts[j]), non_blocking=True)  # :1648-1650 / :1670
            else:
                bg.copy_(bg_bank.at(t))
                for j in range(n_obj):
                    objs[j].copy_(obj_banks[j].at(obj_ts[j]))
            # fusion (:1644-1663) + cat([bg, objs, latents, latents]) (:1676) in one launch
            ops.latent_composite_(latents, bg, objs, mask_f if do_fusion else None, unet_in,
                                  random_noise_ratio, do_fusion, obj_random_noise_fusion)
            pnp_utils.register_time_all(self, t, masks)                          # :1684-1685
            noise_pred = self._unet_forward(unet_in, t, cond)                   # :1688-1699
            pred = self._gather_prediction(noise_pred[n_obj + 1:])              # uncond, cond (:1714-1715)
            a_t, a_prev = sched.step_alphas(t)
            ops.cfg_ddim_step_(pred[0], pred[1], latents, guidance_scale, a_t, a_prev)  # :1717-1731
            if host_io:
                host_out.copy_(latents, non_blocking=False)
            if callback is not None:
                callback(i, t, latents)
        return latents

    def _pinned_out(self, like: torch.Tensor) -> torch.Tensor:
        """Pinned host buffer for the per-step read-back, allocated once per shape (cudaHostAlloc takes tens of
        milliseconds when several ranks call it at once — not something to pay inside every loop call)."""
        key = (tuple(like.shape), like.dtype)
        buf = getattr(self, "_host_out", {}).get(key)
        if buf is None:
            buf = torch.empty(like.shape, dtype=like.dtype).pin_memory()
            if not hasattr(self, "_host_out"):
                self._host_out = {}
            self._host_out[key] = buf
        return buf

    # ------------------------------------------------------------------ inversion
    @torch.no_grad()
    def invert(
        self,
        latents: torch.Tensor,
        prompt_embeds: torch.Tensor,
        image_embeddings: torch.Tensor,
        image_latents: torch.Tensor,
        fps: torch.Tensor,
        num_inference_steps: int = 500,
        guidance_scale: float = 1.0,
        output_dir: Optional[str] = None,
        max_steps: Optional[int] = None,
        keep: bool = True,
        save_dtype=torch.float16,
        on_step: Optional[Callable] = None,
        cond: Optional[Conditioning] = None,
    ) -> Dict[int, torch.Tensor]:
        """DDIM inversion loop, pipeline_i2vgen_xl.py:1914-2003 (guidance 1.0 => batch 1, :517).
        Returns {t: latents at level t}; with output_dir also writes ddim_latents_{t}.pt (:1988-1993)."""
        if guidance_scale > 1.0:
            raise NotImplementedError("inversion with classifier-free guidance is not used by the reference configs")
        sched = DDIMSchedule(num_inference_steps, inverse=True)
        if cond is None:    # callers that invert the same video repeatedly pass the object: graphs are keyed on it
            cond = Conditioning(prompt_embeds, image_embeddings, image_latents, image_latents, fps)
        saved: Dict[int, torch.Tensor] = {}
        x = latents
        for i, t in enumerate(sched.timesteps):
            if max_steps is not None and i >= max_steps:
                break
            noise_pred = self._unet_forward(x.to(self.unet.dtype), t, cond)     # :1952-1961
            pred = self._gather_prediction(noise_pred)
            a_src, a_dst = sched.step_alphas(t)
            ops.ddim_inverse_step_(pred, None, x, 1.0, a_src, a_dst)            # :1979
            if keep:
                saved[t] = x.clone()                                            # :1986
            if output_dir is not None:
                save_ddim_latents_at_t(x, t, output_dir, save_dtype)            # :1988-1993
            if on_step is not None:
                on_step(t, x)
        return saved

    # ------------------------------------------------------------------ plain sampling
    def _plain_input(self, latents: torch.Tensor, nb: int) -> Tuple[torch.Tensor, torch.Tensor]:
        """(4-slot buffer, UNet input [nb, 4, T, h, w]) of `sample` (nb = 2 under guidance, else 1).  The input is
        the tail of a persistent 4-slot buffer that ONE mvoc_latent_composite launch fills from the fp32 latents
        (background, one source branch, uncond, cond: all four are the latents), so the cast and the batch copy are
        a library kernel.  The tail is registered as the static input of its shape: captured graphs read it
        without a further copy."""
        shape = tuple(latents.shape[1:])
        buf = self._plain_in.get(shape)
        if buf is None:
            buf = torch.empty((4,) + shape, dtype=self.unet.dtype, device=latents.device)
            self._plain_in[shape] = buf
        view = buf[4 - nb:]
        key = (nb,) + shape
        old = self._static_in.get(key)
        if old is None or old.data_ptr() != view.data_ptr():
            if old is not None:
                self.drop_graphs()       # graphs captured on the old buffer would read stale input
            self._static_in[key] = view
        return buf, self._static_in[key]

    @torch.no_grad()
    def sample(
        self,
        prompt_embeds: torch.Tensor,
        negative_prompt_embeds: Optional[torch.Tensor],
        image_embeddings: torch.Tensor,
        image_latents: torch.Tensor,
        fps: torch.Tensor,
        num_inference_steps: int = 50,
        guidance_scale: float = 9.0,
        latents: Optional[torch.Tensor] = None,
        generator: Optional[torch.Generator] = None,
        max_steps: Optional[int] = None,
        callback: Optional[Callable] = None,
    ) -> torch.Tensor:
        """Plain I2VGenXL sampling, diffusers 0.27.2 ``I2VGenXLPipeline.__call__`` steps 3-7 (the reference's
        pipelines/pipeline_i2vgen_xl.py:980-1216 derives from it): stock UNet, classifier-free guidance, DDIM.

        Tensors come in the shapes `invert` takes: prompt / negative embeds [1,77,1024], CLIP image embeddings
        [1,1,1024], first-frame image latents [1,4,T,h,w], fps [1].  Guidance is on when guidance_scale > 1; the
        UNet batch is then [uncond, cond]: prompt embeds [negative, prompt], image embeddings [zeros, emb]
        (_encode_image), the image latents and fps twice.  At guidance_scale <= 1 it is batch 1, like `invert`.
        `latents` [1,4,T,h,w] is the start (used as fp32; the caller's tensor is not modified); None draws
        torch.randn((1,4,T,h,w)) in fp32 on the generator's device.  Either is scaled by init_noise_sigma
        (prepare_latents; 1.0 for DDIM).
        Returns the final latents [1,4,T,h,w] fp32.  The plain path is the stock forward: MVOC injection hooks
        installed on the UNet are an error, not something to fire silently."""
        if any(pnp_utils.injection_installed(self.unet)):
            raise ValueError("sample: MVOC injection hooks are installed on this UNet (init_pnp / register_*); the "
                             "plain sampling loop runs the stock forward, so use a pipeline without them")
        cfg = guidance_scale > 1.0                                              # do_classifier_free_guidance
        if cfg and negative_prompt_embeds is None:
            raise ValueError(f"sample: guidance_scale={guidance_scale} > 1 needs negative_prompt_embeds")
        dev, dt = self.device, self.unet.dtype
        sched = DDIMSchedule(num_inference_steps)
        b, c, T, h, w = image_latents.shape
        if latents is None:                                                     # prepare_latents
            latents = torch.randn((1, 4, T, h, w), generator=generator, dtype=torch.float32,
                                  device=generator.device if generator is not None else dev)
        x = latents.to(dev, torch.float32) * sched.init_noise_sigma             # scales given latents too (a copy)
        prompt_embeds, image_embeddings = prompt_embeds.to(dev, dt), image_embeddings.to(dev, dt)
        image_latents, fps = image_latents.to(dev, dt), fps.to(dev)
        if cfg:
            prompt_embeds = torch.cat([negative_prompt_embeds.to(dev, dt), prompt_embeds])
            image_embeddings = torch.cat([torch.zeros_like(image_embeddings), image_embeddings])
            image_latents = torch.cat([image_latents, image_latents])
            fps = torch.cat([fps, fps])
        cond = Conditioning(prompt_embeds, image_embeddings, image_latents, image_latents, fps)
        slots, unet_in = self._plain_input(x, 2 if cfg else 1)
        for i, t in enumerate(sched.timesteps):
            if max_steps is not None and i >= max_steps:
                break
            # slots <- [x, x, x, x] in the UNet dtype.  z, bg and objs alias one buffer, which the kernel's __restrict__
            # pointers allow only because it never writes z when do_fusion is off (csrc/latent.cu): keep that so.
            ops.latent_composite_(x, x, x, None, slots, 0.0, False)
            noise_pred = self._unet_forward(unet_in, t, cond)
            pred = self._gather_prediction(noise_pred)
            a_t, a_prev = sched.step_alphas(t)
            ops.cfg_ddim_step_(pred[0], pred[1] if cfg else None, x, guidance_scale, a_t, a_prev)
            if callback is not None:
                callback(i, t, x)
        return x


# --------------------------------------------------------------------------
# composite.py:38-69
# --------------------------------------------------------------------------
def init_pnp(pipe: I2VGenXLPipeline, scheduler: DDIMSchedule, config) -> dict:
    """Fractions of n_steps -> leading slices of the FULL timestep grid; installs the hooks.
    `config` needs n_steps, pnp_f_t, pnp_spatial_attn_t, pnp_temp_attn_t, inject_background."""
    conv_t = int(config.n_steps * config.pnp_f_t)
    spa_t = int(config.n_steps * config.pnp_spatial_attn_t)
    tmp_t = int(config.n_steps * config.pnp_temp_attn_t)
    ts = scheduler.timesteps
    conv_ts = ts[:conv_t] if conv_t >= 0 else []
    spa_ts = ts[:spa_t] if spa_t >= 0 else []
    tmp_ts = ts[:tmp_t] if tmp_t >= 0 else []
    pnp_utils._MASKS.clear()       # a new run: drop the token masks (and graphs keyed on them) of the previous one
    pipe.drop_graphs()
    pnp_utils.modify_diffuser_attention_forward(pipe.unet)
    pnp_utils.register_temp_attention_pnp(pipe, tmp_ts, config.inject_background)
    pnp_utils.register_spatial_attention_pnp(pipe, spa_ts, config.inject_background)
    pnp_utils.register_temp_conv_injection(pipe, conv_ts)
    pnp_utils.register_out_conv_injection(pipe, conv_ts)
    pnp_utils.register_resnet_injection(pipe, conv_ts)
    pipe.scheduler = scheduler
    return {"conv": conv_ts, "spatial": spa_ts, "temporal": tmp_ts}
