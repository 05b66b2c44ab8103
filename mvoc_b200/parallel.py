"""Multi-GPU partition of the composition path: one process per GPU, frames sharded across ranks.

The path shards naturally along the frame axis (SURVEY §8e): resnets, spatial transformers,
cross-attention, down/up-sampling and every mask blend are independent per frame, so each rank owns
T/P frames of ALL n_obj+3 branches — which also keeps MVOC's source->composite Q/K injection local to a
rank (no Q/K exchange at all).  Only the temporal operators (temporal conv, temporal attention,
5-D GroupNorm statistics) need every frame of a pixel; around those the activation is re-laid out from
frame shards to pixel shards and back with one NCCL all-to-all each way over NVLink/NVSwitch.

world_size == 1 is a strict no-op (no process group is created).
"""
from __future__ import annotations

import os
from typing import Optional

import torch
import torch.distributed as dist


class _RawDeviceMemory:
    """__cuda_array_interface__ view of a raw device pointer (torch.as_tensor wraps it without copying)."""

    def __init__(self, ptr: int, nbytes: int):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 3}


class PeerExchange:
    """The frame-shard <-> pixel-shard exchange as one-sided puts over NVLink peer memory (csrc/exchange.cu,
    include/mvoc_b200.h `mvoc_exchange_*`): every rank owns an arena that all peers map through CUDA IPC; buffers are
    bump-allocated in lockstep on all ranks (same sizes, same order => same offset everywhere) and the bump pointer
    and the site counter are reset at the start of every UNet forward, so a forward always uses the same addresses
    (what a captured CUDA graph needs).  torch.distributed only carries the 64-byte IPC handles at start-up.

    Re-use of the arena between two forwards is safe because every step gathers the noise prediction of all ranks
    (an NCCL collective on the same stream) after its last exchange: no rank can start the puts of forward k+1
    before every rank has finished reading the buffers of forward k."""

    def __init__(self, group, world: int, rank: int, device, arena_bytes: int):
        import ctypes

        from . import _cabi

        self.world, self.rank, self.device = world, rank, torch.device(device)
        self._lib = _cabi.load()
        self._ct = ctypes
        self.header = int(self._lib.mvoc_exchange_header_bytes())
        self.max_sites = int(self._lib.mvoc_exchange_max_sites())
        self.bytes = int(arena_bytes)
        base = ctypes.c_void_p()
        handle = ctypes.create_string_buffer(64)
        _cabi.check(self._lib.mvoc_exchange_arena_create(self.bytes, ctypes.byref(base), handle),
                    "mvoc_exchange_arena_create")
        self.base = base.value
        handles = [None] * world
        dist.all_gather_object(handles, bytes(handle.raw), group=group)
        self.peer_bases = (ctypes.c_void_p * world)()
        self._opened = []
        for r in range(world):
            if r == rank:
                self.peer_bases[r] = self.base
                continue
            p = ctypes.c_void_p()
            _cabi.check(self._lib.mvoc_exchange_arena_open(ctypes.create_string_buffer(handles[r], 64), ctypes.byref(p)),
                        "mvoc_exchange_arena_open")
            self.peer_bases[r] = p.value
            self._opened.append(p.value)
        self._mem = torch.as_tensor(_RawDeviceMemory(self.base, self.bytes), device=self.device)
        # put + wait of an exchange as ONE launch (the put kernel's last CTA waits for the peers); MVOC_EXCHANGE_WAIT=
        # separate keeps the two-launch form (A/B switch)
        self.fused_wait = os.environ.get("MVOC_EXCHANGE_WAIT", "fused") != "separate"
        self._flag = _cabi.MVOC_EXCHANGE_WAIT_FUSED if self.fused_wait else 0
        self.reset()
        dist.barrier(group=group)      # every arena is mapped everywhere before the first put

    def reset(self) -> None:
        """Start of a UNet forward: the same allocation sequence yields the same offsets and sites."""
        self._cursor = self.header
        self._site = 0

    def _alloc(self, shape, dtype):
        n = 1
        for d in shape:
            n *= int(d)
        nbytes = n * torch.empty(0, dtype=dtype).element_size()
        off = self._cursor
        self._cursor = (off + nbytes + 255) // 256 * 256
        if self._cursor > self.bytes:
            raise MemoryError(f"exchange arena of {self.bytes >> 20} MiB exhausted (MVOC_EXCHANGE_ARENA_MB)")
        return off, self._mem[off:off + nbytes].view(dtype).view(*shape)

    def _next_site(self) -> int:
        s = self._site
        self._site += 1
        if s >= self.max_sites:
            raise RuntimeError(f"more than {self.max_sites} exchanges in one forward")
        return s

    def _stream(self) -> int:
        return torch.cuda.current_stream().cuda_stream

    def _wait(self, site: int) -> None:
        """The data of every peer has arrived when this returns (in stream order)."""
        from . import _cabi, ops

        if self.fused_wait:            # the put kernel already waited
            ops._count(1)
            return
        _cabi.check(self._lib.mvoc_exchange_wait(self.base, self.world, site, self._stream()), "mvoc_exchange_wait")
        ops._count(2)

    def to_pixel_shards(self, x: torch.Tensor, b: int, tl: int, S: int, C: int) -> torch.Tensor:
        """x contiguous [b*tl, ..., C] (this rank's frames) -> [b*T, 1, S/P, C] (all frames, this rank's pixels)."""
        from . import _cabi, ops

        P = self.world
        off, out = self._alloc((b * tl * P, 1, S // P, C), x.dtype)
        site = self._next_site()
        with ops._Timed(("exchange", "to_pixel", b * tl, S, C), 2.0 * x.numel() * x.element_size()):
            _cabi.check(self._lib.mvoc_exchange_to_pixel_shards(x.data_ptr(), self.peer_bases, off, self.rank, P, b, tl,
                                                                S, C, ops._dt(x), site | self._flag, self._stream()),
                        "mvoc_exchange_to_pixel_shards")
            self._wait(site)
        return out

    def to_frame_shards(self, y: torch.Tensor, b: int, T: int, sp: int, C: int, h: int, w: int) -> torch.Tensor:
        """y contiguous [b*T, 1, S/P, C] -> [b*tl, h, w, C] (this rank's frames, all pixels)."""
        from . import _cabi, ops

        P = self.world
        off, out = self._alloc((b * (T // P), h, w, C), y.dtype)
        site = self._next_site()
        with ops._Timed(("exchange", "to_frame", b * T, sp, C), 2.0 * y.numel() * y.element_size()):
            _cabi.check(self._lib.mvoc_exchange_to_frame_shards(y.data_ptr(), self.peer_bases, off, self.rank, P, b, T, sp,
                                                                C, ops._dt(y), site | self._flag, self._stream()),
                        "mvoc_exchange_to_frame_shards")
            self._wait(site)
        return out

    def allgather(self, t: torch.Tensor) -> torch.Tensor:
        """[...] fp32 / any dtype, contiguous, a multiple of 16 bytes -> [P, ...] (rank order)."""
        from . import _cabi, ops

        P = self.world
        nbytes = t.numel() * t.element_size()
        off, out = self._alloc((P,) + tuple(t.shape), t.dtype)
        site = self._next_site()
        with ops._Timed(("exchange", "allgather", nbytes), float(nbytes) * P):
            _cabi.check(self._lib.mvoc_exchange_allgather(t.data_ptr(), nbytes, self.peer_bases, off, self.rank, P,
                                                          site | self._flag, self._stream()), "mvoc_exchange_allgather")
            self._wait(site)
        return out

    def close(self) -> None:
        for p in self._opened:
            self._lib.mvoc_exchange_arena_close(p)
        self._opened = []
        if self.base:
            self._mem = None
            self._lib.mvoc_exchange_arena_destroy(self.base)
            self.base = None


def exchange_arena_mb(n_branches: int, n_frames: int, latent_h: int, latent_w: int, world: int) -> int:
    """MiB of peer-exchange arena a composition of this geometry needs on each of `world` ranks.  Every temporal
    operator of a forward bump-allocates two buffers of (tensor / P) bytes, about 60 tensors of the first level's
    size (n_branches x n_frames x h x w x 320 channels, bf16); clamped to [4096, 32768].  MVOC_EXCHANGE_ARENA_MB,
    when set, wins."""
    env = os.environ.get("MVOC_EXCHANGE_ARENA_MB")
    if env:
        return int(env)
    l0 = n_branches * n_frames * latent_h * latent_w * 320 * 2
    return int(min(32768, max(4096, 60 * l0 / world / 2 ** 20)))


class FrameParallel:
    def __init__(self, group=None, world: int = 1, rank: int = 0, device=None):
        self.group = group
        self.world = world
        self.rank = rank
        self.device = device
        self.peer: Optional[PeerExchange] = None     # NVLink peer-memory exchange (CUDA devices, world > 1)

    # ------------------------------------------------------------------ setup
    @classmethod
    def single(cls, device=None) -> "FrameParallel":
        return cls(None, 1, 0, device)

    @classmethod
    def from_env(cls, device=None, backend: Optional[str] = None, arena_mb: Optional[int] = None) -> "FrameParallel":
        """The partition torchrun's environment describes.  The peer-exchange arena is `arena_mb` MiB
        (exchange_arena_mb), or MVOC_EXCHANGE_ARENA_MB / 6144 when it is not given."""
        world = int(os.environ.get("WORLD_SIZE", "1"))
        if world == 1:
            return cls.single(device)
        if not dist.is_initialized():
            if backend is None:
                backend = "nccl" if (device is not None and torch.device(device).type == "cuda") else "gloo"
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group(backend=backend)
        fp = cls(dist.group.WORLD, dist.get_world_size(), dist.get_rank(), device)
        # MVOC_EXCHANGE=nccl keeps the NCCL all-to-all / all-gather exchange (the A/B baseline of bench.py)
        if (device is not None and torch.device(device).type == "cuda"
                and os.environ.get("MVOC_EXCHANGE", "peer") != "nccl"):
            mb = arena_mb if arena_mb is not None else int(os.environ.get("MVOC_EXCHANGE_ARENA_MB", "6144"))
            fp.peer = PeerExchange(fp.group, fp.world, fp.rank, device, mb << 20)
        return fp

    def begin_forward(self) -> None:
        """Called by the pipeline at the start of every UNet forward."""
        if self.peer is not None:
            self.peer.reset()

    def shutdown(self) -> None:
        if self.peer is not None:
            torch.cuda.synchronize()
            if dist.is_initialized():
                dist.barrier(group=self.group)
            self.peer.close()
            self.peer = None
        if self.world > 1 and dist.is_initialized():
            dist.destroy_process_group()

    def describe(self) -> str:
        if self.world == 1:
            return "single GPU"
        how = "NVLink peer-memory puts (mvoc_exchange_*)" if self.peer is not None else "NCCL all-to-all"
        return f"frame-parallel x{self.world} (re-layout around temporal ops: {how})"

    # ------------------------------------------------------------------ plumbing
    def barrier(self) -> None:
        if self.world > 1:
            dist.barrier(group=self.group)

    def broadcast_module(self, module: torch.nn.Module, src: int = 0) -> None:
        """Overwrite every parameter and buffer of `module` in place with rank `src`'s (random-init weights are
        then the same on every rank, however much of its RNG each rank has drawn)."""
        if self.world == 1:
            return
        for t in module.state_dict().values():
            dist.broadcast(t, src=src, group=self.group)

    def max_over_ranks(self, value: float) -> float:
        if self.world == 1:
            return float(value)
        t = torch.tensor([float(value)], dtype=torch.float64, device=self.device if self.device is not None else "cpu")
        dist.all_reduce(t, op=dist.ReduceOp.MAX, group=self.group)
        return float(t.item())

    # ------------------------------------------------------------------ shard geometry
    def frame_range(self, n_frames: int):
        """(lo, hi) of the frames this rank owns."""
        if n_frames % self.world != 0:
            raise ValueError(f"n_frames={n_frames} is not divisible by world_size={self.world}")
        per = n_frames // self.world
        return (self.rank * per, (self.rank + 1) * per)

    def pixel_range(self, n_pixels: int):
        """(lo, hi) of the pixels this rank owns while a temporal operator runs."""
        if n_pixels % self.world != 0:
            raise ValueError(f"h*w={n_pixels} is not divisible by world_size={self.world}")
        per = n_pixels // self.world
        return (self.rank * per, (self.rank + 1) * per)

    # ------------------------------------------------------------------ re-layout (the exchange step)
    def to_pixel_shards(self, x: torch.Tensor, num_frames: int) -> torch.Tensor:
        """[(b t_local), h, w, C] (this rank's frames, all pixels) -> [(b T), 1, S/P, C] (all frames, this
        rank's pixels): one all-to-all.  Rows stay in (video, frame, pixel) order."""
        P = self.world
        btl, h, w, C = x.shape
        tl = num_frames // P
        b, S = btl // tl, h * w
        sp = S // P
        if S % P != 0:
            raise ValueError(f"h*w={S} is not divisible by world_size={P}")
        if self.peer is not None:
            return self.peer.to_pixel_shards(x.contiguous(), b, tl, S, C)
        send = x.contiguous().view(b, tl, P, sp, C).permute(2, 0, 1, 3, 4).contiguous()   # [dst, b, tl, sp, C]
        recv = torch.empty_like(send)                                            # [src, b, tl, sp, C]
        dist.all_to_all_single(recv, send, group=self.group)
        return recv.permute(1, 0, 2, 3, 4).contiguous().view(b * num_frames, 1, sp, C)   # frame = src*tl + i

    def to_frame_shards(self, y: torch.Tensor, num_frames: int, h: int, w: int) -> torch.Tensor:
        """Inverse of to_pixel_shards: [(b T), 1, S/P, C] -> [(b t_local), h, w, C]."""
        P = self.world
        bT, _, sp, C = y.shape
        b, tl = bT // num_frames, num_frames // P
        if self.peer is not None:
            return self.peer.to_frame_shards(y.contiguous(), b, num_frames, sp, C, h, w)
        send = y.contiguous().view(b, P, tl, sp, C).permute(1, 0, 2, 3, 4).contiguous()   # [dst(frame owner), b, tl, sp, C]
        recv = torch.empty_like(send)                                            # [src(pixel owner), b, tl, sp, C]
        dist.all_to_all_single(recv, send, group=self.group)
        return recv.permute(1, 2, 0, 3, 4).contiguous().view(b * tl, h, w, C)    # pixel = src*sp + j

    def gather_partials(self, partial: torch.Tensor) -> torch.Tensor:
        """GroupNorm partial statistics of every rank's pixel shard: [N,G,chunks,2] -> [P,N,G,chunks,2]."""
        partial = partial.contiguous()
        if self.peer is not None and (partial.numel() * partial.element_size()) % 16 == 0:
            return self.peer.allgather(partial)
        out = torch.empty((self.world * partial.shape[0],) + tuple(partial.shape[1:]), dtype=partial.dtype,
                          device=partial.device)
        dist.all_gather_into_tensor(out, partial, group=self.group)   # concatenated along dim 0
        return out.view((self.world,) + tuple(partial.shape))

    def gather_frames(self, x: torch.Tensor) -> torch.Tensor:
        """[k, t_local, ...] on every rank -> [k, T, ...] (frames in rank order)."""
        x = x.contiguous()
        out = torch.empty((self.world * x.shape[0],) + tuple(x.shape[1:]), dtype=x.dtype, device=x.device)
        dist.all_gather_into_tensor(out, x, group=self.group)
        out = out.view((self.world,) + tuple(x.shape))
        k, tl = x.shape[0], x.shape[1]
        return out.permute(1, 0, 2, *range(3, out.dim())).contiguous().view(k, self.world * tl, *x.shape[2:])

    # ------------------------------------------------------------------ temporal operators, replicated
    # When a level's h*w does not divide by the number of ranks (config 5's 11x20 level on 8 GPUs) — or is at
    # most MVOC_FP_GATHER_MAX_PIXELS (off by default; the low-resolution levels are latency-bound) — the frames
    # are all-gathered instead, every rank runs the temporal operator on all pixels and keeps its own frames:
    # one collective instead of two, no GroupNorm statistics exchange, P-fold redundant work on a small tensor.
    _GATHER_MAX_PIXELS = int(os.environ.get("MVOC_FP_GATHER_MAX_PIXELS", "0") or 0)

    def _replicate(self, h: int, w: int) -> bool:
        return (h * w) % self.world != 0 or h * w <= self._GATHER_MAX_PIXELS

    def _temporal_replicated(self, module, hidden_states: torch.Tensor, num_frames: int) -> torch.Tensor:
        btl, h, w, C = hidden_states.shape
        tl = num_frames // self.world
        b = btl // tl
        full = self.gather_frames(hidden_states.contiguous().view(b, tl, h, w, C)).view(b * num_frames, h, w, C)
        y = module.forward_local(full, num_frames, None)
        f0, f1 = self.frame_range(num_frames)
        return y.view(b, num_frames, h, w, C)[:, f0:f1].contiguous().view(b * tl, h, w, C)

    # ------------------------------------------------------------------ temporal operators on pixel shards
    def temporal_transformer(self, module, hidden_states: torch.Tensor, num_frames: int) -> torch.Tensor:
        _, h, w, _ = hidden_states.shape
        if self._replicate(h, w):
            return self._temporal_replicated(module, hidden_states, num_frames)   # ctx.full_hw stays None
        xs = self.to_pixel_shards(hidden_states, num_frames)
        module.ctx.full_hw = (h, w)
        try:
            ys = module.forward_local(xs, num_frames, self.gather_partials)
        finally:
            module.ctx.full_hw = None
        return self.to_frame_shards(ys, num_frames, h, w)

    def temporal_conv(self, module, hidden_states: torch.Tensor, num_frames: int) -> torch.Tensor:
        _, h, w, _ = hidden_states.shape
        if self._replicate(h, w):
            return self._temporal_replicated(module, hidden_states, num_frames)
        xs = self.to_pixel_shards(hidden_states, num_frames)
        ys = module.forward_local(xs, num_frames, self.gather_partials)
        return self.to_frame_shards(ys, num_frames, h, w)
