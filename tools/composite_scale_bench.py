"""composite.py end to end, frame-parallel over N GPUs of one node: where the time of a composition goes.

    python tools/composite_scale_bench.py [--gpus 1 2 4 8] [--out profiles/r08_composite_scale.jsonl]

For each N this runs `python -m torch.distributed.run --standalone --nproc-per-node N` on this file in worker mode,
which calls `mvoc_b200.composite.main` on one entry of BASELINE config 2's geometry: 16 frames of 512 x 512 px
(64 x 64 latents), background + 2 objects, 50 DDIM steps from the first (ddim_init_latents_t_idx 0, the boat_surf
injection knobs bench.py uses), `--synthetic` inputs and random-init UNet weights (rank 0's, broadcast), and a
full-width random-init AutoencoderKL decoder file, so every rank decodes and writes its own frames.  Each rank times
the phases of the run with host clocks around device synchronisations (the loop's steps with CUDA events recorded in
the step callback, so the loop itself is not synchronised), and the slowest rank's time of each phase is reported:

  init_s          FrameParallel.from_env: process group, CUDA-IPC peer arena (sized by parallel.exchange_arena_mb)
  weights_s       UNet random init, broadcast from rank 0, VAE decoder load, pipeline built
  conditioning_s  the entry's hooks, synthetic inputs and latent banks (run_entry up to the first step)
  first_step_ms   the first loop step, which captures the CUDA graph of its hook configuration
  ms_per_step     median of the steps that capture no graph; capture_steps lists the steps that do
  decode_s        decode_latents of this rank's frames; write_frames_s / write_latents_s the PNG and .pt writes
  e2e_s           composite.main from call to return (ends with a barrier), frames_per_s = 16 / e2e_s

One JSON line per N, with the GPU's name, power limit and SM clock read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

FRAMES, PX, N_OBJ, STEPS = 16, 512, 2, 50


def entry(data_dir: str) -> dict:
    return {"active": True, "video_name": "config2", "edited_video_name": "scale", "data_dir": data_dir,
            "image_size": [PX, PX], "n_frames": FRAMES, "n_steps": STEPS, "ddim_init_latents_t_idx": 0,
            "pnp_f_t": 0.1, "pnp_spatial_attn_t": 1.0, "pnp_temp_attn_t": 1.0, "random_noise_ratio": 0.0,
            "fusion_step": [0, 1], "obj_mask_path": [f"obj{j}_mask" for j in range(N_OBJ)],
            "obj_ddim_latents_path": [f"obj{j}/ddim_latents" for j in range(N_OBJ)]}


def worker(args) -> None:
    """One rank: composite.main with the phase timers wrapped around the library calls it makes."""
    from mvoc_b200 import composite, parallel, pipeline, vae

    rank = int(os.environ.get("RANK", "0"))
    rec = {"steps_ms": [], "capture_steps": []}
    sync = torch.cuda.synchronize

    def timed(owner, name, key):
        real = getattr(owner, name)

        def wrapper(*a, **kw):
            sync()
            t = time.perf_counter()
            out = real(*a, **kw)
            sync()
            rec[key] = rec.get(key, 0.0) + time.perf_counter() - t
            return out

        setattr(owner, name, wrapper)

    real_from_env = parallel.FrameParallel.from_env

    def from_env(*a, **kw):
        t = time.perf_counter()
        out = real_from_env(*a, **kw)
        sync()
        rec["init_s"] = time.perf_counter() - t
        rec["t_init_end"] = time.perf_counter()
        return out

    parallel.FrameParallel.from_env = from_env
    real_init = pipeline.I2VGenXLPipeline.__init__

    def init(self, *a, **kw):
        real_init(self, *a, **kw)
        sync()
        rec["weights_s"] = time.perf_counter() - rec["t_init_end"]
        rec["t_pipe"] = time.perf_counter()

    pipeline.I2VGenXLPipeline.__init__ = init
    real_loop = pipeline.I2VGenXLPipeline.sample_with_pnp_pipeline_with_edit_prompt_extraction_with_attn_injection

    def loop(self, *a, **kw):
        sync()
        rec["conditioning_s"] = time.perf_counter() - rec["t_pipe"]
        ev = [torch.cuda.Event(enable_timing=True)]
        graphs = [len(self._graphs)]

        def mark(i, t, lat):
            e = torch.cuda.Event(enable_timing=True)
            e.record()
            ev.append(e)
            if len(self._graphs) > graphs[-1]:
                rec["capture_steps"].append(i)
            graphs.append(len(self._graphs))

        ev[0].record()
        t = time.perf_counter()
        out = real_loop(self, *a, callback=mark, **kw)
        sync()
        rec["loop_s"] = time.perf_counter() - t
        rec["steps_ms"] = [ev[i].elapsed_time(ev[i + 1]) for i in range(len(ev) - 1)]
        return out

    pipeline.I2VGenXLPipeline.sample_with_pnp_pipeline_with_edit_prompt_extraction_with_attn_injection = loop
    timed(pipeline.I2VGenXLPipeline, "decode_latents", "decode_s")
    timed(vae, "save_frames", "write_frames_s")
    timed(torch, "save", "write_latents_s")

    t0 = time.perf_counter()
    done = composite.main(args.template, args.configs_json, synthetic_inputs=True, vae_state_dict=args.vae)
    rec["e2e_s"] = time.perf_counter() - t0
    rec["entries"] = done
    with open(os.path.join(args.rank_dir, f"rank{rank}.json"), "w") as f:
        json.dump(rec, f)


def summarise(n: int, ranks: list, wall_s: float) -> dict:
    def slowest(key):
        vals = [r[key] for r in ranks if key in r]
        return round(max(vals), 4) if vals else None

    r0 = ranks[0]
    steady = [ms for i, ms in enumerate(r0["steps_ms"]) if i not in r0["capture_steps"]]
    ms_step = statistics.median(steady)
    return {
        "n_gpus": n, "workload": f"config 2 geometry: {FRAMES} x {PX}x{PX} px, bg + {N_OBJ} objects, {STEPS} steps, "
                                 "synthetic inputs, random-init UNet and decoder, decode + PNG write",
        "init_s": slowest("init_s"), "weights_s": slowest("weights_s"), "conditioning_s": slowest("conditioning_s"),
        "first_step_ms": round(max(r["steps_ms"][0] for r in ranks), 2),
        "capture_steps": r0["capture_steps"],
        "capture_steps_ms": [round(r0["steps_ms"][i], 2) for i in r0["capture_steps"]],
        "ms_per_step": round(ms_step, 2), "ms_per_step_min_max": [round(min(steady), 2), round(max(steady), 2)],
        "steps_timed": len(steady), "loop_s": slowest("loop_s"),
        "loop_frames_per_s": round(FRAMES / (STEPS * ms_step / 1e3), 3),
        "decode_s": slowest("decode_s"), "write_frames_s": slowest("write_frames_s"),
        "write_latents_s": slowest("write_latents_s"), "e2e_s": slowest("e2e_s"),
        "frames_per_s": round(FRAMES / max(r["e2e_s"] for r in ranks), 3),
        "torchrun_wall_s": round(wall_s, 2),
        "timing": "per phase: host clock around torch.cuda.synchronize on each rank, the slowest rank reported; "
                  "loop steps: CUDA events recorded in the step callback on rank 0",
    }


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--gpus", type=int, nargs="+", default=[1, 2, 4, 8])
    ap.add_argument("--out", default=None, help="append the JSON lines to this file")
    ap.add_argument("--worker", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--template", help=argparse.SUPPRESS)
    ap.add_argument("--configs_json", help=argparse.SUPPRESS)
    ap.add_argument("--vae", help=argparse.SUPPRESS)
    ap.add_argument("--rank_dir", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.worker:
        return worker(args)
    if not torch.cuda.is_available():
        raise SystemExit("composite_scale_bench.py needs CUDA devices (B200); there is no CPU path")
    from mvoc_b200.vae import AutoencoderKLDecoder
    from tools.vae_decode_bench import gpu_info

    have = torch.cuda.device_count()
    with tempfile.TemporaryDirectory() as tmp:
        vae_path = os.path.join(tmp, "vae.pt")
        torch.manual_seed(1)
        torch.save(AutoencoderKLDecoder().state_dict(), vae_path)
        template = os.path.join(ROOT, "configs", "group_composite", "template.yaml")
        for n in args.gpus:
            if n > have:
                print(json.dumps({"n_gpus": n, "skipped": f"{have} GPUs visible"}), flush=True)
                continue
            run_dir = os.path.join(tmp, f"n{n}")
            os.makedirs(run_dir)
            cfg = os.path.join(run_dir, "group.json")
            with open(cfg, "w") as f:
                json.dump([entry(run_dir)], f)
            cmd = [sys.executable, "-m", "torch.distributed.run", "--standalone", "--nproc-per-node", str(n),
                   os.path.abspath(__file__), "--worker", "--template", template, "--configs_json", cfg,
                   "--vae", vae_path, "--rank_dir", run_dir]
            env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""))
            t = time.perf_counter()
            subprocess.run(cmd, check=True, cwd=ROOT, env=env)
            wall = time.perf_counter() - t
            ranks = []
            for r in range(n):
                with open(os.path.join(run_dir, f"rank{r}.json")) as f:
                    ranks.append(json.load(f))
            frames = sorted(os.listdir(os.path.join(run_dir, "Results", "MVOC-B200", "i2vgen-xl", "config2", "scale",
                                                    "composite_frames.synthetic")))
            line = summarise(n, ranks, wall)
            line["frames_written"] = len(frames)
            line.update(gpu_info())
            print(json.dumps(line), flush=True)
            if args.out:
                with open(args.out, "a") as f:
                    f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
