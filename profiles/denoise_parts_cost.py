"""Cost of denoising a frame rendered in parts (rt3_denoise_stage / rt3_denoise_staged, DESIGN.md 3.8), one process per GPU.

    torchrun --nproc_per_node N profiles/denoise_parts_cost.py [out.jsonl] [--reps R] [--configs c2,c4]

For each configuration (its spp and depth, 16 AOV samples, 5 iterations, rows dealt one by one as bench.py deals them):
every rank renders its rows and their AOVs, then stages them into rank 0's stage (distributed.SharedFrame over CUDA IPC:
the stores of the other ranks travel over NVLink; ranks beyond the GPU count share GPUs round-robin, and the line records
both counts), and rank 0 filters the whole frame from it. After a warm-up of every
call, R renders and R_DN stage + filter rounds, each timed by the library's CUDA events (rt3_stats.device_ms, without
copies to the host): the render and the stage as the maximum over the ranks of each repetition, the staged filter on
rank 0. Then rank 0 renders the whole frame alone and records whether rt3_denoise of it equals the staged frame and its
linear rgb bit for bit. Bytes: the stage writes 44 B per pixel (colour and guide 16 B each, albedo 12 B) and 8 B per row;
the share written by ranks other than 0 crosses NVLink when they run on other GPUs. One JSON line per case is printed by rank 0 and appended to the
file (default denoise_parts_cost.jsonl in the working directory), with the GPU's name, power limit and clocks from an
nvidia-smi query in the same run."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import rt3_b200  # noqa: F401,E402
from rt3_b200 import abi, distributed  # noqa: E402
import fullsize as fs  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("out", nargs="?", default="denoise_parts_cost.jsonl")
ap.add_argument("--reps", type=int, default=3)
ap.add_argument("--configs", default="c2,c4")
cli = ap.parse_args()
REPS_DN = 20
ITERATIONS = 5
AOV_SPP = 16
TILE_ROWS = 1

rank = int(os.environ.get("RANK", "0"))
world = int(os.environ.get("WORLD_SIZE", "1"))
local_rank = int(os.environ.get("LOCAL_RANK", "0"))
if not torch.cuda.is_available():
    raise SystemExit("denoise_parts_cost.py needs a CUDA device")
# more ranks than GPUs share them round-robin: the stage's stores then stay in one GPU's HBM instead of crossing NVLink
n_devices = min(world, torch.cuda.device_count())
device = local_rank % torch.cuda.device_count()
torch.cuda.set_device(device)
dev = torch.device("cuda", device)
dist = None
if world > 1:
    import torch.distributed as dist
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    if n_devices == world:
        dist.init_process_group("nccl", device_id=dev)
    else:
        dist.init_process_group("gloo")               # NCCL takes one rank per GPU


def barrier():
    """Host-side: returns when every rank got here (the ranks' stats() calls have waited for their stages)."""
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()


def max_over_ranks(values):
    t = torch.tensor(values, dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return t.cpu().numpy()


def summary(v):
    v = np.asarray(v)
    return round(float(np.median(v)), 3), [round(float(v.min()), 3), round(float(v.max()), 3)]


q = "name,power.limit,clocks.sm,clocks.max.sm"
gpu = subprocess.run(["nvidia-smi", "-i", str(device), f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
ctx = abi.Context(device)
for name in cli.configs.split(","):
    c = fs.CONFIGS[name]
    w, h = c["w"], c["h"]
    scene, cam = c["scene"](w, h)
    ctx.upload(scene)
    part = dict(tile_rows=TILE_ROWS, part_index=rank, part_count=world)
    render, aovs = fs.params_for(c, **part), fs.params_for(c, spp=AOV_SPP, **part)
    shared = distributed.SharedFrame(ctx, dist, abi.denoise_stage_words(w, h), rank, world, dev)
    if not shared.ok:
        raise SystemExit(f"rank {rank}: the stage could not be shared: {shared.error}")
    render_ms, stage_ms, staged_ms = [], [], []
    for rep in range(cli.reps + 1):                  # rep 0 is the warm-up (module load, buffers)
        ctx.render(cam, render)
        if rep:
            render_ms.append(ctx.stats().device_ms)
    ctx.render_path_aovs(cam, aovs)
    frame = rgb = None
    for rep in range(REPS_DN + 1):
        tag = 1000 * (rep + 1) + world
        ctx.denoise_stage(w, h, shared.ptr, tag, iterations=ITERATIONS)
        ms = ctx.stats().device_ms
        if rep:
            stage_ms.append(ms)
        barrier()
        if rank == 0:
            frame, rgb = ctx.denoise_staged(w, h, shared.ptr, tag, iterations=ITERATIONS)
            if rep:
                staged_ms.append(ctx.stats().device_ms)
        barrier()
    render_max, stage_max = max_over_ranks(render_ms), max_over_ranks(stage_ms)
    if rank == 0:
        ctx.render(cam, fs.params_for(c))
        ctx.render_path_aovs(cam, fs.params_for(c, spp=AOV_SPP))
        ref_frame, ref_rgb = ctx.denoise(w, h, iterations=ITERATIONS)
        n = w * h
        rows0 = ctx.lib.rt3_partition_rows(h, TILE_ROWS, 0, world)
        rec = {"config": name, "what": c["what"], "w": w, "h": h, "ranks": world, "gpus": n_devices, "tile_rows": TILE_ROWS, "render_spp": c["spp"], "aov_spp": AOV_SPP,
               "iterations": ITERATIONS, "reps": cli.reps, "denoise_reps": REPS_DN, "gpu": gpu}
        rec["render_ms_median"], rec["render_ms_min_max"] = summary(render_max)
        rec["stage_ms_median"], rec["stage_ms_min_max"] = summary(stage_max)
        rec["staged_filter_ms_median"], rec["staged_filter_ms_min_max"] = summary(staged_ms)
        rec["stage_plus_filter_ms"] = round(rec["stage_ms_median"] + rec["staged_filter_ms_median"], 3)
        rec["denoise_over_render"] = round(rec["stage_plus_filter_ms"] / rec["render_ms_median"], 4)
        rec["stage_bytes"] = 44 * n + 8 * h
        rec["stage_bytes_from_other_ranks"] = (44 * w + 8) * (h - rows0)
        rec["frame_equals_one_gpu_denoise"] = bool(np.array_equal(frame, ref_frame))
        rec["rgb_equals_one_gpu_denoise"] = bool(np.array_equal(rgb.view(np.uint32), ref_rgb.view(np.uint32)))
        print(json.dumps(rec), flush=True)
        os.makedirs(os.path.dirname(cli.out) or ".", exist_ok=True)
        with open(cli.out, "a") as f:
            f.write(json.dumps(rec) + "\n")
    barrier()
    shared.close()
ctx.close()
if world > 1:
    dist.destroy_process_group()
