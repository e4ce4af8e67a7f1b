"""Cost of temporal accumulation for a frame rendered in parts (rt3_denoise_staged_temporal, DESIGN.md 3.10) next to
rt3_denoise_staged on the same stage, one process per GPU.

    torchrun --nproc_per_node N profiles/denoise_parts_temporal_cost.py [out.jsonl] [--reps R] [--configs c2,c4]

For each configuration (4 samples and 4 AOV samples per pixel: the filters' cost does not depend on the sample count; 5
iterations; rows dealt one by one as bench.py deals them): every rank renders its rows and their AOVs and stages them into
rank 0's stage (distributed.SharedFrame over CUDA IPC; ranks beyond the GPU count share GPUs round-robin, and the line
records both counts). Rank 0 then calls rt3_denoise_staged_temporal WARM times on the unchanged camera, so that every
pixel's history holds WARM frames or more, and times R rounds of REPS_DN rt3_denoise_staged calls followed by REPS_DN
rt3_denoise_staged_temporal calls, each by the library's CUDA events (rt3_stats.device_ms: every kernel of the call on its
stream, without the copies to the host). Then rank 0 renders the whole frame alone, runs rt3_denoise_temporal as many
times (the first with reset), timing those calls too, and records whether the last one equals the last staged call's
frame, linear rgb and history length bit for bit. One JSON line per case is printed by rank 0 and appended to the file
(default denoise_parts_temporal_cost.jsonl in the working directory), with the GPU's name, power limit and clocks from
an nvidia-smi query in the same run."""
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
ap.add_argument("out", nargs="?", default="denoise_parts_temporal_cost.jsonl")
ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--configs", default="c2,c4")
cli = ap.parse_args()
REPS_DN = 20
WARM = 8
ITERATIONS = 5
SPP = 4
TILE_ROWS = 1
TAG = 77

rank = int(os.environ.get("RANK", "0"))
world = int(os.environ.get("WORLD_SIZE", "1"))
local_rank = int(os.environ.get("LOCAL_RANK", "0"))
if not torch.cuda.is_available():
    raise SystemExit("denoise_parts_temporal_cost.py needs a CUDA device")
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


def summary(v):
    v = np.asarray(v)
    return round(float(np.median(v)), 3), [round(float(v.min()), 3), round(float(v.max()), 3)]


def same(a, b):
    return all(np.array_equal(x.view(np.uint32), y.view(np.uint32)) for x, y in zip(a, b))


q = "name,power.limit,clocks.sm,clocks.max.sm"
gpu = subprocess.run(["nvidia-smi", "-i", str(device), f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
ctx = abi.Context(device)
for name in cli.configs.split(","):
    c = fs.CONFIGS[name]
    w, h = c["w"], c["h"]
    scene, cam = c["scene"](w, h)
    ctx.upload(scene)
    part = dict(tile_rows=TILE_ROWS, part_index=rank, part_count=world)
    shared = distributed.SharedFrame(ctx, dist, abi.denoise_stage_words(w, h), rank, world, dev)
    if not shared.ok:
        raise SystemExit(f"rank {rank}: the stage could not be shared: {shared.error}")
    ctx.render(cam, fs.params_for(c, spp=SPP, **part))
    ctx.render_path_aovs(cam, fs.params_for(c, spp=SPP, **part))
    ctx.denoise_stage(w, h, shared.ptr, TAG, iterations=ITERATIONS)
    ctx.stats()
    barrier()
    if rank == 0:
        calls = 0
        for i in range(WARM):                         # module load, buffers, and a history of WARM frames everywhere
            staged_temporal = ctx.denoise_staged_temporal(w, h, shared.ptr, TAG, reset=i == 0, iterations=ITERATIONS)
            calls += 1
        ctx.denoise_staged(w, h, shared.ptr, TAG, iterations=ITERATIONS)
        times = {"staged": [], "staged_temporal": []}
        for rep in range(cli.reps):
            for _ in range(REPS_DN):
                ctx.denoise_staged(w, h, shared.ptr, TAG, iterations=ITERATIONS)
                times["staged"].append(ctx.stats().device_ms)
            for _ in range(REPS_DN):
                staged_temporal = ctx.denoise_staged_temporal(w, h, shared.ptr, TAG, iterations=ITERATIONS)
                calls += 1
                times["staged_temporal"].append(ctx.stats().device_ms)
        # the same number of calls on a one-context render of the same frame
        ctx.render(cam, fs.params_for(c, spp=SPP))
        ctx.render_path_aovs(cam, fs.params_for(c, spp=SPP))
        times["one_context_temporal"] = []
        for i in range(calls):
            one = ctx.denoise_temporal(w, h, reset=i == 0, iterations=ITERATIONS)
            if i >= WARM:
                times["one_context_temporal"].append(ctx.stats().device_ms)
        rec = {"config": name, "what": c["what"], "w": w, "h": h, "ranks": world, "gpus": n_devices, "tile_rows": TILE_ROWS, "spp": SPP, "aov_spp": SPP,
               "iterations": ITERATIONS, "reps": cli.reps * REPS_DN, "history_length_min": float(staged_temporal[2].min()), "gpu": gpu}
        for k, v in times.items():
            rec[k + "_ms_median"], rec[k + "_ms_min_max"] = summary(v)
        rec["staged_temporal_over_staged"] = round(rec["staged_temporal_ms_median"] / rec["staged_ms_median"], 4)
        rec["staged_temporal_over_one_context_temporal"] = round(rec["staged_temporal_ms_median"] / rec["one_context_temporal_ms_median"], 4)
        rec["equals_one_context_temporal"] = same(staged_temporal, one)
        print(json.dumps(rec), flush=True)
        os.makedirs(os.path.dirname(cli.out) or ".", exist_ok=True)
        with open(cli.out, "a") as f:
            f.write(json.dumps(rec) + "\n")
    barrier()
    shared.close()
ctx.close()
if world > 1:
    dist.destroy_process_group()
