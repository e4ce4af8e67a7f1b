"""Cost of the denoiser (rt3_denoise, DESIGN.md 3.8) next to the render and the 16-sample AOV call of the same configuration.

For C2, C3 (through the hierarchy) and C4 at 5 iterations: after a warm-up of every call, REPS alternating repetitions of
the render (the configuration's spp and depth), the AOV call (16 samples) and REPS_DN denoise calls, each timed by the
library's CUDA events (rt3_stats.device_ms: every kernel of the call on its stream, without the copy to the host). Each line
also gives the bytes the kernels must move, computed from the shape (every pixel's input read once and its output written
once per kernel; the 5x5 taps of a pass are assumed to come from L1 / L2), the time those bytes take at the HBM3e data-sheet
rate of 7.7 TB/s, the achieved fraction of that bound, and the working set of the passes (two ping-pong colour buffers and the
guides, 48 bytes per pixel) against the 126 MB L2. One JSON line per case, to stdout and to the file given (default
denoise_cost.jsonl in the working directory), with the GPU's name, power limit and SM clocks read by an nvidia-smi query.
Usage: python profiles/denoise_cost.py [out.jsonl] [--reps N]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import rt3_b200  # noqa: F401,E402
from rt3_b200 import abi  # noqa: E402
import fullsize as fs  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("out", nargs="?", default="denoise_cost.jsonl")
ap.add_argument("--reps", type=int, default=5)
cli = ap.parse_args()
out_path, reps = cli.out, cli.reps
REPS_DN = 20
ITERATIONS = 5
HBM_BYTES_S = 7.7e12
L2_BYTES = 126e6

q = "name,power.limit,clocks.sm,clocks.max.sm"
gpu = subprocess.run(["nvidia-smi", "-i", "0", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()


def bytes_moved(n_pixels, iterations):
    """Per pixel: prepare reads 3 u64 accumulators, albedo, normal (3 floats each) and depth, writes colour and guide (float4 each);
    the variance kernel and each pass read colour and guide and write colour; the last pass also reads the albedo and writes the
    packed pixel and the linear rgb."""
    prepare = 24 + 12 + 12 + 4 + 16 + 16
    variance = 16 + 16 + 16
    middle = (iterations - 1) * (16 + 16 + 16)
    last = 16 + 16 + 12 + 4 + 12
    return n_pixels * (prepare + variance + middle + last)


CASES = [("c2", 0), ("c3", abi.FLAG_BVH), ("c4", 0)]
ctx = abi.Context(0)
os.makedirs(os.path.dirname(out_path) or ".", exist_ok=True)
with open(out_path, "w") as f:
    for name, flags in CASES:
        c = fs.CONFIGS[name]
        scene, cam = c["scene"](c["w"], c["h"])
        ctx.upload(scene)
        w, h = c["w"], c["h"]
        render, aovs = fs.params_for(c, flags), fs.params_for(c, flags, spp=16)
        times = {"render": [], "aov": [], "denoise": [], "denoise_kernels": []}
        for rep in range(reps + 1):                     # rep 0 is the warm-up (module load, hierarchy build, buffers)
            ctx.render(cam, render)
            if rep:
                times["render"].append(ctx.stats().device_ms)
            ctx.render_path_aovs(cam, aovs)
            if rep:
                times["aov"].append(ctx.stats().device_ms)
            for _ in range(REPS_DN if rep else 2):
                ctx.denoise(w, h, iterations=ITERATIONS)
                st = ctx.stats()
                if rep:
                    times["denoise"].append(st.device_ms)
                    times["denoise_kernels"].append(st.trace_kernel_ms)
        n = w * h
        moved = bytes_moved(n, ITERATIONS)
        rec = {"config": name, "what": c["what"], "w": w, "h": h, "render_spp": c["spp"], "aov_spp": 16, "iterations": ITERATIONS,
               "path": "bvh" if flags & abi.FLAG_BVH else "sweep", "reps": reps, "denoise_reps": reps * REPS_DN, "gpu": gpu}
        for k, v in times.items():
            v = np.array(v)
            rec[k + "_ms_median"] = round(float(np.median(v)), 3)
            rec[k + "_ms_min_max"] = [round(float(v.min()), 3), round(float(v.max()), 3)]
        rec["denoise_over_render"] = round(rec["denoise_ms_median"] / rec["render_ms_median"], 4)
        rec["bytes_moved"] = moved
        rec["working_set_bytes"] = 48 * n
        rec["working_set_fits_l2"] = 48 * n < L2_BYTES
        rec["hbm_bound_ms"] = round(moved / HBM_BYTES_S * 1e3, 4)
        rec["hbm_bound_fraction"] = round(rec["hbm_bound_ms"] / rec["denoise_ms_median"], 4)
        rec["achieved_gb_s"] = round(moved / (rec["denoise_ms_median"] * 1e-3) / 1e9, 1)
        rec["mpixel_passes_s"] = round(n * ITERATIONS / (rec["denoise_ms_median"] * 1e-3) / 1e6, 1)
        print(json.dumps(rec), flush=True)
        f.write(json.dumps(rec) + "\n")
ctx.close()
