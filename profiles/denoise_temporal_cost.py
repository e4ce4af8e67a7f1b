"""Cost of the temporal denoiser (rt3_denoise_temporal, DESIGN.md 3.9) next to rt3_denoise on the same frame.

For C2, C3 (through the hierarchy) and C4 at 5 iterations: one render and AOV call (4 samples each: the denoisers' cost does
not depend on the sample count), a warm-up of both calls, then REPS rounds of REPS_DN rt3_denoise calls followed by REPS_DN
rt3_denoise_temporal calls on an unchanged camera (every pixel has history), each timed by the library's CUDA events
(rt3_stats.device_ms: every kernel of the call on its stream, without the copies to the host). Medians and ranges, plus the
bytes the temporal kernel must move per pixel, computed from the shape. One JSON line per case, to stdout and to the file
given (default denoise_temporal_cost.jsonl in the working directory), with the GPU's name, power limit and SM clocks read by
an nvidia-smi query in the same run.
Usage: python profiles/denoise_temporal_cost.py [out.jsonl] [--reps N]"""
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
ap.add_argument("out", nargs="?", default="denoise_temporal_cost.jsonl")
ap.add_argument("--reps", type=int, default=5)
cli = ap.parse_args()
out_path, reps = cli.out, cli.reps
REPS_DN = 20
ITERATIONS = 5

q = "name,power.limit,clocks.sm,clocks.max.sm"
gpu = subprocess.run(["nvidia-smi", "-i", "0", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()

# denoise_temporal_kernel per pixel: the accumulators (24 B), albedo, normal (12 B each) and depth (4 B); up to 4 history taps of
# colour + length, moments and guide (40 B each; neighbours share them through L1 / L2); the next history (40 B), the accumulated
# colour and the guide (16 B each). The variance kernel then reads colour and guide, length and moments, and writes colour.
TEMPORAL_BYTES = (24 + 12 + 12 + 4) + 4 * 40 + 40 + 16 + 16
TEMPORAL_VARIANCE_BYTES = 16 + 16 + 16 + 8 + 16

CASES = [("c2", 0), ("c3", abi.FLAG_BVH), ("c4", 0)]
ctx = abi.Context(0)
os.makedirs(os.path.dirname(out_path) or ".", exist_ok=True)
with open(out_path, "w") as f:
    for name, flags in CASES:
        c = fs.CONFIGS[name]
        scene, cam = c["scene"](c["w"], c["h"])
        ctx.upload(scene)
        w, h = c["w"], c["h"]
        ctx.render(cam, fs.params_for(c, flags, spp=4))
        ctx.render_path_aovs(cam, fs.params_for(c, flags, spp=4))
        ctx.denoise(w, h, iterations=ITERATIONS)
        ctx.denoise_temporal(w, h, reset=True, iterations=ITERATIONS)
        times = {"denoise": [], "temporal": []}
        for rep in range(reps):
            for _ in range(REPS_DN):
                ctx.denoise(w, h, iterations=ITERATIONS)
                times["denoise"].append(ctx.stats().device_ms)
            for _ in range(REPS_DN):
                _, _, length = ctx.denoise_temporal(w, h, iterations=ITERATIONS)
                times["temporal"].append(ctx.stats().device_ms)
        rec = {"config": name, "what": c["what"], "w": w, "h": h, "iterations": ITERATIONS, "path": "bvh" if flags & abi.FLAG_BVH else "sweep",
               "reps": reps * REPS_DN, "history_length_min": float(length.min()), "gpu": gpu}
        for k, v in times.items():
            v = np.array(v)
            rec[k + "_ms_median"] = round(float(np.median(v)), 3)
            rec[k + "_ms_min_max"] = [round(float(v.min()), 3), round(float(v.max()), 3)]
        rec["temporal_over_denoise"] = round(rec["temporal_ms_median"] / rec["denoise_ms_median"], 4)
        rec["temporal_kernel_bytes_per_pixel"] = TEMPORAL_BYTES
        rec["temporal_variance_bytes_per_pixel"] = TEMPORAL_VARIANCE_BYTES
        print(json.dumps(rec), flush=True)
        f.write(json.dumps(rec) + "\n")
ctx.close()
