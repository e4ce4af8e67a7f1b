"""Cost of the path-traced AOV pass (rt3_render_path_aovs, DESIGN.md 3.7) against the render of the same configuration.

For C2 (16 and 500 AOV samples, sweep), C3 through the hierarchy (16 and 256) and C5 (64, hierarchy): after a warm-up of
both calls, REPS alternating repetitions of the render (the configuration's spp and depth) and of the AOV call, each timed
by the library's CUDA events (rt3_stats.device_ms: every kernel and memset of the call on its stream; trace_kernel_ms: the
trace kernel alone). One JSON line per case, written to stdout and to the file given (default aov_cost.jsonl in the working directory), with
the GPU's name, power limit and SM clocks read by an nvidia-smi query.
Usage: python profiles/aov_cost.py [out.jsonl] [--reps N]"""
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
ap.add_argument("out", nargs="?", default="aov_cost.jsonl")
ap.add_argument("--reps", type=int, default=5)
cli = ap.parse_args()
out_path, reps = cli.out, cli.reps

q = "name,power.limit,clocks.sm,clocks.max.sm"
gpu = subprocess.run(["nvidia-smi", "-i", "0", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()

# (config, AOV samples, flags)
CASES = [("c2", 16, 0), ("c2", 500, 0), ("c3", 16, abi.FLAG_BVH), ("c3", 256, abi.FLAG_BVH), ("c5", 64, abi.FLAG_BVH)]
ctx = abi.Context(0)
os.makedirs(os.path.dirname(out_path) or ".", exist_ok=True)
loaded = None
with open(out_path, "w") as f:
    for name, aov_spp, flags in CASES:
        c = fs.CONFIGS[name]
        if loaded != name:
            scene, cam = c["scene"](c["w"], c["h"])
            ctx.upload(scene)
            loaded = name
        render = fs.params_for(c, flags)
        aovs = fs.params_for(c, flags, spp=aov_spp)
        times = {"render": [], "aov": []}
        for rep in range(reps + 1):                     # rep 0 is the warm-up (module load, hierarchy build)
            for what, p in (("render", render), ("aov", aovs)):
                if what == "render":
                    ctx.render(cam, p)
                else:
                    ctx.render_path_aovs(cam, p)
                st = ctx.stats()
                if rep:
                    times[what].append((st.device_ms, st.trace_kernel_ms, st.rays))
        rec = {"config": name, "what": c["what"], "w": c["w"], "h": c["h"], "render_spp": c["spp"], "aov_spp": aov_spp,
               "path": "bvh" if flags & abi.FLAG_BVH else "sweep", "reps": reps, "gpu": gpu}
        for what in times:
            dev = np.array([t[0] for t in times[what]])
            rec[what + "_device_ms_median"] = round(float(np.median(dev)), 3)
            rec[what + "_device_ms_min_max"] = [round(float(dev.min()), 3), round(float(dev.max()), 3)]
            rec[what + "_kernel_ms_median"] = round(float(np.median([t[1] for t in times[what]])), 3)
            rec[what + "_rays"] = int(times[what][-1][2])
        rec["aov_over_render"] = round(rec["aov_device_ms_median"] / rec["render_device_ms_median"], 4)
        rec["aov_mrays_s"] = round(rec["aov_rays"] / rec["aov_kernel_ms_median"] / 1e3, 1)
        print(json.dumps(rec), flush=True)
        f.write(json.dumps(rec) + "\n")
ctx.close()
