#!/usr/bin/env python
"""bench.py — Mrays/s of the per-pixel render path on N B200s (one process per GPU).

Workload (BASELINE.json configs[1]): RTIOW book-1 cover scene (~484 analytic
spheres, mixed materials, thin lens), 1200x800, 500 spp, depth 50. One "step" is
one full frame: camera in, packed uint32 framebuffer out.

  value : device-timed (CUDA events on the render stream) whole-job Mrays/s with
          the scene and frame resident in HBM; rays = ray segments the kernel counted.
  e2e   : the same frame through the reference-facing C-ABI call rt3_render() with a
          HOST frame buffer (N=1), or device render + NCCL gather + D2H into pinned
          host memory on rank 0 (N>1); host<->device copies inside the timed region.
  --impl reference : the CPU implementation of the same path (the oracle port of the
          RTIOW semantics -- the reference itself has no bounce loop) on all host threads.

N>1: the frame's row tiles are dealt round-robin to the ranks (no data-path collective
while rendering); the packed framebuffer is gathered with NCCL at frame end. The frame
is fixed, so scaling is strong.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

W, H, SPP, DEPTH, SEED, TILE_ROWS = 1200, 800, 500, 50, 1, 1   # rows dealt one by one: halves the systematic cost offset between ranks
FLOP_PER_SPHERE_TEST, FLOP_PER_FACE_TEST = 17, 45  # SURVEY.md section 8d
CPU_SAMPLE = dict(width=480, height=320, spp=48)    # bounded sample of the same workload for the CPU legs (~20 M ray segments)
NOMINAL_FP32_TFLOPS = 148 * 128 * 2 * 1.965e9 / 1e12
NCU_COUNTERS = os.path.join(ROOT, "profiles", "ncu_counters.json")  # written by profiles/ncu_counters.py from an ncu capture of this command
DUMP_BYTES = 64_000_000   # most a --dump-outputs directory may hold: larger frames are dumped as a fixed sample of their rows


def dump_frame(out_dir, frame):
    """--dump-outputs: the packed frame [H, W] (r<<24 | g<<16 | b<<8 | a) as DIR/frame.npy, [H, W, 4] float32 channel levels 0..255
    (float32 holds each 8-bit level exactly). A frame above DUMP_BYTES keeps the rows of a fixed seeded sample, in order, and their
    indices go to DIR/frame_rows.npy (float64)."""
    import numpy as np
    frame = np.asarray(frame).view(np.uint32)
    levels = np.stack([(frame >> s) & 0xFF for s in (24, 16, 8, 0)], -1).astype(np.float32)
    os.makedirs(out_dir, exist_ok=True)
    if levels.nbytes > DUMP_BYTES:
        n_rows = (DUMP_BYTES - 4096) // (levels[0].nbytes + 8)   # 4096: room for the two .npy headers
        rows = np.sort(np.random.default_rng(0).choice(len(levels), n_rows, replace=False))
        levels = levels[rows]
        np.save(os.path.join(out_dir, "frame_rows.npy"), rows.astype(np.float64))
    np.save(os.path.join(out_dir, "frame.npy"), levels)


def profiled_counters(kernel, width, height, spp, depth, n_prims, world):
    """Per-launch ncu counters of the dominant kernel for EXACTLY this workload (same kernel, frame, spp, depth, scene size,
    GPU count), or (None, why). The file is committed with the ncu capture it was extracted from (profiles/ncu_counters.py)."""
    try:
        table = json.load(open(NCU_COUNTERS))
    except Exception as e:
        return None, f"{os.path.relpath(NCU_COUNTERS, ROOT)} unreadable ({e})"
    for row in table.get("captures", []):
        w = row.get("workload", {})
        if (row.get("kernel") == kernel and w.get("width") == width and w.get("height") == height and w.get("spp") == spp and
                w.get("max_depth") == depth and w.get("n_prims") == n_prims and w.get("n_gpus", 1) == world):
            return row, row.get("source", os.path.relpath(NCU_COUNTERS, ROOT))
    return None, f"no ncu capture of {kernel} at {width}x{height}, {spp} spp, depth {depth}, {n_prims} primitives, {world} GPU(s) in {os.path.relpath(NCU_COUNTERS, ROOT)}"


def hbm_line(kernel_ms, traffic_bytes):
    """Achieved DRAM bandwidth of the dominant kernel (ncu traffic / event time) against the measured copy bandwidth."""
    peak, src = 6650.0, "built-in fallback: no MEASURED_PEAKS.json"
    try:
        peak, src = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]), "MEASURED_PEAKS.json"
    except Exception:
        pass
    achieved = traffic_bytes / (kernel_ms * 1e-3) / 1e9 if kernel_ms > 0 else 0.0
    return {"achieved_gbs": achieved, "peak_gbs": peak, "frac": achieved / peak, "peak_source": src}


def workload_config():
    which = "configs[1]" if (W, H, SPP) == (1200, 800, 500) else "configs[3]: not the configuration the metric is quoted on"
    return {"workload": f"RTIOW book-1 cover scene, {W}x{H}, {SPP} spp, depth {DEPTH} (BASELINE {which})",
            "width": W, "height": H, "spp": SPP, "max_depth": DEPTH, "tile_rows": TILE_ROWS,
            "l2": "256 MiB buffer written between timed steps (L2 flush); scene+accumulators re-read from HBM"}


def cpu_arm_config():
    """The GPU arm's workload, with the bounded sample the CPU arm really renders spelled out: the rate (Mrays/s) is of that
    sample -- same scene, camera, depth and sampling, fewer pixels and samples per pixel -- not of a full 1200x800x500 frame."""
    cfg = workload_config()
    cfg["workload"] += (f" -- CPU arm times a bounded sample of it: {CPU_SAMPLE['width']}x{CPU_SAMPLE['height']}, {CPU_SAMPLE['spp']} spp per step "
                        "(same scene, camera, depth); Mrays/s is a rate, nothing is extrapolated")
    cfg["timed_sample"] = dict(CPU_SAMPLE, max_depth=DEPTH)
    cfg.pop("l2", None)
    return cfg


class ClockSampler:
    """Samples SM clocks / throttle reasons during the timed region (nvidia-smi, 200 ms)."""

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        rows = [r for r in self.rows if len(r) >= 7 and r[0].isdigit()]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm = sorted(int(r[0]) for r in rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[3 + i] == "Active" for r in rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": int(rows[0][1]), "reasons": reasons, "samples": len(rows),
                "power_w_max": max(float(r[2]) for r in rows)}


def usable_cores():
    """Host cores this process may actually use: the affinity mask, capped by the cgroup CPU quota when there is one."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            fields = open(path).read().split()
            if path.endswith("cpu.max"):
                quota, period = fields[0], float(fields[1])
            else:
                quota, period = fields[0], float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if quota not in ("max", "-1") and period > 0:
                n = max(1, min(n, int(float(quota) / period + 0.5)))
            break
        except (OSError, ValueError, IndexError):
            continue
    return n


def cpu_port_rate(n_threads, steps=1, warmup=0):
    """Mrays/s of the oracle port on a bounded sample of the workload (all ray segments counted), seconds per step, a label
    of the sample, and the last step's packed frame."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import rt3_b200  # noqa: F401
    from rt3_b200 import abi, scenes
    import oraclelib
    w, h, spp = CPU_SAMPLE["width"], CPU_SAMPLE["height"], CPU_SAMPLE["spp"]
    scene, cam = scenes.rtiow_cover(w, h)
    params = abi.make_params(w, h, mode=abi.MODE_PATHTRACE, spp=spp, max_depth=DEPTH, seed=SEED)
    for _ in range(warmup):
        oraclelib.oracle_pathtrace(scene, cam, params, n_threads=n_threads)
    t0 = time.perf_counter()
    rays = 0
    frame = None
    for _ in range(steps):
        frame, _, r = oraclelib.oracle_pathtrace(scene, cam, params, n_threads=n_threads)
        rays += r
    dt = time.perf_counter() - t0
    sample = f"same scene and camera at {w}x{h}, {spp} spp, depth {DEPTH}: {rays // max(steps, 1)} ray segments per step"
    return rays / dt / 1e6, dt / max(steps, 1), sample, frame


def reference_native_rate():
    """The compiled reference's own render loop (oracle/_ref) on its default-scene shape: 1 core, 1 spp, depth 1."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    try:
        import oraclelib
        if not oraclelib.have_ref() or not os.path.exists(oraclelib.REF_TEDDY):
            return None
        rs = oraclelib.RefScene()
        rs.add_object(oraclelib.REF_TEDDY, (0, 0, -3), 1.0 / 17.0, (1, 0, 0))
        rs.add_sphere((-2, 0, -5), 1.0, 8, 8, (0, 0, 1))
        rs.prerender()
        w, h = 200, 113
        _, sec = rs.render(w, h)
        return {"kind": "reference", "what": f"reference SequentialRenderer::render, Main.cpp default scene (3288 faces), {w}x{h}, 1 spp, depth 1",
                "cores": 1, "value": w * (h - 1) / sec / 1e6, "unit": "Mrays/s", "seconds": round(sec, 3)}
    except Exception as e:  # the reference leg is informative only
        return {"kind": "reference", "error": str(e)}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n_threads = usable_cores()
    rate, sec_per_step, sample, frame = cpu_port_rate(n_threads, steps=args.steps, warmup=min(args.warmup, 1))
    if args.dump_outputs:
        dump_frame(args.dump_outputs, frame)
    line = {
        "impl": "reference", "metric": "Mrays/s", "value": rate, "unit": "Mrays/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": min(args.warmup, 1), "ms_per_step": sec_per_step * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cpu_arm_config(),
        "cpu_baseline": {"value": rate, "unit": "Mrays/s", "cores": n_threads, "kind": "port", "sample": sample,
                         "note": "the reference has no bounce loop/materials (raytracer_v4.glsl:279); this is the CPU restatement of the same path"},
        "e2e": {"value": rate, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "reference_native": reference_native_rate(),
    }
    print(json.dumps(line), flush=True)


def positive_int(text):
    n = int(text)
    if n < 1:
        raise argparse.ArgumentTypeError(f"must be at least 1, got {n}")
    return n


def main():
    global W, H, SPP
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=positive_int, default=3, help="timed steps (at least 1)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="rt3", choices=["rt3", "reference"])
    ap.add_argument("--spp", type=int, default=SPP, help="override samples per pixel (non-default values are not the BASELINE config)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-c4", action="store_true", help="skip the extra C4 leg (3840x2160, 1024 spp) after the timed C2 region")
    ap.add_argument("--config", default="c2", choices=["c2", "c4"],
                    help="c2 (default, the metric's configuration) or c4: the same scene at 3840x2160, 1024 spp (BASELINE configs[3], the multi-GPU one)")
    ap.add_argument("--gather", choices=("peer", "nccl"), default="peer",
                    help="N>1 frame end: 'peer' = every rank's kernels store their rows into rank 0's frame over NVLink (CUDA IPC mapping) "
                         "and the frame ends with a one-element all-reduce; 'nccl' = pack + NCCL gather + de-interleave")
    ap.add_argument("--bvh", action="store_true", help="time the hierarchy path (RT3_FLAG_BVH) instead of the brute-force sweep: not the headline configuration")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the frame of the last one to DIR/frame.npy ([H, W, 4] float32 r, g, b, a levels; see dump_frame) "
                         "so that two builds can be compared output for output on the same seeded inputs")
    args = ap.parse_args()
    if args.config == "c4":
        W, H, SPP = 3840, 2160, 1024
        if args.spp == 500:
            args.spp = SPP
    if args.impl == "reference":
        run_reference_arm(args)
        return
    # stdout carries exactly one JSON line: whatever libraries print there while we run (NCCL's version banner) goes to stderr
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    import numpy as np
    import torch
    import rt3_b200  # noqa: F401
    from rt3_b200 import abi, distributed, scenes

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the render core has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    spp = args.spp
    stream = torch.cuda.Stream(device=dev)  # a real (non-NULL) stream: kernels, NCCL and the timing events all go here
    torch.cuda.set_stream(stream)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    ctx = abi.Context(local_rank)
    lib = ctx.lib
    launches_per_step = 3  # clear_accum + pathtrace + resolve

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    class Job:
        """One frame configuration (the cover scene at w x h, n spp) split over the ranks: buffers, the per-frame device step,
        and the check of the assembled frame against rank 0 rendering every row itself."""

        def __init__(self, w, h, n_spp, gather):
            self.w, self.h, self.spp = w, h, n_spp
            self.scene, self.cam = scenes.rtiow_cover(w, h)
            self.flags = abi.FLAG_BVH if args.bvh else 0
            self.params = abi.make_params(w, h, mode=abi.MODE_PATHTRACE, spp=n_spp, max_depth=DEPTH, seed=SEED, flags=self.flags,
                                          tile_rows=TILE_ROWS, part_index=rank, part_count=world)
            self.peer = world > 1 and gather == "peer"
            self.shared = distributed.SharedFrame(ctx, dist, h * w, rank, world, dev) if self.peer else None
            if self.shared and not self.shared.ok:   # agreed on by all ranks: no mapping somewhere -> plain NCCL gather everywhere
                print(f"[bench] rank {rank}: shared frame unavailable ({self.shared.error}); gathering with NCCL", file=sys.stderr)
                self.shared.close()
                self.shared, self.peer = None, False
            self.frame = self.shared.tensor if (self.peer and rank == 0) else torch.zeros(h * w, dtype=torch.int32, device=dev)
            self.frame_ptr = self.shared.ptr if self.peer else self.frame.data_ptr()
            max_rows = max(lib.rt3_partition_rows(h, TILE_ROWS, r, world) for r in range(world))
            self.slab = torch.zeros(max_rows * w, dtype=torch.int32, device=dev) if (world > 1 and not self.peer) else None

        def device_step(self):
            """Render this rank's rows. N>1, peer: the rows land in rank 0's frame as they are resolved, the frame ends with a
            stream-ordered one-element all-reduce. N>1, nccl: pack, gather onto rank 0 (NCCL), de-interleave."""
            ctx.render_device(self.cam, self.params, self.frame_ptr, stream.cuda_stream)
            if self.peer:
                self.shared.finish()
            elif world > 1:
                ctx.pack_partition(self.frame.data_ptr(), self.slab.data_ptr(), self.w, self.h, TILE_ROWS, rank, world, stream.cuda_stream)
                gathered = distributed.gather_slabs(dist, self.slab, rank, world)  # NCCL, frame end only
                if rank == 0:
                    for r in range(1, world):
                        ctx.unpack_partition(gathered[r].data_ptr(), self.frame.data_ptr(), self.w, self.h, TILE_ROWS, r, world, stream.cuda_stream)

        def timed(self, steps, warmup):
            """(max-over-ranks total ms of `steps` device-timed frames, whole-job ray segments per frame, last step's stats)."""
            for _ in range(max(warmup, 0)):
                flush.fill_(1)
                self.device_step()
            sync_all()
            rays_step = torch.tensor([ctx.stats().rays], dtype=torch.int64, device=dev)
            if world > 1:
                dist.all_reduce(rays_step)
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
            sync_all()
            for k in range(steps):
                flush.fill_(k)  # L2 flush, outside the per-step events
                ev[k][0].record(stream)
                self.device_step()
                ev[k][1].record(stream)
            sync_all()
            total = torch.tensor([sum(a.elapsed_time(b) for a, b in ev)], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(total, op=dist.ReduceOp.MAX)
            return float(total.item()), int(rays_step.item()), ctx.stats()  # rays: deterministic, identical every step

        def frame_matches_single_gpu(self):
            """N>1: the assembled frame must be the one-GPU frame, bit for bit (untimed; rank 0 renders every row itself)."""
            if world == 1:
                return None
            self.device_step()
            sync_all()
            ok = True
            if rank == 0:
                whole = torch.zeros(self.h * self.w, dtype=torch.int32, device=dev)
                one = abi.make_params(self.w, self.h, mode=abi.MODE_PATHTRACE, spp=self.spp, max_depth=DEPTH, seed=SEED, flags=self.flags, tile_rows=TILE_ROWS)
                ctx.render_device(self.cam, one, whole.data_ptr(), stream.cuda_stream)
                torch.cuda.synchronize()
                ok = bool(torch.equal(whole, self.frame))
            flag = torch.tensor([1 if ok else 0], dtype=torch.int32, device=dev)
            dist.broadcast(flag, src=0)
            if not int(flag.item()):
                raise SystemExit(f"the {self.w}x{self.h} frame assembled from {world} partitions differs from the one-GPU frame")
            sync_all()
            return True

        def close(self):
            if self.shared:
                torch.cuda.synchronize()
                self.frame = None
                self.shared.close()
                self.shared = None

    job = Job(W, H, spp, args.gather)
    scene, cam, params, peer = job.scene, job.cam, job.params, job.peer
    ctx.upload(scene)
    host_frame_t = torch.zeros(H * W, dtype=torch.int32).pin_memory()
    host_frame = host_frame_t.numpy().view(np.uint32).reshape(H, W)

    # ---- warm-up + timed: device-resident ----
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    total_ms, rays_per_step, st = job.timed(args.steps, args.warmup)   # st: last step's dominant-kernel time and counters (this rank)
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        dump_frame(args.dump_outputs, job.frame.cpu().numpy().reshape(H, W))   # before the legs below render into the same buffer

    # ---- timed: end to end with host buffers ----
    e2e_steps = args.steps
    if world == 1:
        ctx.render(cam, params, out=host_frame)  # untimed: first call allocates the context's own frame buffer
    sync_all()
    t0 = time.perf_counter()
    for s in range(e2e_steps):
        if world == 1:
            ctx.render(cam, params, out=host_frame)     # rt3_render: blocking, D2H into the pinned host frame
        else:
            job.device_step()
            if rank == 0:
                host_frame_t.copy_(job.frame, non_blocking=True)
            if peer:
                job.shared.finish()  # the other ranks' next frame may only overwrite the shared frame once rank 0 has read this one
            torch.cuda.synchronize()
    sync_all()
    e2e_s = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e_s = float(e2e_s.item())
    st_e2e = ctx.stats()

    frame_matches = job.frame_matches_single_gpu()

    # ---- informational: the same frame through the hierarchy (RT3_FLAG_BVH), device-timed, not part of `value` ----
    hierarchy = None
    if world == 1 and not args.bvh:
        bvh_params = abi.make_params(W, H, mode=abi.MODE_PATHTRACE, spp=spp, max_depth=DEPTH, seed=SEED, flags=abi.FLAG_BVH, tile_rows=TILE_ROWS)
        ctx.render_device(cam, bvh_params, job.frame.data_ptr(), stream.cuda_stream)   # builds the hierarchy, warms up
        torch.cuda.synchronize()
        flush.fill_(7)
        ctx.render_device(cam, bvh_params, job.frame.data_ptr(), stream.cuda_stream)
        torch.cuda.synchronize()
        sb = ctx.stats()
        hierarchy = {"value": sb.rays / (sb.device_ms * 1e-3) / 1e6, "unit": "Mrays/s", "ms_per_step": sb.device_ms, "build_ms": sb.accel_build_ms,
                     "node_visits_per_ray": sb.accel_node_visits / max(sb.rays, 1), "prim_tests_per_ray": sb.accel_prim_tests / max(sb.rays, 1),
                     "beam_rays": sb.beam_rays, "beam_tests_per_ray": sb.beam_tests / max(sb.beam_rays, 1),
                     "note": "same workload through the device-built BVH (identical frame; primary rays against the candidates of a beam's walk of the trees, "
                             "every other ray segment by traversal); informational, the metric is the brute-force sweep"}

    # ---- BASELINE configs[3] (C4: the same scene at 3840x2160, 1024 spp -- the configuration named for 2/4/8 GPUs), as an extra
    #      key of the same line: device-timed like `value`, same split and frame end, assembled frame checked (N>1) ----
    c4 = None
    if args.config == "c2" and spp == SPP and not args.no_c4:
        job.close()
        c4_job = Job(3840, 2160, 1024, args.gather)   # same scene arrays (the camera's aspect differs): no new upload needed, but keep it explicit
        ctx.upload(c4_job.scene)
        c4_steps = 2
        c4_ms, c4_rays, c4_st = c4_job.timed(c4_steps, 1)
        c4_match = c4_job.frame_matches_single_gpu()
        c4 = {"workload": "RTIOW book-1 cover scene, 3840x2160, 1024 spp, depth 50 (BASELINE configs[3])", "steps": c4_steps, "warmup": 1,
              "ms_per_step": c4_ms / c4_steps, "value": c4_rays * c4_steps / (c4_ms * 1e-3) / 1e6, "unit": "Mrays/s", "rays_per_step": c4_rays,
              "kernel_ms_rank0": c4_st.trace_kernel_ms, "frame_matches_single_gpu": c4_match, "n_gpus": world,
              "timing": "CUDA events around each frame incl. the frame end, max over ranks; L2 flushed between frames"}
        c4_job.close()
        job = None

    if rank == 0:
        ms_per_step = total_ms / args.steps
        value = rays_per_step * args.steps / (total_ms * 1e-3) / 1e6
        e2e_value = rays_per_step * e2e_steps / e2e_s / 1e6
        # roofline of the dominant kernel (pathtrace_kernel), this rank's launch
        flops = FLOP_PER_SPHERE_TEST * st.sphere_tests + FLOP_PER_FACE_TEST * st.face_tests
        achieved = flops / (st.trace_kernel_ms * 1e-3) / 1e12 if st.trace_kernel_ms > 0 else 0.0
        peak = ctx.measure_fma_peak()
        # executed (not credited) FP32 work and DRAM traffic: per-launch ncu counters of this exact workload, from the committed capture
        # (resident sphere scenes trace their primary rays against per-chunk candidate lists: the BEAM instantiation, template arguments <1,1,0,0,1>)
        kernel_name = "pathtrace_kernel<1,0,1>" if args.bvh else ("pathtrace_kernel<1,1,0,0,1>" if st.beam_rays else "pathtrace_kernel<1,1,0>")
        prof, prof_src = profiled_counters(kernel_name, W, H, spp, DEPTH, scene.n_spheres, world)
        share = 1.0
        if not prof and world > 1:
            # ncu is never run on a multi-rank command: take the one-GPU capture of the same frame and scale it by this rank's share of
            # the ray segments (the work per ray segment does not depend on which GPU traces it; the accumulators scale with the rows)
            prof, prof_src = profiled_counters(kernel_name, W, H, spp, DEPTH, scene.n_spheres, 1)
            if prof and prof.get("rays_per_launch"):
                share = st.rays / prof["rays_per_launch"]
                prof = dict(prof, **{k: prof[k] * share for k in ("ffma_thread_inst", "ffma2_thread_inst", "fmul_thread_inst", "fadd_thread_inst",
                                                                 "dram_bytes_read", "dram_bytes_write")})
                prof_src += f" (one-GPU capture scaled by rank 0's share of the ray segments, {share:.4f}: ncu does not run on multi-rank commands)"
            else:
                prof = None
        executed_tflops = executed_frac = traffic = hbm = None
        executed_note = prof_src
        if prof:
            # thread-level instruction counts: an FFMA is 2 FLOP, FMUL / FADD 1. ncu's op_ffma counter does not include the packed
            # FFMA2 (fma.rn.f32x2: two FMAs = 4 FLOP per thread instruction); its count comes from the per-opcode sums of the
            # source page of the same capture (profiles/ncu_counters.py) and is consistent with op_fp32
            fl = 2.0 * prof["ffma_thread_inst"] + 4.0 * prof.get("ffma2_thread_inst", 0) + prof["fmul_thread_inst"] + prof["fadd_thread_inst"]
            executed_tflops = fl / (st.trace_kernel_ms * 1e-3) / 1e12 if st.trace_kernel_ms > 0 else None
            executed_frac = executed_tflops / peak if (peak and executed_tflops is not None) else None
            traffic = prof["dram_bytes_read"] + prof["dram_bytes_write"]
            hbm = hbm_line(st.trace_kernel_ms, traffic)
            executed_note = (f"{prof_src}: smsp__sass_thread_inst_executed_op_ffma/fmul/fadd_pred_on.sum of one launch of this workload "
                             f"(FFMA {prof['ffma_thread_inst']:.4g} x 2 FLOP, packed FFMA2 {prof.get('ffma2_thread_inst', 0):.4g} x 4 FLOP from the source page; "
                             f"fmul {prof['fmul_thread_inst']:.4g}; fadd {prof['fadd_thread_inst']:.4g}) / this run's kernel time; "
                             f"pipe_fma_cycles_active {prof.get('pipe_fma_cycles_active_pct')} %, issue slots busy {prof.get('issue_active_pct')} %")
        line = {
            "metric": "Mrays/s", "value": value, "unit": "Mrays/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": workload_config(),
            "rays_per_step": rays_per_step, "spheres": scene.n_spheres,
            "clocks": clocks, "gpu_launches": launches_per_step * args.steps + (0 if (world == 1 or peer) else (1 + (world - 1)) * args.steps),
            "e2e": {"value": e2e_value, "unit": "Mrays/s", "h2d_bytes_per_step": ctypes.sizeof(abi.Camera) + ctypes.sizeof(abi.Params),
                    "d2h_bytes_per_step": W * H * 4, "ms_per_step": e2e_s / e2e_steps * 1e3,
                    "last_step_device_ms": st_e2e.device_ms, "last_step_d2h_ms": st_e2e.d2h_ms,
                    "path": "rt3_render (C ABI), pinned host frame" if world == 1 else
                            ("rt3_render_device into rank 0's frame over NVLink (rt3_frame_import) + all-reduce barrier + D2H on rank 0" if peer
                             else "rt3_render_device + NCCL gather + D2H on rank 0")},
            "roofline": {"bound": "fp32-issue", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak if peak else None,
                         "executed_tflops": executed_tflops, "executed_frac": executed_frac, "executed_source": executed_note,
                         "traffic": traffic,
                         "traffic_source": (f"dram__bytes_read.sum + dram__bytes_write.sum of one launch of this workload, ncu --set full ({prof_src}); "
                                            "the accumulators, the scene is 13 KB") if prof else prof_src,
                         "kernel": "pathtrace_kernel", "kernel_ms": st.trace_kernel_ms,
                         "algorithmic": (f"{FLOP_PER_SPHERE_TEST} FLOP x {st.sphere_tests} ray-sphere tests (rank 0 launch): {st.rays - st.beam_rays} swept ray segments x "
                                         f"{scene.n_spheres} spheres + {st.beam_tests} candidate tests of the {st.beam_rays} primary rays that were traced against "
                                         "their chunk's candidate list instead of the whole scene"),
                         "peak_source": "FFMA micro-kernel measured in this run (MEASURED_PEAKS.json has no FP32 figure)",
                         "note": "the path is neither HBM- nor tensor-bound (DRAM ~0 % busy). `achieved` / `frac` CREDIT 17 algorithmic FLOP per ray-sphere test "
                                 "(SURVEY 8d); the conservative prefilter executes 3 FMA per test, so the credited fraction can exceed 1 and does not measure "
                                 "pipe utilisation. `executed_tflops` / `executed_frac` count the FP32 instructions really executed (ncu) and are the figures "
                                 "to hold against the >= 60 % FP32-FMA target (DESIGN.md 3.1)",
                         "peak_nominal": NOMINAL_FP32_TFLOPS, "frac_of_nominal": achieved / NOMINAL_FP32_TFLOPS,
                         "hbm": hbm},
        }
        if c4:
            line["c4"] = c4
        if hierarchy:
            line["hierarchy"] = hierarchy
        if world > 1:
            line["frame_matches_single_gpu"] = frame_matches
            line["config"]["frame_end"] = ("each rank's kernels store its rows into rank 0's frame over NVLink (CUDA IPC mapping), one-element all-reduce as barrier"
                                           if peer else "pack + NCCL gather onto rank 0 + de-interleave")
        if args.bvh:
            line["config"]["workload"] += " [--bvh: hierarchy traversal instead of the brute-force sweep; roofline figures do not apply]"
            line["accel"] = {"node_visits": st.accel_node_visits, "prim_tests": st.accel_prim_tests, "build_ms": st.accel_build_ms}
        if spp != SPP:
            line["config"]["workload"] += f" [OVERRIDE spp={spp}: not the BASELINE config]"
            line["config"]["spp"] = spp
        if world == 1 and not args.no_cpu_baseline:
            n_threads = usable_cores()
            rate, _, sample, _ = cpu_port_rate(n_threads)
            line["cpu_baseline"] = {"value": rate, "unit": "Mrays/s", "cores": n_threads, "kind": "port", "sample": sample}
            line["reference_native"] = reference_native_rate()
        sys.stdout.flush()
        os.write(json_fd, (json.dumps(line) + "\n").encode())
    if job:
        job.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
