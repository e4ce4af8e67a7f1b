"""bench.py's contract: the reference arm (`--impl reference`: the CPU restatement on the host's cores, a bounded sample of the GPU
arm's workload) prints one JSON line with the agreed keys, the product arm refuses to run -- loudly, with no CPU fallback -- when there
is no CUDA device, and `--dump-outputs` writes the frame the timed path computed in its last step."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(*args, timeout=300):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=timeout, cwd=ROOT)


def levels(frame):
    """Packed frame [H, W] -> [H, W, 4] float32 channel levels r, g, b, a: the layout of --dump-outputs' frame.npy."""
    return np.stack([(frame >> s) & 0xFF for s in (24, 16, 8, 0)], -1).astype(np.float32)


def test_reference_arm_line(tmp_path):
    r = run_bench("--impl", "reference", "--steps", "1", "--warmup", "0", "--dump-outputs", str(tmp_path))
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, "exactly one JSON line"
    line = json.loads(lines[0])
    assert line["impl"] == "reference" and line["metric"] == "Mrays/s" and line["unit"] == "Mrays/s" and line["higher_is_better"] is True
    assert line["n_gpus"] == 1 and line["steps"] == 1 and line["warmup"] == 0 and line["value"] > 0 and line["ms_per_step"] > 0
    assert line["vs_baseline"] is None and line["data"] == "synthetic" and line["dtype"] == "f32"
    cfg = line["config"]
    assert (cfg["width"], cfg["height"], cfg["spp"], cfg["max_depth"]) == (1200, 800, 500, 50), "the GPU arm's workload (BASELINE configs[1])"
    assert "timed_sample" in cfg and "bounded sample" in cfg["workload"], "the label says what is really rendered per step"
    cb = line["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["value"] == line["value"] and cb["sample"]
    assert line["e2e"] == {"value": line["value"], "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    # --dump-outputs: the frame of the timed sample (its layout is checked exactly by the large-frame test below)
    assert os.listdir(tmp_path) == ["frame.npy"]
    got = np.load(tmp_path / "frame.npy")
    s = cfg["timed_sample"]
    assert got.dtype == np.float32 and got.shape == (s["height"], s["width"], 4)
    assert (got == np.round(got)).all() and got.min() >= 0 and got.max() <= 255 and (got[..., 3] == 255).all() and got[..., :3].std() > 0
    r = run_bench("--impl", "reference", "--steps", "0")
    assert r.returncode == 2 and "at least 1" in r.stderr, "--steps sets the number of timed steps: zero is refused"


def test_dump_of_a_large_frame_is_a_fixed_row_sample(tmp_path):
    """A frame above the dump's size limit (a 3840x2160 one, as --config c4 times) is written as the same seeded sample of rows every time."""
    sys.path.insert(0, ROOT)
    import bench
    frame = np.random.default_rng(5).integers(0, 1 << 32, (2160, 3840), dtype=np.uint32)
    for d in ("a", "b"):
        bench.dump_frame(str(tmp_path / d), frame)
    a, b = tmp_path / "a", tmp_path / "b"
    assert sum(f.stat().st_size for f in a.iterdir()) <= bench.DUMP_BYTES
    rows = np.load(a / "frame_rows.npy")
    assert rows.dtype == np.float64 and (np.diff(rows) > 0).all() and rows[-1] < 2160
    assert np.array_equal(rows, np.load(b / "frame_rows.npy")) and np.array_equal(np.load(a / "frame.npy"), np.load(b / "frame.npy"))
    assert np.array_equal(np.load(a / "frame.npy"), levels(frame[rows.astype(np.int64)]))


@pytest.mark.skipif(torch.cuda.is_available(), reason="needs a machine without a GPU")
def test_product_arm_fails_loudly_without_a_gpu():
    r = run_bench("--steps", "1", "--warmup", "0", "--no-cpu-baseline", "--no-c4", timeout=120)
    assert r.returncode != 0, "no CPU fallback: the product arm must not produce a number without a CUDA device"
    assert not [l for l in r.stdout.splitlines() if l.startswith("{") and '"value"' in l]


@pytest.mark.gpu
def test_product_arm_dumps_the_timed_frame(built, tmp_path):
    """--dump-outputs on the GPU arm: the last timed frame is the frame rt3_render returns for the same workload."""
    r = run_bench("--steps", "2", "--warmup", "1", "--spp", "4", "--no-c4", "--no-cpu-baseline", "--dump-outputs", str(tmp_path), timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][0])
    assert line["steps"] == 2
    from rt3_b200 import abi, scenes
    w, h = line["config"]["width"], line["config"]["height"]
    scene, cam = scenes.rtiow_cover(w, h)
    ctx = abi.Context(0)
    try:
        ctx.upload(scene)
        want = ctx.render(cam, abi.make_params(w, h, mode=abi.MODE_PATHTRACE, spp=4, max_depth=line["config"]["max_depth"], seed=1,
                                               tile_rows=line["config"]["tile_rows"]))
    finally:
        ctx.close()
    got = np.load(tmp_path / "frame.npy")
    assert got.dtype == np.float32 and np.array_equal(got, levels(want))
