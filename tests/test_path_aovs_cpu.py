"""The AOVs of the path tracer's primary rays (rt3_render_path_aovs) on the CPU: the restatement's values on cases that can be
checked by hand, and the ABI struct's layout against include/rt3cuda.h. No GPU needed."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

import path_aov_lib as pal
from rt3_b200 import abi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
W, H = 41, 31   # odd: the centre pixel's primary ray is the camera axis


def one_sphere(kind, albedo=(0.25, 0.5, 0.75), centre=(0, 0, -3)):
    mats = np.zeros(1, abi.MATERIAL_DTYPE)
    mats["kind"], mats["albedo"], mats["ior"] = kind, albedo, 1.5
    return abi.SceneArrays(spheres=np.array([[*centre, 1.0]], np.float32), sphere_material=np.zeros(1, np.uint32),
                           sphere_entity=np.array([7], np.uint32), materials=mats)


def params(flags=abi.FLAG_NO_JITTER, spp=4, **kw):
    return abi.make_params(W, H, mode=abi.MODE_PATHTRACE, spp=spp, max_depth=0, seed=3, flags=flags, **kw)


def sky(cam, width, height):
    """shade_miss with throughput 1 for the un-jittered pinhole rays, in fp32 as the oracle and the kernel compute it."""
    f = np.float32
    x = np.arange(width, dtype=f)[None, :]
    y = np.arange(height)[:, None]
    u = (x + f(0)) / (f(width) - f(1))
    v = (f(1) * (height - 1 - y).astype(f) + f(0)) / (f(height) - f(1))
    o, hor, ver, llc = (np.array(getattr(cam, k), f) for k in ("origin", "horizontal", "vertical", "lower_left_corner"))
    d = ((llc + u[..., None] * hor) + v[..., None] * ver) - o
    inv = f(1) / np.sqrt((d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2])
    t = f(0.5) * (d[..., 1] * inv + f(1))
    a = f(1) - t
    return np.stack([a * f(1) + t * f(0.5), a * f(1) + t * f(0.7), a * f(1) + t * f(1)], -1).astype(f)


def test_one_material_scene_has_that_albedo_on_every_hit_pixel():
    cam = abi.reference_camera(W, H)
    out = pal.oracle_path_aovs(one_sphere(abi.MAT_LAMBERTIAN), cam, params())
    hit = out["hit_prim"] != abi.NO_HIT
    assert 0 < hit.sum() < W * H
    assert np.array_equal(out["albedo"][hit], np.broadcast_to(np.float32([0.25, 0.5, 0.75]), (hit.sum(), 3)))
    assert (out["hit_entity"][hit] == 7).all() and (out["hit_t"][hit] > 0).all()
    metal = pal.oracle_path_aovs(one_sphere(abi.MAT_METAL), cam, params())
    assert np.array_equal(metal["albedo"], out["albedo"])


def test_dielectric_albedo_is_one():
    out = pal.oracle_path_aovs(one_sphere(abi.MAT_DIELECTRIC), abi.reference_camera(W, H), params())
    hit = out["hit_prim"] != abi.NO_HIT
    assert hit.any() and (out["albedo"][hit] == 1.0).all()


def test_misses_get_the_sky_zero_normal_no_hit_and_infinity():
    cam = abi.reference_camera(W, H)
    scene = one_sphere(abi.MAT_LAMBERTIAN, centre=(0, 0, 5))   # behind the camera: every primary ray misses
    out = pal.oracle_path_aovs(scene, cam, params())
    assert (out["hit_prim"] == abi.NO_HIT).all() and (out["hit_entity"] == abi.NO_HIT).all()
    assert np.isposinf(out["hit_t"]).all() and (out["normal"] == 0).all()
    q = (sky(cam, W, H) * np.float32(2 ** 24) + np.float32(0.5)).astype(np.uint64)   # to_fixed: the sums are 2^24 fixed point
    assert np.array_equal(out["albedo"], (q.astype(np.float64) / 2 ** 24).astype(np.float32))
    white = pal.oracle_path_aovs(scene, cam, params(abi.FLAG_NO_JITTER | abi.FLAG_UNIFORM_SKY))
    assert (white["albedo"] == 1.0).all()


def test_sphere_seen_along_its_axis():
    out = pal.oracle_path_aovs(one_sphere(abi.MAT_LAMBERTIAN), abi.reference_camera(W, H), params(spp=3))
    cy, cx = H // 2, W // 2
    assert out["hit_prim"][cy, cx] == 0 and out["hit_t"][cy, cx] == 2.0
    assert np.array_equal(out["normal"][cy, cx], np.float32([0, 0, 1]))
    # every hit normal is a mean of unit front-facing normals: towards the camera
    hit = out["hit_prim"] != abi.NO_HIT
    assert (out["normal"][hit][:, 2] > 0).all()


def test_jittered_means_are_means_of_the_samples():
    """spp samples = the mean of the spp one-sample passes (first_sample = 0 .. spp - 1), up to the float resolve."""
    cam = abi.reference_camera(W, H)
    scene = one_sphere(abi.MAT_LAMBERTIAN)
    many = pal.oracle_path_aovs(scene, cam, params(flags=0, spp=5))
    ones = [pal.oracle_path_aovs(scene, cam, params(flags=0, spp=1, first_sample=s)) for s in range(5)]
    for k in ("albedo", "normal"):
        assert np.allclose(many[k], np.mean([o[k] for o in ones], axis=0), atol=1e-6)
    for k in ("hit_prim", "hit_t"):
        assert np.array_equal(many[k], ones[0][k])


def test_rows_of_other_partitions_are_untouched():
    cam = abi.reference_camera(W, H)
    scene = one_sphere(abi.MAT_LAMBERTIAN)
    full = pal.oracle_path_aovs(scene, cam, params(flags=0, spp=2))
    part = pal.oracle_path_aovs(scene, cam, params(flags=0, spp=2, tile_rows=2, part_index=1, part_count=3))
    owned = (np.arange(H) // 2) % 3 == 1
    for k in pal.AOV_KEYS:
        assert np.array_equal(part[k][owned].view(np.uint32), full[k][owned].view(np.uint32)), k
        assert (part[k][~owned] == 0).all(), k


@pytest.mark.skipif(shutil.which(os.environ.get("CC", "gcc")) is None, reason="no C compiler")
def test_path_aovs_struct_matches_header(tmp_path):
    src = tmp_path / "layout.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "rt3cuda.h"\nint main(void) {\n'
                   '  printf("%zu", sizeof(rt3_path_aovs));\n'
                   + "".join(f'  printf(" %zu", offsetof(rt3_path_aovs, {k}));\n' for k in pal.AOV_KEYS) + "  return 0;\n}\n")
    exe = tmp_path / "layout"
    subprocess.run([os.environ.get("CC", "gcc"), "-std=c99", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)], check=True)
    size, *offsets = (int(v) for v in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split())
    assert size == C.sizeof(abi.PathAovs)
    assert offsets == [getattr(abi.PathAovs, k).offset for k in pal.AOV_KEYS]
    assert "rt3_render_path_aovs" in abi.EXPORTED_SYMBOLS
