"""Host backend (C++): the ECS scene API and the flatten step produce, bit for bit, the arrays the
reference renders from (reference Sphere.cpp:120-351, Object.cpp:131-199, Triangle.cpp:58-76,
SequentialRenderer.cpp:174-266). CPU only."""
import json
import os

import numpy as np
import pytest

import hostlib
import oraclelib as ol
from conftest import ROOT, load_golden
from rt3_b200 import abi, scenes

META = json.load(open(os.path.join(ROOT, "tests", "golden", "goldens.json")))


def same_scene(a: abi.SceneArrays, b: abi.SceneArrays):
    assert a.n_faces == b.n_faces and len(a.vertices) == len(b.vertices)
    assert np.array_equal(a.faces["v"], b.faces["v"])
    for field in ("normal", "color"):
        assert np.array_equal(a.faces[field].view(np.uint32), b.faces[field].view(np.uint32)), field
    assert np.array_equal(a.vertices.view(np.uint8), b.vertices.view(np.uint8))
    assert np.array_equal(a.face_entity, b.face_entity)


@pytest.mark.parametrize("name", ["triangle_400x225", "sphere8_400x225"])
def test_flatten_matches_golden_scene(built, name):
    _, golden = load_golden(name)
    hs = hostlib.HostScene()
    if name.startswith("triangle"):
        hs.add_triangle((1, 0, -3), (-1, 0, -3), (0, 1, -3), (1, 0, 0))
    else:
        hs.add_sphere((0, 0, -3), 1.0, 8, 8, (1, 0, 0))
    same_scene(hs.flatten(), golden)


def test_large_tessellated_sphere_counts(built):
    """create_sphere(.., 225, 225, ..): the ~100k-triangle mesh of config C3 (SURVEY.md section 0)."""
    hs = hostlib.HostScene()
    hs.add_sphere((0, 0, -3), 1.0, 225, 225, (1, 0, 0))
    flat = hs.flatten()
    m = META["sphere225_64x36"]
    assert (flat.n_faces, len(flat.vertices)) == (m["n_faces"], m["n_vertices"]) == (100350, 50177)
    # the restatement renders this flatten to the reference's golden image
    frame, _, _, _ = ol.oracle_reference(flat, abi.reference_camera(64, 36), 64, 36)
    assert f"{ol.fnv64(frame[:35]):016x}" == m["frame_fnv64_rows_0_to_Hm2"]


def teddy_obj_from_golden(path, golden):
    """Writes an OBJ of the teddy (entity 0 of the reference's default scene) whose vertices the reference's transform maps exactly
    onto the reference's own export of them in tests/golden/default_400x225.npz: v = (p - centre) / scale, moved by whole ulps until
    fp32 centre + scale * v gives p back. The original teddy.obj is not in the repository; its faces are written as exported."""
    f = np.float32
    scale, centre = f(1.0) / f(17.0), np.array([0, 0, -3], f)
    faces = golden.faces["v"][golden.face_entity == 0]
    want = golden.vertices.view(f).reshape(-1, 4)[:int(faces.max()) + 1, :3]
    guess = ((want.astype(np.float64) - centre) / np.float64(scale)).astype(f)
    v = np.full(want.shape, np.nan, f)
    for k in range(-8, 9):
        cand = guess
        for _ in range(abs(k)):
            cand = np.nextafter(cand, f(np.inf) if k > 0 else f(-np.inf))
        found = np.isnan(v) & (centre + scale * cand == want)
        v[found] = cand[found]
    assert not np.isnan(v).any()
    with open(path, "w") as fh:
        fh.writelines(f"v {float(x)!r} {float(y)!r} {float(z)!r}\n" for x, y, z in v)   # repr: strtof reads each value back exactly
        fh.writelines(f"f {a + 1} {b + 1} {c + 1}\n" for a, b, c in faces)


def test_flatten_matches_compiled_reference(built, tmp_path):
    """The reference's default scene (src/Main.cpp:278-283: teddy at (0, 0, -3) scaled 1/17, an 8x8 sphere) through the host's OBJ
    loader and flatten equals the reference's own export of it, bit for bit: faces, normals, colours, vertices, entity map. With
    the compiled reference built, a five-entity scene with the original teddy.obj is also compared with it directly."""
    _, golden = load_golden("default_400x225")
    teddy = str(tmp_path / "teddy.obj")
    teddy_obj_from_golden(teddy, golden)
    hs = hostlib.HostScene()
    hs.add_object(teddy, (0, 0, -3), 1.0 / 17.0, (1, 0, 0))
    hs.add_sphere((-2, 0, -5), 1.0, 8, 8, (0, 0, 1))
    same_scene(hs.flatten(), golden)
    if not ol.have_ref():
        return
    ref, hs = ol.RefScene(), hostlib.HostScene()
    for s in (ref, hs):
        s.add_object(ol.REF_TEDDY, (0, 0, -3), 1.0 / 17.0, (1, 0, 0))
        s.add_sphere((-2, 0, -5), 1.0, 8, 8, (0, 0, 1))
        s.add_triangle((2, -1, -5), (-2, -1, -5), (0, 2, -6), (0.1, 0.2, 1.0))
        s.add_sphere((0.6, 0.2, -4), 0.9, 12, 9, (0.2, 0.9, 0.3))
        s.add_sphere((0.1, 0.2, -2), 0.3, 5, 3, (0.2, 0.9, 0.3))   # fewest parallels the reference supports
    ref.prerender()
    same_scene(hs.flatten(), ref.export())
    assert hs.flatten().n_faces == 3192 + 96 + 1 + 2 * 12 * 7 + 10


def test_obj_loader_tolerates_what_the_reference_rejects(built, tmp_path):
    p = tmp_path / "quad.obj"
    p.write_text("# comment\n\nv 0 0 -3\nv 1 0 -3\nv 1 1 -3\nv 0 1 -3\nvn 0 0 1\nf 1/1/1 2/2/1 3/3/1\nf 1 3 4\n")
    hs = hostlib.HostScene()
    hs.add_object(str(p), (0, 0, 0), 1.0, (1, 1, 1))
    flat = hs.flatten()
    assert flat.n_faces == 2 and len(flat.vertices) == 4
    assert flat.faces["v"].tolist() == [[0, 1, 2], [0, 2, 3]]
    assert np.allclose(np.abs(flat.faces["normal"]), [[0, 0, 1], [0, 0, 1]])


def test_missing_obj_is_fatal(built):
    hs = hostlib.HostScene()
    with pytest.raises(hostlib.HostError, match="Could not open file"):
        hs.add_object("/nonexistent/teddy.obj", (0, 0, 0), 1.0, (1, 1, 1))


def test_look_at_camera_matches_python_builder(built):
    look = (13, 2, 3, 0, 0, 0, 0, 1, 0, 20.0, 0.1, 10.0)
    got = hostlib.camera_vectors(1200, 800, look)
    cam = scenes.look_at_camera((13, 2, 3), (0, 0, 0), (0, 1, 0), 20.0, 1200 / 800, aperture=0.1, focus_dist=10.0)
    want = np.array(list(cam.origin) + list(cam.horizontal) + list(cam.vertical) + list(cam.lower_left_corner) + [cam.lens_radius] +
                    list(cam.lens_u) + list(cam.lens_v), np.float32)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))


@pytest.mark.parametrize("fmt", ["ppm", "png"])
def test_frame_writers_round_trip(built, tmp_path, fmt):
    """Frame::to_ppm / Frame::to_png (reference Frame.cpp:82-148): what an image reader gets back is the frame."""
    from PIL import Image
    rng = np.random.default_rng(3)
    for w, h in ((1, 1), (37, 11), (400, 225)):      # the last one needs several 64 KiB deflate blocks
        frame = (rng.integers(0, 1 << 24, (h, w), dtype=np.uint32) << 8) | 0xFF
        path = tmp_path / f"f{w}x{h}.{fmt}"
        hostlib.write_image(frame, path, fmt)
        img = Image.open(path)
        assert img.size == (w, h) and img.mode == ("RGBA" if fmt == "png" else "RGB")
        px = np.array(img).astype(np.uint32)
        back = (px[..., 0] << 24) | (px[..., 1] << 16) | (px[..., 2] << 8) | 0xFF
        assert np.array_equal(back, frame)
        if fmt == "png":
            assert np.all(px[..., 3] == 255)
    with pytest.raises(hostlib.HostError, match="Could not open"):
        hostlib.write_image(frame, tmp_path / "no_such_dir" / "x.png", fmt)
