"""Pins the CPU restatement (oracle/rt3_oracle.c) to the reference.

* against the committed golden vectors (generated from the compiled reference by
  tests/golden/make_goldens.py) -- runs anywhere;
* against the compiled reference itself (oracle/_ref/libref_seq.so, built from
  the reference's sources by oracle/Makefile) when it is present, and otherwise against
  the scenes, frames and camera vectors stored by tests/golden/make_pinned_scenes.py.
Bar: bit-exact packed pixels on rows 0..H-2 (the reference never writes the last
row, SequentialRenderer.cpp:286).
"""
import json
import os

import numpy as np
import pytest

import oraclelib as ol
from conftest import ROOT, load_golden
from rt3_b200 import abi

META = json.load(open(os.path.join(ROOT, "tests", "golden", "goldens.json")))


@pytest.mark.parametrize("name", ["triangle_400x225", "sphere8_400x225", "default_400x225"])
def test_restatement_matches_golden(built, name):
    g, scene = load_golden(name)
    m = META[name]
    w, h = m["width"], m["height"]
    assert scene.n_faces == m["n_faces"] and len(scene.vertices) == m["n_vertices"]
    frame, prim, ent, t = ol.oracle_reference(scene, abi.reference_camera(w, h), w, h)
    assert np.array_equal(frame[:h - 1], g["frame"])
    assert np.array_equal(prim[:h - 1], g["prim"])
    assert np.array_equal(t[:h - 1].view(np.uint32), g["t_bits"])
    assert f"{ol.fnv64(frame[:h - 1]):016x}" == m["frame_fnv64_rows_0_to_Hm2"]
    assert f"{int(frame[0, 0]):08x}" == m["pixel_0"] and f"{int(frame[h // 2, w // 2]):08x}" == m["pixel_centre"]
    ids, counts = np.unique(ent[:h - 1], return_counts=True)
    assert {f"{int(i):x}": int(c) for i, c in zip(ids, counts)} == m["entity_histogram"]


def test_survey_known_answers():
    """Numbers SURVEY.md section 8c quotes for the default scene at 400x225."""
    m = META["default_400x225"]
    assert (m["n_faces"], m["n_vertices"]) == (3288, 1648)
    assert m["entity_histogram"] == {"0": 18883, "1": 5824, "ffffffff": 64893}
    assert m["pixel_0"] == "a9cbffff" and m["pixel_centre"] == "bd0000ff"
    g, _ = load_golden("default_400x225")
    t = g["t_bits"].view(np.float32)
    hit = np.isfinite(t)
    assert abs(float(t[hit].min()) - 1.08735) < 1e-5 and abs(float(t[hit].max()) - 2.49954) < 1e-5


needs_ref = pytest.mark.skipif(not ol.have_ref(), reason="oracle/_ref/libref_seq.so not built (needs the reference's sources)")
# what the tests below compare with when the compiled reference is not built (tests/golden/make_pinned_scenes.py says where it comes from)
PINS = np.load(os.path.join(ROOT, "tests", "golden", "pinned_scenes.npz"))


def pinned_scene(prefix):
    return abi.SceneArrays(faces=PINS[prefix + "_faces"].view(abi.FACE_DTYPE).ravel(),
                           vertices=PINS[prefix + "_vertices"].view(abi.VERTEX_DTYPE).ravel(), face_entity=PINS[prefix + "_face_entity"])


def _ref_scene(kind):
    s = ol.RefScene()
    ol.add_scene(s, kind)
    s.prerender()
    return s


def reference_rows(kind, w, h):
    """(scene, the reference's frame rows 0..H-2): rendered by the compiled reference when it is built, else stored -- the
    reference's goldens for the triangle and sphere8 scenes at 400x225, tests/golden/pinned_scenes.npz for the mixed one."""
    if ol.have_ref():
        rs = _ref_scene(kind)
        ref_frame, _ = rs.render(w, h)
        assert (ref_frame[h - 1] == 0).all(), "the reference is expected to leave the last row unwritten"
        return rs.export(), ref_frame[:h - 1]
    if kind == "mixed":
        return pinned_scene("mixed"), PINS[f"mixed_{w}x{h}"]
    g, scene = load_golden(f"{kind}_{w}x{h}")
    return scene, g["frame"]


@pytest.mark.parametrize("kind,w,h", [("triangle", 400, 225), ("sphere8", 400, 225), ("mixed", 161, 97), ("mixed", 2, 2)])
def test_restatement_matches_compiled_reference(built, kind, w, h):
    scene, ref_rows = reference_rows(kind, w, h)
    frame, prim, ent, t = ol.oracle_reference(scene, abi.reference_camera(w, h), w, h)
    assert np.array_equal(frame[:h - 1], ref_rows)
    # entity map: contiguous face ranges in entity order
    hit = prim != abi.NO_HIT
    assert np.array_equal(ent[hit], scene.face_entity[prim[hit]])


@needs_ref
def test_golden_hashes_reproduce_from_compiled_reference(built):
    for name in ("triangle_400x225", "sphere8_400x225"):
        m = META[name]
        rs = _ref_scene(m["scene"])
        frame, _ = rs.render(m["width"], m["height"])
        assert f"{ol.fnv64(frame[:m['height'] - 1]):016x}" == m["frame_fnv64_rows_0_to_Hm2"]


@pytest.mark.parametrize("w,h", [(400, 225), (800, 600), (1200, 800), (7, 3)])
def test_camera_vectors_match_reference(w, h):
    """Camera::update's vectors (the compiled reference's when built, else the stored ones), bit for bit."""
    if ol.have_ref():
        import ctypes as C
        out = (C.c_float * 12)()
        vw = float(np.float32(np.float32(w) / np.float32(h)) * np.float32(2.0))
        assert ol.ref().ref_camera_vectors(w, h, 2.0, vw, 2.0, out) == 0
        want = np.array(list(out), np.float32)
    else:
        want = PINS[f"camera_{w}x{h}"]
    cam = abi.reference_camera(w, h)
    mine = list(cam.origin) + list(cam.horizontal) + list(cam.vertical) + list(cam.lower_left_corner)
    assert np.array_equal(np.array(mine, np.float32).view(np.uint32), want.view(np.uint32))


@pytest.mark.parametrize("seed", range(10))
def test_restatement_matches_compiled_reference_on_random_scenes(built, seed):
    """Randomised pinning: triangles and tessellated spheres at random places (in front of, around and behind the camera,
    overlapping, some degenerate), random frame sizes; pixels of rows 0..H-2 bit-equal to the compiled reference (when it is
    not built: to the stored scenes and frames)."""
    if ol.have_ref():
        s = ol.RefScene()
        w, h = ol.add_random_scene(s, seed)
        s.prerender()
        scene = s.export()
        ref_frame, _ = s.render(w, h)
        ref_rows = ref_frame[:h - 1]
    else:
        scene = pinned_scene(f"random{seed}")
        w, h = (int(x) for x in PINS[f"random{seed}_size"])
        ref_rows = PINS[f"random{seed}_frame"]
    frame, prim, ent, t = ol.oracle_reference(scene, abi.reference_camera(w, h), w, h)
    assert np.array_equal(frame[:h - 1], ref_rows), f"{int((frame[:h - 1] != ref_rows).sum())} pixels differ ({scene.n_faces} faces, {w}x{h})"
