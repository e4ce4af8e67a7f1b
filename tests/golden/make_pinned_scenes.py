"""Regenerates tests/golden/pinned_scenes.npz: what tests/test_oracle_pinned.py compares the CPU restatement with when the
compiled reference (oracle/_ref/libref_seq.so) is not built.

    python tests/golden/make_pinned_scenes.py

Stored: the 'mixed' scene and its frames at 161x97 and 2x2, the ten seeded random scenes with their frames (rows 0..H-2, the
rows the reference writes), and the reference camera vectors at four sizes. With the compiled reference built, scenes, frames
and vectors are the reference's own (its ECS export, its Sequential renderer, its Camera::update) and the restatement is checked
equal to them first. Without it, the scenes come from the host backend's flatten and the frames and vectors from the restatement
(oracle/rt3_oracle.c, abi.reference_camera): the values these tests had pinned bit-equal to the compiled reference. `source`
in the file says which.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, os.path.dirname(HERE))
import hostlib  # noqa: E402
import oraclelib as ol  # noqa: E402
from rt3_b200 import abi  # noqa: E402

MIXED_SIZES = [(161, 97), (2, 2)]
CAMERA_SIZES = [(400, 225), (800, 600), (1200, 800), (7, 3)]
N_RANDOM = 10


def scene_arrays(prefix, scene):
    return {prefix + "_faces": scene.faces.view(np.uint8).reshape(-1, 48), prefix + "_vertices": scene.vertices.view(np.uint8).reshape(-1, 16),
            prefix + "_face_entity": scene.face_entity}


def build(add, *args):
    """(scene arrays, frame renderer (w, h) -> rows 0..H-2, what `add` returned) of the scene `add` builds, from the reference or
    the restatement."""
    if ol.have_ref():
        s = ol.RefScene()
        ret = add(s, *args)
        s.prerender()
        scene = s.export()

        def render(w, h):
            frame, _ = s.render(w, h)
            mine, _, _, _ = ol.oracle_reference(scene, abi.reference_camera(w, h), w, h)
            assert np.array_equal(frame[:h - 1], mine[:h - 1]), "the restatement differs from the compiled reference"
            return frame[:h - 1]
    else:
        s = hostlib.HostScene()
        ret = add(s, *args)
        scene = s.flatten()

        def render(w, h):
            return ol.oracle_reference(scene, abi.reference_camera(w, h), w, h)[0][:h - 1]
    return scene, render, ret


def camera_vectors(w, h):
    if ol.have_ref():
        import ctypes as C
        out = (C.c_float * 12)()
        vw = float(np.float32(np.float32(w) / np.float32(h)) * np.float32(2.0))
        assert ol.ref().ref_camera_vectors(w, h, 2.0, vw, 2.0, out) == 0
        return np.array(list(out), np.float32)
    cam = abi.reference_camera(w, h)
    return np.array(list(cam.origin) + list(cam.horizontal) + list(cam.vertical) + list(cam.lower_left_corner), np.float32)


def main():
    out = {"source": np.array("compiled reference" if ol.have_ref() else "restatement (oracle/rt3_oracle.c, abi.reference_camera)")}
    scene, render, _ = build(ol.add_scene, "mixed")
    out.update(scene_arrays("mixed", scene))
    for w, h in MIXED_SIZES:
        out[f"mixed_{w}x{h}"] = render(w, h)
    for seed in range(N_RANDOM):
        scene, render, (w, h) = build(ol.add_random_scene, seed)
        out.update(scene_arrays(f"random{seed}", scene))
        out[f"random{seed}_frame"] = render(w, h)
        out[f"random{seed}_size"] = np.array([w, h], np.uint32)
    for w, h in CAMERA_SIZES:
        out[f"camera_{w}x{h}"] = camera_vectors(w, h)
    path = os.path.join(HERE, "pinned_scenes.npz")
    np.savez_compressed(path, **out)
    print(path, out["source"], os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
