"""The scenes of tests/pathtrace_edges.py on the CPU restatement (oracle/rt3_oracle.c): each has the property the GPU half
(tests/test_gpu_pathtrace_edges.py) relies on, so that a GPU failure there is the kernel's and not the scene's. Buried padding
changes neither the frame nor the ray count at any count of the ladder; a bit-identical copy of a sphere at a higher id changes
nothing, and the same copy at a LOWER id changes many pixels (the case can see a wrong winner); and the GPU cases reach every
path-tracer instantiation."""
import numpy as np
import pytest

import oraclelib as ol
import pathtrace_edges as pe

W, H, SPP, DEPTH = 48, 27, 8, 50


@pytest.fixture(scope="module")
def c1_frame():
    scene, cam = pe.c1_padded(4, W, H)
    frame, _, rays = ol.oracle_pathtrace(scene, cam, pe.pt(W, H, SPP, DEPTH))
    assert (frame != frame[0, 0]).sum() > W * H // 2   # a real picture, not the sky
    return frame, rays


@pytest.mark.parametrize("faces", [0, 1], ids=["spheres", "mixed"])
@pytest.mark.parametrize("n", [n for n in pe.LADDER if n >= 5])
def test_buried_padding_changes_nothing(c1_frame, n, faces):
    """C1 padded with buried spheres (and, mixed, with buried triangles ahead of its spheres: faces take the low ids) to n."""
    scene, cam = pe.c1_padded(n, W, H, faces=(n - 4) // 2 if faces else 0)
    assert scene.n_faces + scene.n_spheres == n
    frame, _, rays = ol.oracle_pathtrace(scene, cam, pe.pt(W, H, SPP, DEPTH))
    assert rays == c1_frame[1]
    assert np.array_equal(frame, c1_frame[0]), f"{int((frame != c1_frame[0]).sum())} pixels differ"


def test_buried_padding_of_the_cover_scene_changes_nothing():
    """C2 (484 spheres) padded to 769 and 1025: a few rows of the 1200x800 frame, as one-row partitions."""
    base, cam = pe.c2_padded(485, 1200, 800)
    for y in (400, 640):
        p = pe.pt(1200, 800, 2, 50, tile_rows=1, part_index=y, part_count=800)
        ref, _, rays = ol.oracle_pathtrace(base, cam, p)
        for total in (769, 1025):
            scene, _ = pe.c2_padded(total, 1200, 800)
            frame, _, r = ol.oracle_pathtrace(scene, cam, p)
            assert r == rays and np.array_equal(frame[y], ref[y]), (y, total)


@pytest.mark.parametrize("name", list(pe.TIE_CASES))
def test_copy_after_the_original_changes_nothing(c1_frame, name):
    (scene, cam), without = pe.tie_scene(name, W, H)
    frame, _, rays = ol.oracle_pathtrace(scene, cam, pe.pt(W, H, SPP, DEPTH))
    assert rays == c1_frame[1] and np.array_equal(frame, c1_frame[0]), f"{int((frame != c1_frame[0]).sum())} pixels differ"
    plain, _, _ = ol.oracle_pathtrace(without, cam, pe.pt(W, H, SPP, DEPTH))
    assert np.array_equal(plain, c1_frame[0])


@pytest.mark.parametrize("original_at,copy_at,total", [(32, 31, 40), (512, 511, 520), (1024, 1023, 1032)])
def test_copy_before_the_original_changes_many_pixels(c1_frame, original_at, copy_at, total):
    """The sensitivity of the tie cases: with the metal copy at the lower id, the copy wins and the middle sphere turns metal."""
    scene, cam = pe.with_copies(total, W, H, original_at, [copy_at])
    frame, _, _ = ol.oracle_pathtrace(scene, cam, pe.pt(W, H, SPP, DEPTH))
    assert (frame != c1_frame[0]).sum() > W * H // 5


def test_ladder_scenes_have_the_planned_counts():
    for n in pe.LADDER:
        for form in pe.FORMS:
            scene, _ = pe.ladder_scene(n, form, pe.LADDER_W, pe.LADDER_H)
            assert (scene.n_faces, scene.n_spheres) == pe.ladder_split(n, form)
    assert {pe.ladder_split(n, "mixed")[0] for n in pe.LADDER} >= set(pe.FACE_SPLITS)
    # the bank decision is made on the padded count: 761..768 are resident, 769 is streamed
    assert pe.kernel_for(0, 760, 4, False)[0] == pe.kernel_for(0, 768, 4, False)[0] == 1 and pe.kernel_for(0, 769, 4, False)[0] == 0


def test_ladder_scenes_are_seen_up_to_their_last_ids():
    """A ladder scene's high ids are hit by its rays (on a coarse depth-1 image), so a dropped tail tile would show."""
    for n, form in ((1025, "spheres"), (1537, "mixed"), (2049, "mixed_materials")):
        scene, cam = pe.ladder_scene(n, form, pe.LADDER_W, pe.LADDER_H)
        _, prim, _, _ = ol.oracle_reference(scene, cam, 160, 96)
        assert (prim >= n - 1 - (n - 1) % 1024).any(), f"{form} {n}: nothing of the last tile is visible"


def test_gpu_cases_reach_every_pathtrace_instantiation():
    reached = pe.planned_kernels()
    assert set(reached) == pe.KERNELS, f"missing {pe.KERNELS - set(reached)}, unknown {set(reached) - pe.KERNELS}"
