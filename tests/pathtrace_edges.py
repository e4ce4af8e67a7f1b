"""Scenes that move the path tracer across the counts and ids where its sweep changes shape, used by the CPU half
(tests/test_pathtrace_edges_cpu.py: each builder has the property the GPU tests rely on) and the GPU half
(tests/test_gpu_pathtrace_edges.py: the kernels against the CPU restatement and against themselves).

Where the sweep changes shape (raytracer-3_b200/csrc/rt3_device.cuh): the primitive array is padded to a multiple of 8
(RT3_PAD_PRIMS) with never-surviving records; survivor masks hold 32 primitives a word; 16 words (512 primitives) are swept
before they are drained; a scene whose PADDED count is at most 768 is swept out of the constant bank, a larger one is
streamed in 1 024-primitive tiles, the last one ragged. Ids are faces first, then spheres, and ties go to the lower id.

Three kinds of scene:
  * buried padding: spheres or triangles deep inside a ground sphere. Camera rays start outside it and Lambertian bounces
    leave its surface outward, so no ray reaches them: the frame and the ray count are those of the unpadded scene at
    every count, and a scene can be moved across every edge at its real shape.
  * ties: a visible sphere copied bit for bit with another material, the copy at a higher id on the far side of an edge
    (or a crowd of coincident copies): the lower id wins, so the frame is the one without the copies.
  * the count ladder: primitives a ray can reach at every id, so a dropped primitive or a wrong winner shows in the frame.
"""
import numpy as np

from rt3_b200 import abi, scenes

LADDER = [1, 7, 8, 9, 31, 32, 33, 511, 512, 513, 760, 768, 769, 1023, 1024, 1025, 1535, 1536, 1537, 2048, 2049]
FACE_SPLITS = [31, 32, 511, 512, 1023, 1024]   # face/sphere id boundaries the mixed ladder puts on word, chunk and tile edges
FORMS = ["spheres", "mixed", "mixed_materials"]

# the plan rules of enqueue_render / plan_trace (raytracer-3_b200/csrc/rt3_core.cu) and their constants
CONST_PRIMS, PAD_PRIMS, BIN_MIN_FACES, BIN_MAX_SPP = 768, 8, 1024, 8
# every pathtrace_kernel<RESIDENT, SPHERES_ONLY, ACCEL, BIN, BEAM> the library instantiates
KERNELS = {(1, 1, 0, 0, 0), (1, 0, 0, 0, 0), (0, 1, 0, 0, 0), (0, 0, 0, 0, 0), (1, 1, 0, 0, 1), (1, 0, 1, 0, 0),
           (1, 0, 1, 0, 1), (1, 0, 1, 1, 0), (1, 0, 1, 2, 0), (1, 0, 1, 3, 0), (1, 0, 1, 3, 1)}


def padded(n):
    return (n + PAD_PRIMS - 1) // PAD_PRIMS * PAD_PRIMS


def kernel_for(n_faces, n_spheres, spp, bvh, env=None):
    """The pathtrace_kernel instantiation a render takes, restated from enqueue_render: scene counts, spp, RT3_FLAG_BVH and
    the RT3_BEAM / RT3_BINNING / RT3_BEAM_BVH environment switches (`env`, strings as in the environment)."""
    env = env or {}
    spheres_only = n_faces == 0
    if not bvh:
        resident = padded(n_faces + n_spheres) <= CONST_PRIMS
        beam = resident and spheres_only and int(env.get("RT3_BEAM", "1")) != 0
        return (int(resident), int(spheres_only), 0, 0, int(beam))
    binning = 0
    if n_faces >= BIN_MIN_FACES:   # a face tree with a root node (n_faces >= 2)
        binning = 1 if spp <= BIN_MAX_SPP else 3
        if "RT3_BINNING" in env:
            binning = int(env["RT3_BINNING"])
    beam = binning == 0
    if "RT3_BEAM_BVH" in env:
        beam = binning in (0, 3) and int(env["RT3_BEAM_BVH"]) != 0
    if binning not in (0, 1, 2, 3):
        binning = 0
    return (1, 0, 1, binning, int(beam))


def normals(p):
    """Face normals as the reference computes them, normalize(cross(p3 - p1, p2 - p1)) in fp32 (Triangle.cpp:48): p is [n, 3, 3]."""
    a, b = p[:, 2] - p[:, 0], p[:, 1] - p[:, 0]
    c = np.stack([a[:, 1] * b[:, 2] - b[:, 1] * a[:, 2], a[:, 2] * b[:, 0] - b[:, 2] * a[:, 0], a[:, 0] * b[:, 1] - b[:, 0] * a[:, 1]], 1).astype(np.float32)
    inv = (np.float32(1.0) / np.sqrt((c[:, 0] * c[:, 0] + c[:, 1] * c[:, 1]) + c[:, 2] * c[:, 2], dtype=np.float32)).astype(np.float32)
    return c * inv[:, None]


def triangles(p, colors):
    """Faces and vertices of the triangles p [n, 3, 3] (three vertices of their own each)."""
    n = len(p)
    verts = np.zeros(3 * n, abi.VERTEX_DTYPE)
    verts["xyz"] = p.reshape(-1, 3).astype(np.float32)
    faces = np.zeros(n, abi.FACE_DTYPE)
    faces["v"] = np.arange(3 * n, dtype=np.uint32).reshape(-1, 3)
    faces["normal"] = normals(verts["xyz"].reshape(-1, 3, 3))
    faces["color"] = colors
    return faces, verts


def buried_spheres(k, rng, centre=(0.0, -100.5, -1.0)):
    """k spheres of radius 0.3..1 with centres at y in [-80, -60] under `centre` (C1's ground sphere: radius 100)."""
    c = np.asarray(centre, np.float64)
    xyz = np.stack([c[0] + rng.uniform(-8, 8, k), rng.uniform(-80, -60, k), c[2] + rng.uniform(-8, 8, k)], 1)
    return np.concatenate([xyz, rng.uniform(0.3, 1.0, (k, 1))], 1).astype(np.float32)


def buried_triangles(k, rng, centre=(0.0, -100.5, -1.0)):
    """k triangles of about a unit across, as deep inside the ground sphere as buried_spheres."""
    c = np.asarray(centre, np.float64)
    mid = np.stack([c[0] + rng.uniform(-8, 8, k), rng.uniform(-80, -60, k), c[2] + rng.uniform(-8, 8, k)], 1)
    return (mid[:, None, :] + rng.uniform(-0.6, 0.6, (k, 3, 3))).astype(np.float32)


def assemble(faces_p, face_color, face_mat, spheres, sphere_color, sphere_mat, mats):
    """SceneArrays from triangle corners [nf, 3, 3] and spheres [ns, 4]; material arrays may be None (Lambertian in the colour)."""
    kw = {}
    if len(faces_p):
        kw["faces"], kw["vertices"] = triangles(np.asarray(faces_p, np.float32), np.asarray(face_color, np.float32))
        kw["face_entity"] = np.zeros(len(faces_p), np.uint32)
        if face_mat is not None:
            kw["face_material"] = np.asarray(face_mat, np.uint32)
    if len(spheres):
        kw["spheres"], kw["sphere_color"] = np.asarray(spheres, np.float32), np.asarray(sphere_color, np.float32)
        kw["sphere_entity"] = np.arange(len(spheres), dtype=np.uint32)
        if sphere_mat is not None:
            kw["sphere_material"] = np.asarray(sphere_mat, np.uint32)
    if mats is not None:
        kw["materials"] = mats
    return abi.SceneArrays(**kw)


def c1_padded(total, w, h, faces=0, seed=0):
    """C1 with buried padding up to `total` primitives: `faces` buried triangles first (ids 0..faces-1, a mixed scene), then
    C1's four spheres, then buried spheres."""
    rng = np.random.default_rng(seed)
    base, cam = scenes.rtiow_four_spheres(w, h)
    k = total - faces - 4
    assert k >= 0
    spheres = np.concatenate([base.spheres, buried_spheres(k, rng)])
    mat = np.concatenate([base.sphere_material, np.zeros(k, np.uint32)])
    col = np.concatenate([base.sphere_color, np.full((k, 3), 0.5, np.float32)])
    scene = assemble(buried_triangles(faces, rng), np.full((faces, 3), 0.5, np.float32), np.zeros(faces, np.uint32), spheres, col, mat, base.materials)
    return scene, cam


def c2_padded(total, w, h, seed=0):
    """C2's cover scene (ground sphere of radius 1000 at y = -1000) with buried spheres up to `total`."""
    rng = np.random.default_rng(seed)
    base, cam = scenes.rtiow_cover(w, h)
    k = total - base.n_spheres
    assert k >= 0
    xyz = np.stack([rng.uniform(-20, 20, k), rng.uniform(-80, -60, k), rng.uniform(-20, 20, k)], 1)
    extra = np.concatenate([xyz, rng.uniform(0.3, 1.0, (k, 1))], 1).astype(np.float32)
    scene = assemble([], [], None, np.concatenate([base.spheres, extra]), np.concatenate([base.sphere_color, np.full((k, 3), 0.5, np.float32)]),
                     np.concatenate([base.sphere_material, np.zeros(k, np.uint32)]), base.materials)
    return scene, cam


# C1's sphere ids: 0 ground, 1 the blue Lambertian in the middle, 2 glass, 3 metal
BLUE, METAL_MAT = 1, 3


def with_copies(total, w, h, original_at, copies_at, faces=0, seed=0):
    """C1 with its blue sphere at id `original_at` and bit-identical copies of it, in C1's metal, at the ids `copies_at`;
    the other three spheres take the lowest free sphere ids and buried padding the rest (`faces` buried triangles first).
    `copies_at=[]` gives the same scene without the copies (buried spheres in their places)."""
    rng = np.random.default_rng(seed)
    base, cam = scenes.rtiow_four_spheres(w, h)
    ns = total - faces
    spheres = buried_spheres(ns, rng)
    mat = np.zeros(ns, np.uint32)
    col = np.full((ns, 3), 0.5, np.float32)
    taken = {original_at - faces} | {c - faces for c in copies_at}
    assert min(taken) >= 0 and max(taken) < ns and len(taken) == 1 + len(copies_at)
    free = iter(i for i in range(ns) if i not in taken)
    for src in (0, 2, 3):
        i = next(free)
        spheres[i], mat[i], col[i] = base.spheres[src], base.sphere_material[src], base.sphere_color[src]
    spheres[original_at - faces], mat[original_at - faces], col[original_at - faces] = base.spheres[BLUE], BLUE, base.sphere_color[BLUE]
    for c in copies_at:
        spheres[c - faces], mat[c - faces], col[c - faces] = base.spheres[BLUE], METAL_MAT, base.materials[METAL_MAT]["albedo"]
    scene = assemble(buried_triangles(faces, rng), np.full((faces, 3), 0.5, np.float32), np.zeros(faces, np.uint32), spheres, col, mat, base.materials)
    return scene, cam


# (total, original id, copy ids, buried faces): a copy straddling a word edge (31 | 32), a chunk edge (511 | 512), the bank
# (767 of 768 resident, 768 of 769 streamed) and a tile edge (1023 | 1024), in sphere-only and in mixed scenes, and 53 coincident
# spheres (one original, 52 copies) in a resident sphere scene, more than the 48 candidates a BEAM chunk list holds; the other
# three spheres come after the crowd there, so a truncated list would lose them
TIE_CASES = {
    "word": (40, 31, [32], 0),
    "word_last_id": (40, 1, [31], 0),
    "chunk": (520, 511, [512], 0),
    "chunk_last_id": (520, 1, [511], 0),
    "bank_resident": (768, 1, [767], 0),
    "bank_streamed": (769, 1, [768], 0),
    "tile": (1032, 1023, [1024], 0),
    "tile_last_id": (1032, 1, [1023], 0),
    "mixed_word": (48, 31, [32], 20),
    "mixed_chunk": (700, 511, [512], 300),
    "mixed_tile": (1100, 1023, [1024], 600),
    "beam_overflow": (56, 0, list(range(1, 53)), 0),
}


def tie_scene(name, w, h):
    total, orig, copies, faces = TIE_CASES[name]
    return with_copies(total, w, h, orig, copies, faces=faces), with_copies(total, w, h, orig, [], faces=faces)[0]


def ladder_split(n, form):
    """(n_faces, n_spheres) of ladder count n: sphere-only, or the largest FACE_SPLITS boundary below n (half the scene when
    none is)."""
    if form == "spheres":
        return 0, n
    below = [s for s in FACE_SPLITS if s < n]
    nf = below[-1] if below else max(1, n // 2)
    return nf, n - nf


def ladder_scene(n, form, w, h, seed=0):
    """n primitives a ray can reach in front of the camera: a ground sphere (the first sphere) under random triangles and
    spheres in the box [-3, 3] x [-1, 2] x [-9, -2]; random materials (all three kinds) for "mixed_materials", Lambertian in
    the primitive's colour otherwise. Primitives shrink as n grows so the last ids stay visible."""
    rng = np.random.default_rng(1000 * seed + n + 7 * FORMS.index(form))
    nf, ns = ladder_split(n, form)
    size = 0.6 * min(1.0, (16.0 / n) ** 0.5) + 0.05
    mid = rng.uniform([-3, -1, -9], [3, 2, -2], (nf, 1, 3))
    faces_p = (mid + rng.normal(0, size, (nf, 3, 3))).astype(np.float32)
    spheres = np.concatenate([rng.uniform([-3, -1, -9], [3, 2, -2], (ns, 3)), rng.uniform(0.3, 1.0, (ns, 1)) * size], 1).astype(np.float32)
    if ns:
        spheres[0] = (0, -1001.2, -5, 1000)
    mats = None
    fm = sm = None
    if form == "mixed_materials":
        mats = np.zeros(6, abi.MATERIAL_DTYPE)
        mats["kind"] = [abi.MAT_LAMBERTIAN, abi.MAT_METAL, abi.MAT_DIELECTRIC, abi.MAT_METAL, abi.MAT_LAMBERTIAN, abi.MAT_DIELECTRIC]
        mats["albedo"] = rng.uniform(0.2, 0.95, (6, 3))
        mats["fuzz"] = [0, 0.3, 0, 0.0, 0, 0]
        mats["ior"] = [1, 1, 1.5, 1, 1, 1.33]
        fm, sm = rng.integers(0, 6, nf), rng.integers(0, 6, ns)
    scene = assemble(faces_p, rng.uniform(0.1, 1, (nf, 3)), fm, spheres, rng.uniform(0.1, 1, (ns, 3)), sm, mats)
    cam = abi.reference_camera(w, h, focal_length=1.0)
    return scene, cam


# how the GPU half renders each scene: (name, RT3_FLAG_BVH, environment)
SWEEP, NO_BEAM, BVH = ("sweep", False, {}), ("no_beam", False, {"RT3_BEAM": "0"}), ("bvh", True, {})
TIE_MODES = [SWEEP, NO_BEAM, BVH, ("bvh_beam0", True, {"RT3_BEAM_BVH": "0"}), ("bvh_beam1", True, {"RT3_BEAM_BVH": "1"})]
BIN_MODES = [(f"bin{b}" + ("_beam1" if beam else ""), True, {"RT3_BINNING": str(b), **({"RT3_BEAM_BVH": "1"} if beam else {})})
             for b in range(4) for beam in (False, True)]
LADDER_W, LADDER_H, LADDER_SPP, LADDER_DEPTH = 40, 24, 4, 8
BIN_FACES, BIN_SPP = [1023, 1024], [8, 9]


def ladder_modes(n, form):
    """The sweep and the hierarchy, and the plain sweep too where the sweep's default is the BEAM kernel."""
    nf, ns = ladder_split(n, form)
    return [SWEEP, BVH] + ([NO_BEAM] if kernel_for(nf, ns, LADDER_SPP, False)[4] else [])


def planned_kernels():
    """{instantiation: [case, ...]} over every render of tests/test_gpu_pathtrace_edges.py's ladder, tie and binning tests."""
    reached = {}
    for n in LADDER:
        for form in FORMS:
            nf, ns = ladder_split(n, form)
            for mode, bvh, env in ladder_modes(n, form):
                reached.setdefault(kernel_for(nf, ns, LADDER_SPP, bvh, env), []).append(f"ladder {form} {n} {mode}")
    for name, (total, _, _, faces) in TIE_CASES.items():
        for mode, bvh, env in TIE_MODES:
            reached.setdefault(kernel_for(faces, total - faces, LADDER_SPP, bvh, env), []).append(f"tie {name} {mode}")
    for nf in BIN_FACES:
        for spp in BIN_SPP:
            for mode, bvh, env in [BVH] + BIN_MODES:
                reached.setdefault(kernel_for(nf, 2, spp, bvh, env), []).append(f"mesh {nf} faces {spp} spp {mode}")
    return reached


def thin_lens(cam, radius=0.05):
    cam.lens_radius = radius
    cam.lens_u[:] = [1, 0, 0]
    cam.lens_v[:] = [0, 1, 0]
    return cam


def pt(w, h, spp, depth=8, seed=3, flags=0, **kw):
    return abi.make_params(w, h, mode=abi.MODE_PATHTRACE, spp=spp, max_depth=depth, seed=seed, flags=flags, **kw)
