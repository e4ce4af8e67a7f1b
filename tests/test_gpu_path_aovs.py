"""rt3_render_path_aovs on the GPU: bit for bit against the CPU restatement (tests/path_aov_oracle.c) over scenes, cameras,
flags, sample ranges and partitions; sweep == hierarchy; agreement with the path kernel itself; the progressive state left
alone; real shapes on row bands; the host backend and its command line."""
import os
import subprocess

import numpy as np
import pytest

import fullsize as fs
import path_aov_lib as pal
from rt3_b200 import abi, scenes

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
W, H = 40, 24
FLAGS = {"none": 0, "no_jitter": abi.FLAG_NO_JITTER, "uniform_sky": abi.FLAG_UNIFORM_SKY, "bvh": abi.FLAG_BVH}
# (spp, first_sample, partitioned): every spp of 1, 7, 64, both first samples, one partition and three of tile_rows = 2
CASES = [(1, 0, False), (7, 100, True), (64, 0, True), (64, 100, False)]


def make_scene(name):
    if name == "c1":                                     # Lambertian, metal and dielectric
        return scenes.rtiow_four_spheres(W, H)[0]
    if name in ("mixed", "mixed_face_materials"):        # triangles and spheres, with and without per-face materials
        from test_gpu_reference_mode import random_soup
        rng = np.random.default_rng(11)
        soup = random_soup(rng, 200, 30)
        mats = np.zeros(4, abi.MATERIAL_DTYPE)
        mats["kind"] = [0, 1, 2, 0]
        mats["albedo"] = rng.uniform(0.2, 0.95, (4, 3))
        mats["ior"] = [1, 1, 1.5, 1]
        fm = rng.integers(0, 4, soup.n_faces).astype(np.uint32) if name == "mixed_face_materials" else None
        return abi.SceneArrays(faces=soup.faces, vertices=soup.vertices, face_entity=soup.face_entity, face_material=fm,
                               spheres=soup.spheres, sphere_color=soup.sphere_color, sphere_entity=soup.sphere_entity,
                               sphere_material=rng.integers(0, 4, soup.n_spheres).astype(np.uint32), materials=mats)
    if name == "cloud":                                  # more than RT3_CONST_PRIMS: the streamed sweep
        scene = scenes.random_spheres(1500, seed=91, width=W, height=H)[0]
        scene.spheres[:, :3] *= np.float32(0.05)
        scene.spheres[:, 3] *= np.float32(0.5)
        return scene
    if name == "mesh":                                   # a tessellated sphere (2 400 faces) in front of an analytic one
        ctx = abi.Context(0)
        mesh = ctx.tessellate_spheres([((0.3, 0.1, -3), 1.0, 40, 31, (0.8, 0.3, 0.3), 5)])
        ctx.close()
        return abi.SceneArrays(faces=mesh.faces, vertices=mesh.vertices, face_entity=mesh.face_entity,
                               spheres=np.array([[-1.2, -0.4, -4, 1.0]], np.float32), sphere_color=np.array([[0.2, 0.6, 0.9]], np.float32))
    raise KeyError(name)


def camera(lens):
    cam = abi.reference_camera(W, H)
    if lens:
        cam.lens_radius = 0.08
        cam.lens_u[:] = [1, 0, 0]
        cam.lens_v[:] = [0, 1, 0]
    return cam


_scenes = {}


def scene_of(name):
    if name not in _scenes:
        _scenes[name] = make_scene(name)
    return _scenes[name]


def gpu_aovs(ctx, cam, params, partitioned):
    if not partitioned:
        return ctx.render_path_aovs(cam, params)
    out = pal.empty_aovs(params.height, params.width)
    for i in range(3):
        p = abi.make_params(params.width, params.height, mode=abi.MODE_PATHTRACE, spp=params.spp, max_depth=params.max_depth, seed=params.seed,
                            flags=params.flags, tile_rows=2, part_index=i, part_count=3, first_sample=params.first_sample)
        part = ctx.render_path_aovs(cam, p)
        owned = (np.arange(params.height) // 2) % 3 == i
        for k in pal.AOV_KEYS:
            assert (part[k][~owned] == 0).all(), f"{k}: rows of other partitions written"
            out[k][owned] = part[k][owned]
    return out


def assert_equal(gpu, cpu, what):
    for k in pal.AOV_KEYS:
        a, b = gpu[k].view(np.uint32), cpu[k].view(np.uint32)
        bad = int((a != b).sum())
        assert bad == 0, f"{what}: {k} differs from the oracle in {bad} values"


@pytest.mark.parametrize("flag", list(FLAGS))
@pytest.mark.parametrize("lens", [False, True], ids=["pinhole", "thin_lens"])
@pytest.mark.parametrize("name", ["c1", "mixed", "mixed_face_materials", "cloud", "mesh"])
def test_equals_the_oracle(gpu_ctx, name, lens, flag):
    scene, cam = scene_of(name), camera(lens)
    gpu_ctx.upload(scene)
    for spp, first, partitioned in CASES:
        params = abi.make_params(W, H, mode=abi.MODE_PATHTRACE, spp=spp, max_depth=5, seed=9, flags=FLAGS[flag], first_sample=first)
        gpu = gpu_aovs(gpu_ctx, cam, params, partitioned)
        st = gpu_ctx.stats()
        if not partitioned:
            assert st.rays == W * H * spp and st.kernel_launches == 2 and st.accel == (1 if flag == "bvh" else 0)
        assert_equal(gpu, pal.oracle_path_aovs(scene, cam, params), f"{name} spp {spp} first {first} partitioned {partitioned}")


@pytest.mark.parametrize("name", ["c1", "mixed_face_materials", "cloud", "mesh"])
def test_sweep_and_hierarchy_agree(gpu_ctx, name):
    gpu_ctx.upload(scene_of(name))
    for lens in (False, True):
        params = abi.make_params(W, H, mode=abi.MODE_PATHTRACE, spp=33, max_depth=1, seed=2)
        sweep = gpu_ctx.render_path_aovs(camera(lens), params)
        params.flags = abi.FLAG_BVH
        tree = gpu_ctx.render_path_aovs(camera(lens), params)
        assert gpu_ctx.stats().accel_node_visits > 0
        for k in pal.AOV_KEYS:
            assert np.array_equal(sweep[k].view(np.uint32), tree[k].view(np.uint32)), k


@pytest.mark.parametrize("name", ["c1", "mixed", "cloud"])
def test_misses_are_where_the_path_kernel_sees_the_sky(gpu_ctx, name):
    """No oracle: at spp 1 and depth 1 under a white sky, a beauty pixel is white exactly where its one primary ray missed."""
    gpu_ctx.upload(scene_of(name))
    cam = camera(True)
    params = abi.make_params(W, H, mode=abi.MODE_PATHTRACE, spp=1, max_depth=1, seed=4, flags=abi.FLAG_UNIFORM_SKY | abi.FLAG_NO_GAMMA, first_sample=17)
    frame = gpu_ctx.render(cam, params)
    aovs = gpu_ctx.render_path_aovs(cam, params)
    assert np.array_equal(frame == 0xFFFFFFFF, aovs["hit_prim"] == abi.NO_HIT)
    assert np.array_equal(frame != 0xFFFFFFFF, frame == 0x000000FF)


def test_progressive_state_is_left_alone(gpu_ctx):
    scene, cam = scenes.rtiow_four_spheres(W, H)
    gpu_ctx.upload(scene)
    k = 6
    first = abi.make_params(W, H, mode=abi.MODE_PATHTRACE, spp=k, max_depth=8, seed=5)
    gpu_ctx.render(cam, first)
    radiance = gpu_ctx.read_radiance(W, H)
    gpu_ctx.render_path_aovs(cam, abi.make_params(W, H, mode=abi.MODE_PATHTRACE, spp=3, max_depth=8, seed=5, flags=abi.FLAG_BVH, tile_rows=2,
                                                  part_index=1, part_count=2))
    assert np.array_equal(gpu_ctx.read_radiance(W, H), radiance)
    more = gpu_ctx.render(cam, abi.make_params(W, H, mode=abi.MODE_PATHTRACE, spp=k, max_depth=8, seed=5, flags=abi.FLAG_ACCUMULATE, first_sample=k))
    once = gpu_ctx.render(cam, abi.make_params(W, H, mode=abi.MODE_PATHTRACE, spp=2 * k, max_depth=8, seed=5))
    assert np.array_equal(more, once)


def test_rejects_reference_mode(gpu_ctx):
    scene, cam = scenes.rtiow_four_spheres(W, H)
    gpu_ctx.upload(scene)
    with pytest.raises(abi.Rt3Error, match="PATHTRACE"):
        gpu_ctx.render_path_aovs(cam, abi.make_params(W, H))


@pytest.mark.parametrize("name,row,spp,flags", [("c2", 400, 500, 0), ("c5", 540, 64, abi.FLAG_BVH)])
def test_real_shapes_on_a_row_band(gpu_ctx, name, row, spp, flags):
    """A row of the full-size frame (one-row partition, tests/fullsize.py) at the AOV sample count, against the oracle.
    C5 renders without jitter through a pinhole, so its 64 samples of a pixel are one ray: the oracle traces it once."""
    c = fs.CONFIGS[name]
    scene, cam = c["scene"](c["w"], c["h"])
    gpu_ctx.upload(scene)
    gpu = gpu_ctx.render_path_aovs(cam, fs.params_for(c, flags, spp=spp, tile_rows=1, part_index=row, part_count=c["h"]))
    oracle_spp = 1 if name == "c5" else spp
    assert name != "c5" or (c["flags"] & abi.FLAG_NO_JITTER and cam.lens_radius == 0)
    cpu = pal.oracle_path_aovs(scene, cam, fs.params_for(c, spp=oracle_spp, tile_rows=1, part_index=row, part_count=c["h"]))
    assert (gpu["hit_prim"][row] != abi.NO_HIT).any()
    assert_equal({k: v[row] for k, v in gpu.items()}, {k: v[row] for k, v in cpu.items()}, name)


def host_rtiow(w, h, multi):
    import hostlib
    hs = hostlib.HostScene()
    for centre, radius, colour in (((0, -100.5, -1), 100, (0.8, 0.8, 0)), ((0, 0, -1), 0.5, (0.1, 0.2, 0.5)), ((-1, 0, -1), 0.5, (1, 1, 1)),
                                   ((1, 0, -1), 0.5, (0.8, 0.6, 0.2))):
        hs.add_sphere(centre, radius, 8, 8, colour)
    if multi:
        hs.create_renderer_multi([0, 0, 0], mode=abi.MODE_PATHTRACE, spp=8, max_depth=10, seed=1, analytic_spheres=True, tile_rows=2)
    else:
        hs.create_renderer(0, mode=abi.MODE_PATHTRACE, spp=8, max_depth=10, seed=1, analytic_spheres=True)
    hs.set_material(2, abi.MAT_DIELECTRIC, ior=1.5)
    hs.set_material(3, abi.MAT_METAL, albedo=(0.8, 0.6, 0.2))
    hs.prerender()
    return hs


def test_host_backend_and_command_line(built, tmp_path):
    """CudaRenderer::render_path_aovs: one context and the same GPU listed three times give the same arrays; rt3_render --aov
    writes PFMs (albedo, normal, depth) that read back equal to them."""
    w, h = 64, 36
    one = pal.host_path_aovs(host_rtiow(w, h, False), w, h, 5, focal=1.0)
    three = pal.host_path_aovs(host_rtiow(w, h, True), w, h, 5, focal=1.0, pfm_dir=tmp_path)
    for k in pal.AOV_KEYS:
        assert np.array_equal(one[k].view(np.uint32), three[k].view(np.uint32)), k
    assert (one["hit_prim"] != abi.NO_HIT).any() and (one["hit_prim"] == abi.NO_HIT).any()
    exe = os.path.join(ROOT, "raytracer-3_b200", "host", "rt3_render")
    env = dict(os.environ)
    env.pop("RT3_DEVICES", None)
    out = tmp_path / "cli"
    out.mkdir()
    subprocess.run([exe, "-s", "rtiow", "-W", str(w), "-H", str(h), "--spp", "8", "--depth", "10", "-o", str(tmp_path / "f.ppm"), "--aov", str(out),
                    "--aov-spp", "5"], check=True, env=env, stdout=subprocess.DEVNULL, timeout=120)
    for d in (out, tmp_path):
        assert np.array_equal(pal.read_pfm(str(d / "albedo.pfm")), one["albedo"])
        assert np.array_equal(pal.read_pfm(str(d / "normal.pfm")), one["normal"])
        assert np.array_equal(pal.read_pfm(str(d / "depth.pfm")).view(np.uint32), one["hit_t"].view(np.uint32))
