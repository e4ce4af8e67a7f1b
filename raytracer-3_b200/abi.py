"""ctypes view of the C ABI declared in include/rt3cuda.h.

Plumbing only: struct layouts, the loader for ``librt3cuda.so`` and thin
wrappers that turn a non-zero status into ``Rt3Error`` (the reference's
``DLOG(fatal, ...)`` -> ``CppDebugger::Fatal``, src/Main.cpp:305-308).
There is deliberately no CPU fallback: if the CUDA library is missing or no
device is present, loading / ``Context()`` raises.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# RT3_CORE_LIB selects another build of the same library (profiling variants under profiles/); there is still no CPU path
CORE_LIB_PATH = os.environ.get("RT3_CORE_LIB") or os.path.join(_HERE, "csrc", "librt3cuda.so")

MAT_LAMBERTIAN, MAT_METAL, MAT_DIELECTRIC = 0, 1, 2
MODE_REFERENCE, MODE_PATHTRACE = 0, 1
FLAG_NO_JITTER, FLAG_NO_GAMMA, FLAG_BVH, FLAG_ACCUMULATE, FLAG_UNIFORM_SKY = 0x1, 0x2, 0x4, 0x8, 0x10
NO_HIT = 0xFFFFFFFF
IPC_HANDLE_BYTES = 64  # RT3_IPC_HANDLE_BYTES

# numpy record layouts that mirror rt3_face (GFace, reference Vertex.hpp:39-51),
# rt3_vertex (glm::vec4) and rt3_material byte for byte.
FACE_DTYPE = np.dtype({
    "names": ["v", "normal", "color"],
    "formats": [("<u4", 3), ("<f4", 3), ("<f4", 3)],
    "offsets": [0, 16, 32],
    "itemsize": 48,
})
VERTEX_DTYPE = np.dtype([("xyz", "<f4", 3), ("w", "<f4")])
MATERIAL_DTYPE = np.dtype({
    "names": ["kind", "albedo", "fuzz", "ior"],
    "formats": ["<u4", ("<f4", 3), "<f4", "<f4"],
    "offsets": [0, 4, 16, 20],
    "itemsize": 32,
})


class Rt3Error(RuntimeError):
    pass


class Scene(C.Structure):
    _fields_ = [
        ("n_faces", C.c_uint32), ("n_vertices", C.c_uint32),
        ("faces", C.c_void_p), ("vertices", C.c_void_p),
        ("face_material", C.c_void_p), ("face_entity", C.c_void_p),
        ("n_spheres", C.c_uint32), ("n_materials", C.c_uint32),
        ("spheres", C.c_void_p), ("sphere_color", C.c_void_p),
        ("sphere_material", C.c_void_p), ("sphere_entity", C.c_void_p),
        ("materials", C.c_void_p),
    ]


class Camera(C.Structure):
    _fields_ = [
        ("origin", C.c_float * 3), ("horizontal", C.c_float * 3),
        ("vertical", C.c_float * 3), ("lower_left_corner", C.c_float * 3),
        ("lens_radius", C.c_float), ("lens_u", C.c_float * 3), ("lens_v", C.c_float * 3),
    ]


class UvSphere(C.Structure):
    _fields_ = [("center", C.c_float * 3), ("radius", C.c_float), ("n_meridians", C.c_uint32), ("n_parallels", C.c_uint32),
                ("color", C.c_float * 3), ("entity", C.c_uint32)]


class Params(C.Structure):
    _fields_ = [
        ("width", C.c_uint32), ("height", C.c_uint32), ("mode", C.c_uint32),
        ("spp", C.c_uint32), ("max_depth", C.c_uint32), ("seed", C.c_uint32),
        ("flags", C.c_uint32), ("tile_rows", C.c_uint32),
        ("part_index", C.c_uint32), ("part_count", C.c_uint32), ("first_sample", C.c_uint32),
    ]


class Stats(C.Structure):
    _fields_ = [
        ("device_ms", C.c_double), ("trace_kernel_ms", C.c_double), ("h2d_ms", C.c_double), ("d2h_ms", C.c_double),
        ("rays", C.c_uint64), ("sphere_tests", C.c_uint64), ("face_tests", C.c_uint64),
        ("kernel_launches", C.c_uint32), ("rows_rendered", C.c_uint32),
        ("accel_node_visits", C.c_uint64), ("accel_prim_tests", C.c_uint64), ("accel_build_ms", C.c_double),
        ("accel", C.c_uint32), ("accel_stack_overflows", C.c_uint32),
        ("upload_ms", C.c_double), ("upload_device_ms", C.c_double),
        ("beam_rays", C.c_uint64), ("beam_tests", C.c_uint64),
    ]


class PathAovs(C.Structure):
    """rt3_path_aovs: host output pointers of rt3_render_path_aovs (any may be NULL)."""
    _fields_ = [("hit_prim", C.c_void_p), ("hit_entity", C.c_void_p), ("hit_t", C.c_void_p), ("albedo", C.c_void_p), ("normal", C.c_void_p)]


class DenoiseParams(C.Structure):
    """rt3_denoise_params."""
    _fields_ = [("width", C.c_uint32), ("height", C.c_uint32), ("iterations", C.c_uint32), ("sigma_luminance", C.c_float), ("sigma_normal", C.c_float), ("sigma_depth", C.c_float)]


def denoise_params(width=0, height=0, iterations=5, sigma_luminance=4.0, sigma_normal=128.0, sigma_depth=1.0):
    """rt3_denoise_params with SVGF's defaults."""
    return DenoiseParams(width, height, iterations, sigma_luminance, sigma_normal, sigma_depth)


class DenoiseTemporalParams(C.Structure):
    """rt3_denoise_temporal_params."""
    _fields_ = [("filter", DenoiseParams), ("alpha_color", C.c_float), ("alpha_moments", C.c_float), ("depth_tolerance", C.c_float),
                ("normal_cos", C.c_float), ("reset", C.c_uint32)]


def denoise_temporal_params(width=0, height=0, reset=False, alpha_color=0.2, alpha_moments=0.2, depth_tolerance=0.05, normal_cos=0.9, **filter):
    """rt3_denoise_temporal_params with SVGF's defaults; ``filter`` takes denoise_params' keywords."""
    return DenoiseTemporalParams(denoise_params(width, height, **filter), alpha_color, alpha_moments, depth_tolerance, normal_cos, 1 if reset else 0)


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class SceneArrays:
    """Host-side flattened scene: the arrays behind an ``rt3_scene``.

    faces / vertices are in the reference's flattened layout
    (SequentialRenderer.cpp:174-195); spheres are analytic (cx, cy, cz, r).
    Keeps the numpy arrays alive for as long as the ctypes struct is used.
    """

    def __init__(self, faces=None, vertices=None, face_material=None, face_entity=None,
                 spheres=None, sphere_color=None, sphere_material=None, sphere_entity=None, materials=None):
        def arr(a, dtype, shape=None):
            if a is None:
                return None
            a = np.ascontiguousarray(a, dtype=dtype)
            return a if shape is None else a.reshape(shape)
        self.faces = arr(faces, FACE_DTYPE) if faces is not None else np.zeros(0, FACE_DTYPE)
        self.vertices = arr(vertices, VERTEX_DTYPE) if vertices is not None else np.zeros(0, VERTEX_DTYPE)
        self.face_material = arr(face_material, np.uint32)
        self.face_entity = arr(face_entity, np.uint32)
        self.spheres = arr(spheres, np.float32, (-1, 4)) if spheres is not None else np.zeros((0, 4), np.float32)
        self.sphere_color = arr(sphere_color, np.float32, (-1, 3))
        if self.sphere_color is None:
            self.sphere_color = np.ones((len(self.spheres), 3), np.float32)
        self.sphere_material = arr(sphere_material, np.uint32)
        self.sphere_entity = arr(sphere_entity, np.uint32)
        self.materials = arr(materials, MATERIAL_DTYPE) if materials is not None else np.zeros(0, MATERIAL_DTYPE)
        assert len(self.sphere_color) == len(self.spheres)
        for opt, n in ((self.face_material, len(self.faces)), (self.face_entity, len(self.faces)),
                       (self.sphere_material, len(self.spheres)), (self.sphere_entity, len(self.spheres))):
            assert opt is None or len(opt) == n

    @property
    def n_faces(self):
        return len(self.faces)

    @property
    def n_spheres(self):
        return len(self.spheres)

    def as_struct(self):
        s = Scene()
        s.n_faces, s.n_vertices = len(self.faces), len(self.vertices)
        s.faces, s.vertices = _ptr(self.faces), _ptr(self.vertices)
        s.face_material, s.face_entity = _ptr(self.face_material), _ptr(self.face_entity)
        s.n_spheres, s.n_materials = len(self.spheres), len(self.materials)
        s.spheres, s.sphere_color = _ptr(self.spheres), _ptr(self.sphere_color)
        s.sphere_material, s.sphere_entity = _ptr(self.sphere_material), _ptr(self.sphere_entity)
        s.materials = _ptr(self.materials)
        return s


def make_camera(origin, horizontal, vertical, lower_left_corner, lens_radius=0.0, lens_u=(0, 0, 0), lens_v=(0, 0, 0)):
    cam = Camera()
    for name, v in (("origin", origin), ("horizontal", horizontal), ("vertical", vertical),
                    ("lower_left_corner", lower_left_corner), ("lens_u", lens_u), ("lens_v", lens_v)):
        setattr(cam, name, (C.c_float * 3)(*[float(np.float32(c)) for c in v]))
    cam.lens_radius = float(lens_radius)
    return cam


def reference_camera(width, height, focal_length=2.0, viewport_height=2.0, viewport_width=None):
    """The camera Camera::update builds (reference camera/Camera.cpp:77-96), in fp32.

    Main.cpp:272 calls it with viewport_width = (W/H)*2, viewport_height = 2, focal 2.
    """
    f = np.float32
    if viewport_width is None:
        viewport_width = f(f(width) / f(height)) * f(2.0)
    vw, vh, fl = f(viewport_width), f(viewport_height), f(focal_length)
    origin = np.zeros(3, f)
    hor = np.array([vw, 0, 0], f)
    ver = np.array([0, vh, 0], f)
    llc = ((origin - hor / f(2.0)) - ver / f(2.0)) - np.array([0, 0, fl], f)
    return make_camera(origin, hor, ver, llc)


def make_params(width, height, mode=MODE_REFERENCE, spp=1, max_depth=1, seed=0, flags=0,
                tile_rows=8, part_index=0, part_count=1, first_sample=0):
    return Params(width, height, mode, spp, max_depth, seed, flags, tile_rows, part_index, part_count, first_sample)


_core = None


def load_core():
    """Loads librt3cuda.so (built by __graft_entry__.build()). Raises if absent."""
    global _core
    if _core is not None:
        return _core
    if not os.path.exists(CORE_LIB_PATH):
        raise Rt3Error(f"{CORE_LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'`. "
                       "There is no CPU fallback for the render core.")
    lib = C.CDLL(CORE_LIB_PATH)
    vp, u32, u32p = C.c_void_p, C.c_uint32, C.c_void_p
    lib.rt3_last_error.restype = C.c_char_p
    lib.rt3_create.argtypes = [C.POINTER(vp), C.c_int]
    lib.rt3_destroy.argtypes = [vp]
    lib.rt3_scene_upload.argtypes = [vp, C.POINTER(Scene)]
    lib.rt3_scene_upload_device.argtypes = [vp, C.POINTER(Scene)]
    lib.rt3_buffer_alloc.argtypes = [vp, C.c_uint64, C.POINTER(vp)]
    lib.rt3_buffer_free.argtypes = [vp, vp]
    lib.rt3_buffer_write.argtypes = [vp, vp, vp, C.c_uint64]
    lib.rt3_buffer_read.argtypes = [vp, vp, vp, C.c_uint64]
    lib.rt3_tessellate_spheres_device.argtypes = [vp, C.POINTER(UvSphere), u32, u32, u32, vp, vp, vp]
    lib.rt3_render.argtypes = [vp, C.POINTER(Camera), C.POINTER(Params), u32p]
    lib.rt3_render_aov.argtypes = [vp, C.POINTER(Camera), C.POINTER(Params), u32p, u32p, u32p, vp]
    lib.rt3_render_path_aovs.argtypes = [vp, C.POINTER(Camera), C.POINTER(Params), C.POINTER(PathAovs)]
    lib.rt3_render_device.argtypes = [vp, C.POINTER(Camera), C.POINTER(Params), vp, vp]
    lib.rt3_partition_rows.argtypes = [u32, u32, u32, u32]
    lib.rt3_partition_rows.restype = u32
    lib.rt3_pack_partition.argtypes = [vp, vp, vp, u32, u32, u32, u32, u32, vp]
    lib.rt3_unpack_partition.argtypes = [vp, vp, vp, u32, u32, u32, u32, u32, vp]
    lib.rt3_frame_bytes.argtypes = [vp, vp, vp, u32, u32, u32, vp]
    lib.rt3_frame_alloc.argtypes = [vp, C.c_uint64, C.POINTER(vp)]
    lib.rt3_frame_free.argtypes = [vp, vp]
    lib.rt3_frame_export.argtypes = [vp, vp, C.c_char_p]
    lib.rt3_frame_import.argtypes = [vp, C.c_char_p, C.POINTER(vp)]
    lib.rt3_frame_release.argtypes = [vp, vp]
    lib.rt3_frame_attach.argtypes = [vp, vp]
    lib.rt3_frame_read.argtypes = [vp, vp, vp, C.c_uint64]
    lib.rt3_uv_sphere_faces.argtypes = [u32, u32]
    lib.rt3_uv_sphere_faces.restype = u32
    lib.rt3_uv_sphere_vertices.argtypes = [u32, u32]
    lib.rt3_uv_sphere_vertices.restype = u32
    lib.rt3_tessellate_spheres.argtypes = [vp, C.POINTER(UvSphere), u32, u32, vp, vp, vp]
    lib.rt3_read_radiance.argtypes = [vp, vp, u32, u32]
    lib.rt3_denoise.argtypes = [vp, C.POINTER(DenoiseParams), vp, vp]
    lib.rt3_denoise_temporal.argtypes = [vp, C.POINTER(DenoiseTemporalParams), vp, vp, vp]
    lib.rt3_denoise_stage_words.argtypes = [u32, u32]
    lib.rt3_denoise_stage_words.restype = C.c_uint64
    lib.rt3_denoise_stage.argtypes = [vp, C.POINTER(DenoiseParams), C.c_uint64, vp, vp]
    lib.rt3_denoise_staged.argtypes = [vp, C.POINTER(DenoiseParams), C.c_uint64, vp, vp, vp]
    lib.rt3_get_stats.argtypes = [vp, C.POINTER(Stats)]
    lib.rt3_measure_fma_peak.argtypes = [vp, C.POINTER(C.c_double)]
    _core = lib
    return lib


EXPORTED_SYMBOLS = [
    "rt3_last_error", "rt3_create", "rt3_destroy", "rt3_scene_upload", "rt3_scene_upload_device", "rt3_buffer_alloc", "rt3_buffer_free",
    "rt3_buffer_write", "rt3_buffer_read", "rt3_tessellate_spheres_device", "rt3_render", "rt3_render_aov",
    "rt3_render_path_aovs", "rt3_render_device", "rt3_partition_rows", "rt3_pack_partition", "rt3_unpack_partition", "rt3_frame_bytes",
    "rt3_frame_alloc", "rt3_frame_free", "rt3_frame_export", "rt3_frame_import", "rt3_frame_release",
    "rt3_frame_attach", "rt3_frame_read",
    "rt3_uv_sphere_faces", "rt3_uv_sphere_vertices", "rt3_tessellate_spheres",
    "rt3_read_radiance", "rt3_denoise", "rt3_denoise_temporal", "rt3_denoise_stage_words", "rt3_denoise_stage", "rt3_denoise_staged", "rt3_get_stats", "rt3_measure_fma_peak",
]


def denoise_stage_words(width, height):
    """rt3_denoise_stage_words: 32-bit words of the stage of a (width x height) frame rendered in parts (0: too large)."""
    return int(load_core().rt3_denoise_stage_words(width, height))


class Context:
    """One render context on one CUDA device (rt3_create .. rt3_destroy)."""

    def __init__(self, device=0):
        self.lib = load_core()
        self.handle = C.c_void_p()
        self._check(self.lib.rt3_create(C.byref(self.handle), int(device)))
        self._scene_keepalive = None

    def _check(self, status):
        if status != 0:
            raise Rt3Error(f"rt3 status {status}: {self.lib.rt3_last_error().decode()}")

    def close(self):
        if self.handle:
            self.lib.rt3_destroy(self.handle)
            self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def upload(self, scene: SceneArrays):
        st = scene.as_struct()
        self._check(self.lib.rt3_scene_upload(self.handle, C.byref(st)))

    def buffer_alloc(self, nbytes):
        p = C.c_void_p()
        self._check(self.lib.rt3_buffer_alloc(self.handle, nbytes, C.byref(p)))
        return p.value

    def buffer_free(self, ptr):
        self._check(self.lib.rt3_buffer_free(self.handle, C.c_void_p(ptr)))

    def buffer_write(self, ptr, array):
        a = np.ascontiguousarray(array)
        self._check(self.lib.rt3_buffer_write(self.handle, C.c_void_p(ptr), _ptr(a), a.nbytes))

    def buffer_read(self, ptr, array):
        self._check(self.lib.rt3_buffer_read(self.handle, _ptr(array), C.c_void_p(ptr), array.nbytes))
        return array

    def to_device(self, array):
        """A device copy of a host array (rt3_buffer_alloc + rt3_buffer_write); None stays None. The caller frees it."""
        if array is None or array.nbytes == 0:
            return None
        p = self.buffer_alloc(array.nbytes)
        self.buffer_write(p, array)
        return p

    def upload_device(self, n_faces=0, n_vertices=0, faces=None, vertices=None, face_material=None, face_entity=None,
                      n_spheres=0, spheres=None, sphere_color=None, sphere_material=None, sphere_entity=None, n_materials=0, materials=None):
        """rt3_scene_upload_device: every array argument is a DEVICE pointer (int) or None."""
        st = Scene()
        st.n_faces, st.n_vertices, st.n_spheres, st.n_materials = n_faces, n_vertices, n_spheres, n_materials
        st.faces, st.vertices, st.face_material, st.face_entity = faces, vertices, face_material, face_entity
        st.spheres, st.sphere_color, st.sphere_material, st.sphere_entity, st.materials = spheres, sphere_color, sphere_material, sphere_entity, materials
        self._check(self.lib.rt3_scene_upload_device(self.handle, C.byref(st)))

    def tessellate_spheres_device(self, spheres, first_vertex, first_face, faces_ptr, vertices_ptr, entity_ptr=None):
        """rt3_tessellate_spheres_device: the batch is written straight into the caller's device arrays."""
        arr = (UvSphere * len(spheres))()
        for dst, (center, radius, m, p, color, entity) in zip(arr, spheres):
            dst.center = (C.c_float * 3)(*center); dst.radius = radius; dst.n_meridians = m; dst.n_parallels = p
            dst.color = (C.c_float * 3)(*color); dst.entity = entity
        self._check(self.lib.rt3_tessellate_spheres_device(self.handle, arr, len(spheres), first_vertex, first_face, C.c_void_p(faces_ptr),
                                                           C.c_void_p(vertices_ptr), C.c_void_p(entity_ptr or 0)))

    def render(self, camera, params, out=None):
        """rt3_render into a host frame (numpy uint32 [H, W])."""
        if out is None:
            out = np.zeros((params.height, params.width), np.uint32)
        self._check(self.lib.rt3_render(self.handle, C.byref(camera), C.byref(params), _ptr(out)))
        return out

    def render_aov(self, camera, params):
        h, w = params.height, params.width
        frame = np.zeros((h, w), np.uint32)
        prim = np.zeros((h, w), np.uint32)
        ent = np.zeros((h, w), np.uint32)
        t = np.zeros((h, w), np.float32)
        self._check(self.lib.rt3_render_aov(self.handle, C.byref(camera), C.byref(params),
                                            _ptr(frame), _ptr(prim), _ptr(ent), _ptr(t)))
        return frame, prim, ent, t

    def render_path_aovs(self, camera, params):
        """rt3_render_path_aovs: AOVs of the path tracer's primary rays for pathtrace ``params`` (its spp = the AOV samples).

        Returns {"hit_prim", "hit_entity": uint32 [H, W], "hit_t": float32 [H, W], "albedo", "normal": float32 [H, W, 3]};
        rows of other partitions are 0."""
        h, w = params.height, params.width
        out = {"hit_prim": np.zeros((h, w), np.uint32), "hit_entity": np.zeros((h, w), np.uint32), "hit_t": np.zeros((h, w), np.float32),
               "albedo": np.zeros((h, w, 3), np.float32), "normal": np.zeros((h, w, 3), np.float32)}
        aovs = PathAovs(*(_ptr(out[k]) for k in ("hit_prim", "hit_entity", "hit_t", "albedo", "normal")))
        self._check(self.lib.rt3_render_path_aovs(self.handle, C.byref(camera), C.byref(params), C.byref(aovs)))
        return out

    def render_device(self, camera, params, device_ptr, stream_ptr=None):
        self._check(self.lib.rt3_render_device(self.handle, C.byref(camera), C.byref(params),
                                               C.c_void_p(device_ptr), C.c_void_p(stream_ptr or 0)))

    def pack_partition(self, frame_ptr, slab_ptr, width, height, tile_rows, part_index, part_count, stream_ptr=None):
        self._check(self.lib.rt3_pack_partition(self.handle, C.c_void_p(frame_ptr), C.c_void_p(slab_ptr), width, height,
                                                tile_rows, part_index, part_count, C.c_void_p(stream_ptr or 0)))

    def unpack_partition(self, slab_ptr, frame_ptr, width, height, tile_rows, part_index, part_count, stream_ptr=None):
        self._check(self.lib.rt3_unpack_partition(self.handle, C.c_void_p(slab_ptr), C.c_void_p(frame_ptr), width, height,
                                                  tile_rows, part_index, part_count, C.c_void_p(stream_ptr or 0)))

    def tessellate_spheres(self, spheres, first_vertex=0):
        """rt3_tessellate_spheres: [(center, radius, n_meridians, n_parallels, color, entity), ...] -> SceneArrays (faces, vertices)."""
        arr = (UvSphere * len(spheres))()
        for dst, (center, radius, m, p, color, entity) in zip(arr, spheres):
            dst.center = (C.c_float * 3)(*center); dst.radius = radius; dst.n_meridians = m; dst.n_parallels = p
            dst.color = (C.c_float * 3)(*color); dst.entity = entity
        nf = sum(self.lib.rt3_uv_sphere_faces(s[2], s[3]) for s in spheres)
        nv = sum(self.lib.rt3_uv_sphere_vertices(s[2], s[3]) for s in spheres)
        faces, verts, ent = np.zeros(nf, FACE_DTYPE), np.zeros(nv, VERTEX_DTYPE), np.zeros(nf, np.uint32)
        self._check(self.lib.rt3_tessellate_spheres(self.handle, arr, len(spheres), first_vertex, _ptr(faces), _ptr(verts), _ptr(ent)))
        return SceneArrays(faces=faces, vertices=verts, face_entity=ent)

    def frame_bytes(self, frame_ptr, out_ptr, width, height, channels, stream_ptr=None):
        """rt3_frame_bytes: packed device frame -> interleaved RGB (3) / RGBA (4) bytes on the device."""
        self._check(self.lib.rt3_frame_bytes(self.handle, C.c_void_p(frame_ptr), C.c_void_p(out_ptr), width, height, channels,
                                             C.c_void_p(stream_ptr or 0)))

    def frame_alloc(self, n_pixels):
        """rt3_frame_alloc: a zeroed frame of n_pixels packed pixels on this context's GPU (exportable); returns the device pointer."""
        p = C.c_void_p()
        self._check(self.lib.rt3_frame_alloc(self.handle, n_pixels, C.byref(p)))
        return p.value

    def frame_free(self, ptr):
        self._check(self.lib.rt3_frame_free(self.handle, C.c_void_p(ptr)))

    def frame_export(self, ptr):
        """rt3_frame_export: the IPC handle (bytes) another process maps with frame_import."""
        buf = C.create_string_buffer(IPC_HANDLE_BYTES)
        self._check(self.lib.rt3_frame_export(self.handle, C.c_void_p(ptr), buf))
        return buf.raw

    def frame_import(self, handle):
        """rt3_frame_import: maps another process's frame; the returned pointer is a valid `device_frame` for render_device."""
        if len(handle) != IPC_HANDLE_BYTES:
            raise ValueError(f"an IPC handle is {IPC_HANDLE_BYTES} bytes, got {len(handle)}")
        p = C.c_void_p()
        self._check(self.lib.rt3_frame_import(self.handle, handle, C.byref(p)))
        return p.value

    def frame_release(self, ptr):
        self._check(self.lib.rt3_frame_release(self.handle, C.c_void_p(ptr)))

    def frame_attach(self, owner):
        """rt3_frame_attach: this context's GPU may store into frames allocated by ``owner`` (same process)."""
        self._check(self.lib.rt3_frame_attach(self.handle, owner.handle))

    def frame_read(self, ptr, width, height):
        """rt3_frame_read: blocking copy of a device frame into a new (height, width) uint32 array."""
        out = np.zeros((height, width), np.uint32)
        self._check(self.lib.rt3_frame_read(self.handle, C.c_void_p(ptr), _ptr(out), width * height))
        return out

    def read_radiance(self, width, height):
        """rt3_read_radiance: mean linear radiance of the last path-traced render, (height, width, 3) float32."""
        out = np.zeros((height, width, 3), np.float32)
        self._check(self.lib.rt3_read_radiance(self.handle, _ptr(out), width, height))
        return out

    def denoise(self, width, height, **filter):
        """rt3_denoise: the last path-traced render of this (width x height) frame, filtered under the guidance of the last
        render_path_aovs; ``filter`` takes denoise_params' keywords. Returns (frame [H, W] uint32 packed like render's, rgb
        [H, W, 3] float32 linear)."""
        frame = np.zeros((height, width), np.uint32)
        rgb = np.zeros((height, width, 3), np.float32)
        p = denoise_params(width, height, **filter)
        self._check(self.lib.rt3_denoise(self.handle, C.byref(p), _ptr(frame), _ptr(rgb)))
        return frame, rgb

    def denoise_temporal(self, width, height, reset=False, alpha_color=0.2, alpha_moments=0.2, depth_tolerance=0.05, normal_cos=0.9, **filter):
        """rt3_denoise_temporal: ``denoise`` with the context's history of earlier frames reprojected through the camera's motion
        and accumulated (``reset`` drops it first); ``filter`` takes denoise_params' keywords. Render each frame with its own seed.
        Returns (frame [H, W] uint32, rgb [H, W, 3] float32, history_length [H, W] float32)."""
        frame = np.zeros((height, width), np.uint32)
        rgb = np.zeros((height, width, 3), np.float32)
        length = np.zeros((height, width), np.float32)
        p = denoise_temporal_params(width, height, reset, alpha_color, alpha_moments, depth_tolerance, normal_cos, **filter)
        self._check(self.lib.rt3_denoise_temporal(self.handle, C.byref(p), _ptr(frame), _ptr(rgb), _ptr(length)))
        return frame, rgb, length

    def denoise_stage(self, width, height, stage_ptr, tag, stream_ptr=None, **filter):
        """rt3_denoise_stage: this context's rows of a frame rendered in parts, prepared into the stage at ``stage_ptr`` (a device
        pointer of denoise_stage_words(width, height) words, possibly mapped from another process) for frame ``tag``;
        ``filter`` takes denoise_params' keywords. Asynchronous: ``stats()`` waits for it."""
        p = denoise_params(width, height, **filter)
        self._check(self.lib.rt3_denoise_stage(self.handle, C.byref(p), int(tag), C.c_void_p(stage_ptr), C.c_void_p(stream_ptr or 0)))

    def denoise_staged(self, width, height, stage_ptr, tag, **filter):
        """rt3_denoise_staged: on the stage's owner, after every part staged frame ``tag``: the whole frame filtered from the stage
        (``filter``: denoise_params' keywords). Returns (frame [H, W] uint32, rgb [H, W, 3] float32) like ``denoise``."""
        frame = np.zeros((height, width), np.uint32)
        rgb = np.zeros((height, width, 3), np.float32)
        p = denoise_params(width, height, **filter)
        self._check(self.lib.rt3_denoise_staged(self.handle, C.byref(p), int(tag), C.c_void_p(stage_ptr), _ptr(frame), _ptr(rgb)))
        return frame, rgb

    def stats(self):
        st = Stats()
        self._check(self.lib.rt3_get_stats(self.handle, C.byref(st)))
        return st

    def measure_fma_peak(self):
        v = C.c_double()
        self._check(self.lib.rt3_measure_fma_peak(self.handle, C.byref(v)))
        return v.value
