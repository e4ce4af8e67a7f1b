"""Loaders for the parity checkers (TEST INFRASTRUCTURE): the CPU restatement
``oracle/liboracle.so`` and the compiled reference ``oracle/_ref/libref_seq.so``.
Only tests/, __graft_entry__.smoke() and bench.py's CPU-baseline legs import this.
"""
import ctypes as C
import os
import subprocess

import numpy as np

import rt3_b200  # noqa: F401
from rt3_b200 import abi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
PORT_LIB = os.path.join(ORACLE_DIR, "liboracle.so")
BOOK_LIB = os.path.join(ORACLE_DIR, "liboracle_book.so")
REF_LIB = os.path.join(ORACLE_DIR, "_ref", "libref_seq.so")
REF_TEDDY = os.path.join(ORACLE_DIR, "_ref", "teddy.obj")

_port = None
_book = None
_ref = None


def build(which="all"):
    subprocess.run(["make", "-C", ORACLE_DIR, which], check=True, stdout=subprocess.DEVNULL)


def port():
    """The CPU restatement (oracle/rt3_oracle.c)."""
    global _port
    if _port is None:
        if not os.path.exists(PORT_LIB):
            build("port")
        lib = C.CDLL(PORT_LIB)
        vp = C.c_void_p
        lib.orc_render_reference.argtypes = [C.POINTER(abi.Scene), C.POINTER(abi.Camera), C.c_uint32, C.c_uint32, vp, vp, vp, vp]
        lib.orc_render_pathtrace.argtypes = [C.POINTER(abi.Scene), C.POINTER(abi.Camera), C.POINTER(abi.Params), vp, vp,
                                             C.POINTER(C.c_uint64), C.c_int]
        lib.orc_hash1.argtypes = [C.c_uint32]
        lib.orc_hash1.restype = C.c_uint32
        lib.orc_hash4.argtypes = [C.c_uint32] * 4
        lib.orc_hash4.restype = C.c_uint32
        lib.orc_float_construct.argtypes = [C.c_uint32]
        lib.orc_float_construct.restype = C.c_float
        lib.orc_draw.argtypes = [C.c_uint32] * 4
        lib.orc_draw.restype = C.c_float
        lib.orc_sincos_2pi.argtypes = [C.c_float, C.POINTER(C.c_float), C.POINTER(C.c_float)]
        _port = lib
    return _port


def oracle_reference(scene: abi.SceneArrays, camera, width, height):
    """orc_render_reference -> (frame, prim, entity, t), each [H, W]."""
    frame = np.zeros((height, width), np.uint32)
    prim = np.zeros((height, width), np.uint32)
    ent = np.zeros((height, width), np.uint32)
    t = np.zeros((height, width), np.float32)
    st = scene.as_struct()
    rc = port().orc_render_reference(C.byref(st), C.byref(camera), width, height, frame.ctypes.data, prim.ctypes.data,
                                     ent.ctypes.data, t.ctypes.data)
    assert rc == 0
    return frame, prim, ent, t


def oracle_pathtrace(scene: abi.SceneArrays, camera, params, n_threads=0, want_accum=False):
    """orc_render_pathtrace -> (frame [H, W], accum [H, W, 3] or None, rays)."""
    frame = np.zeros((params.height, params.width), np.uint32)
    accum = np.zeros((params.height, params.width, 3), np.uint64) if want_accum else None
    rays = C.c_uint64()
    st = scene.as_struct()
    rc = port().orc_render_pathtrace(C.byref(st), C.byref(camera), C.byref(params), frame.ctypes.data,
                                     accum.ctypes.data if want_accum else None, C.byref(rays), n_threads)
    assert rc == 0
    return frame, accum, rays.value


def book_render(scene: abi.SceneArrays, camera, width, height, spp, max_depth=50, seed=1, flags=0, rows=None, n_threads=0):
    """The independent checker (oracle/rtiow_book.cpp): mean linear radiance [H, W, 3] float32 of rows `rows` = (first, count)."""
    global _book
    if _book is None:
        if not os.path.exists(BOOK_LIB):
            build("book")
        _book = C.CDLL(BOOK_LIB)
        _book.book_render.argtypes = [C.POINTER(abi.Scene), C.POINTER(abi.Camera)] + [C.c_uint32] * 8 + [C.c_void_p, C.c_int]
    first, count = rows if rows is not None else (0, height)
    rgb = np.zeros((height, width, 3), np.float32)
    st = scene.as_struct()
    rc = _book.book_render(C.byref(st), C.byref(camera), width, height, spp, max_depth, seed, flags, first, count, rgb.ctypes.data, n_threads)
    assert rc == 0
    return rgb


def resolve_8bit(rgb, gamma=True):
    """The product's resolve on a float image: gamma 2, then glm::packUnorm4x8 rounding; returns [H, W, 3] uint8 levels as float64."""
    v = np.sqrt(np.maximum(rgb.astype(np.float64), 0)) if gamma else rgb.astype(np.float64)
    return np.floor(np.clip(v, 0, 1) * 255 + 0.5)


def unpack_rgb(frame):
    """Packed frame (r<<24 | g<<16 | b<<8 | a) -> [H, W, 3] float64 levels."""
    return np.stack([(frame >> s) & 0xFF for s in (24, 16, 8)], -1).astype(np.float64)


def psnr_levels(a, b):
    mse = ((a - b) ** 2).mean()
    return 99.0 if mse == 0 else 10 * np.log10(255.0 ** 2 / mse)


def block_mean(img, k):
    h, w = img.shape[0] // k * k, img.shape[1] // k * k
    return img[:h, :w].reshape(h // k, k, w // k, k, -1).mean(axis=(1, 3))


def have_ref():
    return os.path.exists(REF_LIB)


def ref():
    """The compiled reference CPU backend (oracle/ref_driver.cpp + /root/reference sources)."""
    global _ref
    if _ref is None:
        lib = C.CDLL(REF_LIB)
        lib.ref_scene_create.restype = C.c_void_p
        lib.ref_last_error.restype = C.c_char_p
        vp, fp, u32 = C.c_void_p, C.POINTER(C.c_float), C.c_uint32
        lib.ref_scene_destroy.argtypes = [vp]
        lib.ref_scene_add_triangle.argtypes = [vp, fp, fp, fp, fp]
        lib.ref_scene_add_sphere.argtypes = [vp, fp, C.c_float, u32, u32, fp]
        lib.ref_scene_add_object.argtypes = [vp, C.c_char_p, fp, C.c_float, fp]
        lib.ref_scene_prerender.argtypes = [vp]
        for name in ("ref_scene_n_entities", "ref_scene_n_faces", "ref_scene_n_vertices"):
            getattr(lib, name).argtypes = [vp]
            getattr(lib, name).restype = u32
        lib.ref_scene_export.argtypes = [vp, vp, vp]
        lib.ref_scene_entity_counts.argtypes = [vp, vp, vp]
        lib.ref_scene_render.argtypes = [vp, u32, u32, C.c_float, C.c_float, C.c_float, fp, vp, C.POINTER(C.c_double)]
        lib.ref_camera_vectors.argtypes = [u32, u32, C.c_float, C.c_float, C.c_float, fp]
        _ref = lib
    return _ref


def _f3(v):
    return (C.c_float * 3)(*[float(x) for x in v])


class RefScene:
    """A scene built through the reference's own ECS API and Sequential renderer."""

    def __init__(self):
        self.lib = ref()
        self.h = C.c_void_p(self.lib.ref_scene_create())

    def _ok(self, rc):
        if rc != 0:
            raise RuntimeError(self.lib.ref_last_error().decode())

    def add_triangle(self, p1, p2, p3, color):
        self._ok(self.lib.ref_scene_add_triangle(self.h, _f3(p1), _f3(p2), _f3(p3), _f3(color)))

    def add_sphere(self, center, radius, n_meridians, n_parallels, color):
        self._ok(self.lib.ref_scene_add_sphere(self.h, _f3(center), radius, n_meridians, n_parallels, _f3(color)))

    def add_object(self, path, center, scale, color):
        self._ok(self.lib.ref_scene_add_object(self.h, path.encode(), _f3(center), scale, _f3(color)))

    def prerender(self):
        self._ok(self.lib.ref_scene_prerender(self.h))

    def export(self) -> abi.SceneArrays:
        """The flattened GFace / vec4 arrays the reference renders from, plus the face -> entity map."""
        nf, nv, ne = (self.lib.ref_scene_n_faces(self.h), self.lib.ref_scene_n_vertices(self.h),
                      self.lib.ref_scene_n_entities(self.h))
        faces = np.zeros(nf, abi.FACE_DTYPE)
        verts = np.zeros(nv, abi.VERTEX_DTYPE)
        self._ok(self.lib.ref_scene_export(self.h, faces.ctypes.data, verts.ctypes.data))
        fpe = np.zeros(ne, np.uint32)
        vpe = np.zeros(ne, np.uint32)
        self.lib.ref_scene_entity_counts(self.h, fpe.ctypes.data, vpe.ctypes.data)
        entity = np.repeat(np.arange(ne, dtype=np.uint32), fpe)
        return abi.SceneArrays(faces=faces, vertices=verts, face_entity=entity)

    def render(self, width, height, focal=2.0, vh=2.0):
        """Camera::update(W, H, focal, (W/H)*2, 2) + render, as Main.cpp:272,285. Returns (frame, seconds)."""
        frame = np.zeros((height, width), np.uint32)
        sec = C.c_double()
        vw = float(np.float32(np.float32(width) / np.float32(height)) * np.float32(2.0))
        self._ok(self.lib.ref_scene_render(self.h, width, height, focal, vw, vh, None, frame.ctypes.data, C.byref(sec)))
        return frame, sec.value

    def close(self):
        if self.h:
            self.lib.ref_scene_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def add_scene(s, kind):
    """The fixed scenes the pinning tests render, built through the ECS API of `s` (RefScene or hostlib.HostScene)."""
    if kind == "triangle":
        s.add_triangle((1, 0, -3), (-1, 0, -3), (0, 1, -3), (1, 0, 0))
    elif kind == "sphere8":
        s.add_sphere((0, 0, -3), 1.0, 8, 8, (1, 0, 0))
    elif kind == "mixed":
        s.add_sphere((0.6, 0.2, -4), 0.9, 12, 9, (0.2, 0.9, 0.3))
        s.add_triangle((2, -1, -5), (-2, -1, -5), (0, 2, -6), (0.1, 0.2, 1.0))
        s.add_sphere((-0.8, -0.3, -2.5), 0.5, 5, 4, (1, 1, 0))


def add_random_scene(s, seed):
    """Triangles and tessellated spheres at random places (in front of, around and behind the camera, overlapping, some
    degenerate) added to `s`; returns the random frame size (W, H) drawn after them."""
    rng = np.random.default_rng(1000 + seed)
    for _ in range(int(rng.integers(1, 7))):
        if rng.random() < 0.5:
            c = rng.uniform(-3, 3, 3) + np.array([0, 0, -4.0])
            pts = c + rng.uniform(-2, 2, (3, 3))
            if rng.random() < 0.15:
                pts[2] = pts[1]                                  # degenerate: NaN normal in the reference (Triangle.cpp:48)
            s.add_triangle(tuple(pts[0]), tuple(pts[1]), tuple(pts[2]), tuple(rng.uniform(0, 1, 3)))
        else:
            c = rng.uniform(-2.5, 2.5, 3) + np.array([0, 0, -3.0 if rng.random() < 0.8 else 3.0])
            s.add_sphere(tuple(c), float(rng.uniform(0.2, 1.5)), int(rng.integers(3, 14)), int(rng.integers(3, 12)), tuple(rng.uniform(0, 1, 3)))
    return int(rng.integers(2, 140)), int(rng.integers(2, 90))


def fnv64(words):
    """64-bit FNV-1a variant over uint32 words (xor the whole word, then multiply)."""
    h = 0xcbf29ce484222325
    for w in np.ascontiguousarray(words).ravel().astype(np.uint32).tolist():
        h = ((h ^ w) * 0x100000001b3) & 0xFFFFFFFFFFFFFFFF
    return h
