"""Loaders for the path-traced AOVs (TEST INFRASTRUCTURE): the CPU restatement ``tests/path_aov_oracle.c`` (the oracle's
closest-hit code compiled together with the AOV pass) and the host backend's ``render_path_aovs`` / ``write_path_aovs_pfm``.

The restatement is compiled on first use into a temporary directory, keyed by the hash of its sources, so that the
repository tree is never written to."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

import rt3_b200  # noqa: F401
from rt3_b200 import abi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SOURCES = [os.path.join(ROOT, "tests", "path_aov_oracle.c"), os.path.join(ROOT, "oracle", "rt3_oracle.c"), os.path.join(ROOT, "oracle", "rt3_oracle.h"),
           os.path.join(ROOT, "include", "rt3cuda.h"), os.path.join(ROOT, "include", "rt3_rng.h")]
AOV_KEYS = ("hit_prim", "hit_entity", "hit_t", "albedo", "normal")

_oracle = None


def oracle_lib():
    global _oracle
    if _oracle is None:
        digest = hashlib.sha256(b"".join(open(p, "rb").read() for p in SOURCES)).hexdigest()[:16]
        path = os.path.join(tempfile.gettempdir(), f"rt3_path_aov_oracle_{os.getuid()}_{digest}.so")
        if not os.path.exists(path):
            tmp = f"{path}.{os.getpid()}"
            subprocess.run([os.environ.get("CC", "gcc"), "-std=c11", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared", "-pthread",
                            "-Wall", "-Wextra", "-I", os.path.join(ROOT, "include"), "-o", tmp, SOURCES[0], "-lm"], check=True)
            os.replace(tmp, path)
        lib = C.CDLL(path)
        lib.orc_render_path_aovs.argtypes = [C.POINTER(abi.Scene), C.POINTER(abi.Camera), C.POINTER(abi.Params), C.POINTER(abi.PathAovs), C.c_int]
        _oracle = lib
    return _oracle


def empty_aovs(height, width):
    return {"hit_prim": np.zeros((height, width), np.uint32), "hit_entity": np.zeros((height, width), np.uint32),
            "hit_t": np.zeros((height, width), np.float32), "albedo": np.zeros((height, width, 3), np.float32),
            "normal": np.zeros((height, width, 3), np.float32)}


def as_struct(aovs):
    return abi.PathAovs(*(aovs[k].ctypes.data_as(C.c_void_p) for k in AOV_KEYS))


def oracle_path_aovs(scene: abi.SceneArrays, camera, params, n_threads=0):
    """orc_render_path_aovs -> the dict Context.render_path_aovs returns (rows of other partitions 0)."""
    out = empty_aovs(params.height, params.width)
    st = scene.as_struct()
    rc = oracle_lib().orc_render_path_aovs(C.byref(st), C.byref(camera), C.byref(params), C.byref(as_struct(out)), n_threads)
    assert rc == 0
    return out


def host_path_aovs(host_scene, width, height, aov_spp, focal=2.0, vh=2.0, pfm_dir=None):
    """CudaRenderer::render_path_aovs through the host backend's C shim (and write_path_aovs_pfm into `pfm_dir` when given)."""
    import hostlib
    L = hostlib.lib()
    L.rt3host_path_aovs.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_float, C.c_float, C.c_float, C.c_uint32, C.POINTER(abi.PathAovs), C.c_char_p]
    out = empty_aovs(height, width)
    vw = float(np.float32(np.float32(width) / np.float32(height)) * np.float32(2.0))
    rc = L.rt3host_path_aovs(host_scene.h, width, height, focal, vw, vh, aov_spp, C.byref(as_struct(out)), str(pfm_dir).encode() if pfm_dir else None)
    if rc != 0:
        raise hostlib.HostError(L.rt3host_last_error().decode())
    return out


def read_pfm(path):
    """A Portable Float Map -> [H, W, 3] (PF) or [H, W] (Pf) float32, rows top to bottom."""
    with open(path, "rb") as f:
        kind = f.readline().strip()
        w, h = (int(v) for v in f.readline().split())
        scale = float(f.readline())
        data = np.frombuffer(f.read(), "<f4" if scale < 0 else ">f4")
    ch = 3 if kind == b"PF" else 1
    img = data.reshape(h, w, ch)[::-1]
    return img if ch == 3 else img[..., 0]
