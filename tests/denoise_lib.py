"""Loader of the denoiser's CPU restatement (TEST INFRASTRUCTURE): ``tests/denoise_oracle.c``, which calls the filter arithmetic of
``include/rt3_denoise.h`` exactly as the kernels do, and the host backend's ``CudaRenderer::denoise``.

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
SOURCES = [os.path.join(ROOT, "tests", "denoise_oracle.c"), os.path.join(ROOT, "include", "rt3_denoise.h"), os.path.join(ROOT, "oracle", "rt3_oracle.c"),
           os.path.join(ROOT, "oracle", "rt3_oracle.h"), os.path.join(ROOT, "include", "rt3cuda.h"), os.path.join(ROOT, "include", "rt3_rng.h")]

_oracle = None


def oracle_lib():
    global _oracle
    if _oracle is None:
        digest = hashlib.sha256(b"".join(open(p, "rb").read() for p in SOURCES)).hexdigest()[:16]
        path = os.path.join(tempfile.gettempdir(), f"rt3_denoise_oracle_{os.getuid()}_{digest}.so")
        if not os.path.exists(path):
            tmp = f"{path}.{os.getpid()}"
            subprocess.run([os.environ.get("CC", "gcc"), "-std=c11", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared", "-pthread",
                            "-Wall", "-Wextra", "-I", os.path.join(ROOT, "include"), "-o", tmp, SOURCES[0], "-lm"], check=True)
            os.replace(tmp, path)
        lib = C.CDLL(path)
        vp = C.c_void_p
        lib.orc_denoise.argtypes = [C.c_uint32, C.c_uint32, vp, vp, vp, vp, C.POINTER(abi.DenoiseParams), C.c_uint32, vp, vp, C.c_int]
        lib.orc_denoise_check.argtypes = [C.POINTER(abi.DenoiseParams)]
        lib.orc_denoise_check.restype = C.c_char_p
        _oracle = lib
    return _oracle


def _f32(a, shape):
    a = np.ascontiguousarray(a, dtype=np.float32)
    assert a.shape == shape, (a.shape, shape)
    return a


def oracle_denoise(rgb, albedo, normal, depth, flags=0, n_threads=0, **params):
    """orc_denoise on [H, W, 3] radiance / albedo / normal and [H, W] depth -> (frame [H, W] uint32, rgb [H, W, 3] float32).
    Keyword arguments are Context.denoise's (iterations, sigma_luminance, sigma_normal, sigma_depth)."""
    h, w = depth.shape
    ins = [_f32(rgb, (h, w, 3)), _f32(albedo, (h, w, 3)), _f32(normal, (h, w, 3)), _f32(depth, (h, w))]
    frame = np.zeros((h, w), np.uint32)
    out = np.zeros((h, w, 3), np.float32)
    p = abi.denoise_params(w, h, **params)
    rc = oracle_lib().orc_denoise(w, h, *(a.ctypes.data for a in ins), C.byref(p), flags, frame.ctypes.data, out.ctypes.data, n_threads)
    assert rc == 0, "orc_denoise rejected its arguments"
    return frame, out


def check_params(**params):
    """rt3_dn_check_params through the restatement: None when valid, else the message."""
    msg = oracle_lib().orc_denoise_check(C.byref(abi.denoise_params(**params)))
    return None if msg is None else msg.decode()


def host_denoise(host_scene, width, height, focal=2.0, vh=2.0, **params):
    """CudaRenderer::denoise through the host backend's C shim (after render() and render_path_aovs() with the same camera):
    (frame [H, W] uint32, rgb [H, W, 3] float32)."""
    import hostlib
    L = hostlib.lib()
    L.rt3host_denoise.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_float, C.c_float, C.c_float, C.POINTER(abi.DenoiseParams), C.c_void_p, C.c_void_p]
    frame = np.zeros((height, width), np.uint32)
    rgb = np.zeros((height, width, 3), np.float32)
    vw = float(np.float32(np.float32(width) / np.float32(height)) * np.float32(2.0))
    p = abi.denoise_params(width, height, **params)
    rc = L.rt3host_denoise(host_scene.h, width, height, focal, vw, vh, C.byref(p), frame.ctypes.data, rgb.ctypes.data)
    if rc != 0:
        raise hostlib.HostError(L.rt3host_last_error().decode())
    return frame, rgb
