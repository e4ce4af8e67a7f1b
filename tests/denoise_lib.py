"""Loader of the denoiser's CPU restatement (TEST INFRASTRUCTURE): ``tests/denoise_oracle.c``, which calls the filter and
temporal arithmetic of ``include/rt3_denoise.h`` exactly as the kernels do (rt3_denoise_temporal's history is carried between
calls as numpy arrays), and the host backend's ``CudaRenderer::denoise`` and ``CudaRenderer::denoise_temporal``.

The restatement is compiled on first use into a temporary directory, keyed by the hash of its sources, so that the
repository tree is never written to."""
import ctypes as C
import os

import numpy as np

import rt3_b200  # noqa: F401
from rt3_b200 import abi

import path_aov_lib as pal

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SOURCES = [os.path.join(ROOT, "tests", "denoise_oracle.c"), os.path.join(ROOT, "include", "rt3_denoise.h"), *pal.SOURCES]

_oracle = None


def oracle_lib():
    global _oracle
    if _oracle is None:
        lib = pal.load_restatement("denoise", SOURCES)
        vp = C.c_void_p
        lib.orc_denoise.argtypes = [C.c_uint32, C.c_uint32, vp, vp, vp, vp, C.POINTER(abi.DenoiseParams), C.c_uint32, vp, vp, C.c_int]
        lib.orc_denoise_check.argtypes = [C.POINTER(abi.DenoiseParams)]
        lib.orc_denoise_check.restype = C.c_char_p
        lib.orc_denoise_temporal.argtypes = [C.c_uint32, C.c_uint32, vp, vp, vp, vp, C.POINTER(abi.Camera), C.POINTER(abi.Params), C.POINTER(abi.Camera), C.c_int,
                                             vp, vp, vp, C.POINTER(abi.DenoiseTemporalParams), C.c_uint32, vp, vp, vp, vp, vp, vp, C.c_int]
        lib.orc_denoise_temporal_check.argtypes = [C.POINTER(abi.DenoiseTemporalParams)]
        lib.orc_denoise_temporal_check.restype = C.c_char_p
        lib.orc_dn_primary_rays.argtypes = [C.POINTER(abi.Camera), C.POINTER(abi.Params), vp]
        lib.orc_dn_reproject.argtypes = [C.POINTER(abi.Camera), C.POINTER(abi.Camera), C.c_uint32, C.c_uint32, vp, vp, vp, vp, C.c_size_t]
        _oracle = lib
    return _oracle


def _f32(a, shape):
    a = np.ascontiguousarray(a, dtype=np.float32)
    assert a.shape == shape, (a.shape, shape)
    return a


def _inputs(rgb, albedo, normal, depth):
    h, w = depth.shape
    return [_f32(rgb, (h, w, 3)), _f32(albedo, (h, w, 3)), _f32(normal, (h, w, 3)), _f32(depth, (h, w))]


def oracle_denoise(rgb, albedo, normal, depth, flags=0, n_threads=0, **params):
    """orc_denoise on [H, W, 3] radiance / albedo / normal and [H, W] depth -> (frame [H, W] uint32, rgb [H, W, 3] float32).
    Keyword arguments are Context.denoise's (iterations, sigma_luminance, sigma_normal, sigma_depth)."""
    h, w = depth.shape
    ins = _inputs(rgb, albedo, normal, depth)
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


class History:
    """rt3_denoise_temporal's history as numpy arrays: per pixel colour and length ``col`` [H, W, 4] (r, g, b, n), moments
    ``mom`` [H, W, 2] and guide ``guide`` [H, W, 4], and the camera and scene tag of the frame that produced it."""

    def __init__(self, col, mom, guide, camera, scene):
        self.col, self.mom, self.guide, self.camera, self.scene = col, mom, guide, camera, scene


def oracle_denoise_temporal(rgb, albedo, normal, depth, camera, aov_params, history=None, scene=0, flags=0, reset=False, n_threads=0, **params):
    """orc_denoise_temporal: rt3_denoise_temporal on the arrays ``oracle_denoise`` takes, the camera and the abi.Params of the
    AOV call, and the history of the previous call (None: none). The history is used as rt3_denoise_temporal uses the
    context's: not after ``reset``, nor when its size or ``scene`` (a tag of the scene upload) differ. Keyword arguments
    are Context.denoise_temporal's. Returns (frame, rgb, history_length, the new History)."""
    h, w = depth.shape
    ins = _inputs(rgb, albedo, normal, depth)
    have = history is not None and not reset and history.col.shape[:2] == (h, w) and history.scene == scene
    nxt = History(np.zeros((h, w, 4), np.float32), np.zeros((h, w, 2), np.float32), np.zeros((h, w, 4), np.float32), camera, scene)
    frame = np.zeros((h, w), np.uint32)
    out = np.zeros((h, w, 3), np.float32)
    length = np.zeros((h, w), np.float32)
    tp = abi.denoise_temporal_params(w, h, reset, **params)
    prev = [history.col, history.mom, history.guide] if have else [None, None, None]
    prev = [None if a is None else np.ascontiguousarray(a, np.float32).ctypes.data for a in prev]
    rc = oracle_lib().orc_denoise_temporal(w, h, *(a.ctypes.data for a in ins), C.byref(camera), C.byref(aov_params),
                                           C.byref(history.camera) if have else None, 1 if have else 0, *prev, C.byref(tp), flags,
                                           nxt.col.ctypes.data, nxt.mom.ctypes.data, nxt.guide.ctypes.data, frame.ctypes.data, out.ctypes.data,
                                           length.ctypes.data, n_threads)
    assert rc == 0, "orc_denoise_temporal rejected its arguments"
    return frame, out, length, nxt


def check_temporal_params(**params):
    """rt3_dn_check_temporal_params through the restatement: None when valid, else the message."""
    msg = oracle_lib().orc_denoise_temporal_check(C.byref(abi.denoise_temporal_params(**params)))
    return None if msg is None else msg.decode()


def reproject(cur, prev, w, h, xy, rays, depth):
    """rt3_dn_reproject per pixel: xy [N, 2] integer pixel coordinates, rays [N, 6] (origin, unit direction), depth [N] ->
    [N, 4] float32 (x', y', |X - O_prev|, 1 when a position exists)."""
    xy, rays, depth = (np.ascontiguousarray(a, np.float32) for a in (xy, rays, depth))
    out = np.zeros((len(depth), 4), np.float32)
    oracle_lib().orc_dn_reproject(C.byref(cur), C.byref(prev), w, h, xy.ctypes.data, rays.ctypes.data, depth.ctypes.data, out.ctypes.data, len(depth))
    return out


def primary_rays(camera, aov_params):
    """The primary rays rt3_denoise_temporal reprojects (sample first_sample of the AOV call): [H, W, 6] float32, origin and
    unit direction."""
    out = np.zeros((aov_params.height, aov_params.width, 6), np.float32)
    oracle_lib().orc_dn_primary_rays(C.byref(camera), C.byref(aov_params), out.ctypes.data)
    return out


def _host_call(name, host_scene, width, height, focal, vh, p):
    """rt3host_<name> with the reference camera and parameters `p` -> (frame [H, W] uint32, rgb [H, W, 3] float32)."""
    import hostlib
    L = hostlib.lib()
    fn = getattr(L, f"rt3host_{name}")
    fn.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_float, C.c_float, C.c_float, C.POINTER(type(p)), C.c_void_p, C.c_void_p]
    frame = np.zeros((height, width), np.uint32)
    rgb = np.zeros((height, width, 3), np.float32)
    vw = float(np.float32(np.float32(width) / np.float32(height)) * np.float32(2.0))
    rc = fn(host_scene.h, width, height, focal, vw, vh, C.byref(p), frame.ctypes.data, rgb.ctypes.data)
    if rc != 0:
        raise hostlib.HostError(L.rt3host_last_error().decode())
    return frame, rgb


def host_denoise(host_scene, width, height, focal=2.0, vh=2.0, **params):
    """CudaRenderer::denoise through the host backend's C shim (after render() and render_path_aovs() with the same camera):
    (frame [H, W] uint32, rgb [H, W, 3] float32)."""
    return _host_call("denoise", host_scene, width, height, focal, vh, abi.denoise_params(width, height, **params))


def host_denoise_temporal(host_scene, width, height, focal=2.0, vh=2.0, reset=False, **params):
    """CudaRenderer::denoise_temporal through the host backend's C shim: (frame [H, W] uint32, rgb [H, W, 3] float32)."""
    return _host_call("denoise_temporal", host_scene, width, height, focal, vh, abi.denoise_temporal_params(width, height, reset, **params))
