"""ORACLE (test infrastructure): ctypes front-end of oracle/b2d_oracle.c."""
from __future__ import annotations

import ctypes
import math
from typing import Tuple

import numpy as np

from . import build as _build

POSE = np.dtype([("x", "<i4"), ("y", "<i4"), ("z", "<i4"), ("angle", "<u4")])
DEFAULT_FOV_DEG = 65.0           # game/src/player.rs:84


class View(ctypes.Structure):
    _fields_ = [("W", ctypes.c_int32), ("H", ctypes.c_int32), ("F", ctypes.c_int32), ("FY2", ctypes.c_int32)]


_lib = None


def lib():
    global _lib
    if _lib is None:
        path = _build.build()
        L = ctypes.CDLL(path)
        L.b2o_view_init.argtypes = [ctypes.POINTER(View), ctypes.c_int, ctypes.c_int, ctypes.c_double]
        L.b2o_render_t.argtypes = [ctypes.c_void_p, ctypes.POINTER(View), ctypes.c_void_p, ctypes.c_int,
                                   ctypes.c_uint32, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                   ctypes.c_int]
        L.b2o_render_t.restype = ctypes.c_int
        L.b2o_crc32.argtypes = [ctypes.c_void_p, ctypes.c_size_t]
        L.b2o_crc32.restype = ctypes.c_uint32
        L.b2o_sincos_q30.argtypes = [ctypes.c_uint32, ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_int32)]
        L.b2o_plane_dirs.argtypes = [ctypes.POINTER(View), ctypes.c_uint32, ctypes.c_void_p]
        _lib = L
    return _lib


def make_view(width: int, height: int, fov_deg: float = DEFAULT_FOV_DEG) -> View:
    v = View()
    lib().b2o_view_init(ctypes.byref(v), width, height, math.tan(math.radians(fov_deg) / 2.0))
    return v


def make_pose(x: float, y: float, z: float, angle_deg: float) -> np.ndarray:
    p = np.zeros(1, dtype=POSE)
    p["x"] = int(round(x * 65536.0))
    p["y"] = int(round(y * 65536.0))
    p["z"] = int(round(z * 65536.0))
    p["angle"] = int(round(angle_deg / 360.0 * 4294967296.0)) & 0xFFFFFFFF
    return p


def render(blob: bytes, view: View, poses: np.ndarray, rgba: bool = False, threads: int = 1,
           seg_hits: bool = False, tics: int = 0, out: np.ndarray = None):
    """`out`: optional (n, H, W) uint8 array to render into (timing loops reuse it, so that a step does not pay for
    first-touch page faults of a fresh allocation)."""
    poses = np.ascontiguousarray(poses, dtype=POSE)
    n = len(poses)
    W, H = view.W, view.H
    if out is not None:
        assert out.dtype == np.uint8 and out.shape == (n, H, W) and out.flags.c_contiguous
    fb = out if out is not None else np.empty((n, H, W), dtype=np.uint8)
    out_rgba = np.empty((n, H, W), dtype=np.uint32) if rgba else None
    nsegs = int(np.frombuffer(blob, dtype="<u4", count=32)[6])
    hits = np.zeros((n, nsegs), dtype=np.int32) if seg_hits else None
    buf = (ctypes.c_char * len(blob)).from_buffer_copy(blob)
    from . import scene as _scene
    lights = np.ascontiguousarray(_scene.sector_lights_at(blob, tics), dtype=np.int16)   # light effects at `tics`
    rc = lib().b2o_render_t(ctypes.addressof(buf), ctypes.byref(view), poses.ctypes.data, n,
                            int(tics) & 0xFFFFFFFF, lights.ctypes.data if len(lights) else None, fb.ctypes.data,
                          out_rgba.ctypes.data if rgba else None,
                          hits.ctypes.data if seg_hits else None, int(threads))
    if rc != 0:
        raise RuntimeError("b2o_render failed: %d" % rc)
    res = [fb]
    if rgba:
        res.append(out_rgba)
    if seg_hits:
        res.append(hits)
    return res[0] if len(res) == 1 else tuple(res)


def crc32(arr: np.ndarray) -> int:
    a = np.ascontiguousarray(arr)
    return int(lib().b2o_crc32(a.ctypes.data, a.nbytes))


def sincos_q30(angle: int) -> Tuple[int, int]:
    c, s = ctypes.c_int32(), ctypes.c_int32()
    lib().b2o_sincos_q30(angle & 0xFFFFFFFF, ctypes.byref(c), ctypes.byref(s))
    return c.value, s.value


def plane_dirs(view: View, angle: int) -> np.ndarray:
    """(W, 2) int32: direction (ax, ay) of every screen column's ray at yaw `angle` (BAM), Q18, as the flat texel rule
    uses it (DESIGN.md C8)."""
    out = np.zeros((view.W, 2), dtype=np.int32)
    lib().b2o_plane_dirs(ctypes.byref(view), angle & 0xFFFFFFFF, out.ctypes.data)
    return out
