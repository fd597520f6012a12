"""ctypes loader of the depth-image oracle (tests/depth_oracle.c), built like triangulate_oracle.py: the oracle's sources
and depth_oracle.c with the oracle's flags, into a per-user temporary directory.  Test infrastructure only."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

import remap_oracle

_HERE = os.path.dirname(os.path.abspath(__file__))
_SOURCES = remap_oracle._SOURCES[:-1] + [os.path.join(_HERE, "depth_oracle.c")]
_CFLAGS = remap_oracle._CFLAGS

OK, EMPTY, UNPROJECT = 0, 1, 2

_lib = None


def lib():
    global _lib
    if _lib is None:
        h = hashlib.sha256(" ".join(_CFLAGS).encode())
        for f in _SOURCES + [os.path.join(remap_oracle._ORACLE, "acm_oracle.h")]:
            with open(f, "rb") as fh:
                h.update(fh.read())
        out_dir = os.path.join(tempfile.gettempdir(), f"acm_depth_oracle_{os.getuid()}_{h.hexdigest()[:16]}")
        so = os.path.join(out_dir, "libdepthoracle.so")
        if not os.path.exists(so):
            os.makedirs(out_dir, exist_ok=True)
            tmp = so + f".{os.getpid()}"
            subprocess.run([remap_oracle._CC] + _CFLAGS + ["-I", remap_oracle._ORACLE, "-shared", "-o", tmp] + _SOURCES + ["-lm"], check=True)
            os.replace(tmp, so)
        L = C.CDLL(so)
        dp, fp, u8p, u32p = C.POINTER(C.c_double), C.POINTER(C.c_float), C.POINTER(C.c_uint8), C.POINTER(C.c_uint32)
        from oracle.oracle import Model
        mp = C.POINTER(Model)
        L.orc_render_depth.argtypes = [mp, dp, dp, dp, C.c_size_t, fp, u32p, dp]
        L.orc_render_depth.restype = None
        L.orc_depth_to_points.argtypes = [mp, dp, dp, fp, dp, u8p]
        L.orc_depth_to_points.restype = None
        _lib = L
    return _lib


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def _pose(R, t):
    R = np.eye(3) if R is None else R
    t = np.zeros(3) if t is None else t
    return np.ascontiguousarray(R, dtype=np.float64).reshape(9), np.ascontiguousarray(t, dtype=np.float64).reshape(3)


def render_depth(m, xyz, R=None, t=None, want_uv=False):
    """(range (H, W) float32, index (H, W) uint32[, uv (N, 2) of every point, NaN where project fails]) of the world points
    xyz (N, 3) seen through x_cam = R x + t."""
    R, t = _pose(R, t)
    xyz = np.ascontiguousarray(xyz, dtype=np.float64).reshape(-1, 3)
    rng, idx = np.empty((m.height, m.width), np.float32), np.empty((m.height, m.width), np.uint32)
    uv = np.empty((len(xyz), 2)) if want_uv else None
    lib().orc_render_depth(C.byref(m), _dp(R), _dp(t), _dp(xyz), len(xyz), rng.ctypes.data_as(C.POINTER(C.c_float)),
                           idx.ctypes.data_as(C.POINTER(C.c_uint32)), _dp(uv) if want_uv else None)
    return (rng, idx, uv) if want_uv else (rng, idx)


def depth_to_points(m, range_image, R=None, t=None):
    """(points (H, W, 3), status (H, W) uint8) of a (H, W) float32 range image."""
    R, t = _pose(R, t)
    r = np.ascontiguousarray(range_image, dtype=np.float32)
    assert r.shape == (m.height, m.width), r.shape
    xyz, st = np.empty((m.height, m.width, 3)), np.empty((m.height, m.width), np.uint8)
    lib().orc_depth_to_points(C.byref(m), _dp(R), _dp(t), r.ctypes.data_as(C.POINTER(C.c_float)), _dp(xyz),
                              st.ctypes.data_as(C.POINTER(C.c_uint8)))
    return xyz, st
