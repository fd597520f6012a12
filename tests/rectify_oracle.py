"""ctypes loader of the rotated remap oracle (tests/rectify_oracle.c), built like remap_oracle.py: the oracle's sources,
remap_oracle.c and rectify_oracle.c with the oracle's flags, into a per-user temporary directory.  Test infrastructure
only."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

import remap_oracle

_HERE = os.path.dirname(os.path.abspath(__file__))
_SOURCES = remap_oracle._SOURCES + [os.path.join(_HERE, "rectify_oracle.c")]
_CFLAGS = remap_oracle._CFLAGS

_lib = None


def lib():
    global _lib
    if _lib is None:
        h = hashlib.sha256(" ".join(_CFLAGS).encode())
        for f in _SOURCES + [os.path.join(remap_oracle._ORACLE, "acm_oracle.h")]:
            with open(f, "rb") as fh:
                h.update(fh.read())
        out_dir = os.path.join(tempfile.gettempdir(), f"acm_rectify_oracle_{os.getuid()}_{h.hexdigest()[:16]}")
        so = os.path.join(out_dir, "librectifyoracle.so")
        if not os.path.exists(so):
            os.makedirs(out_dir, exist_ok=True)
            tmp = so + f".{os.getpid()}"
            subprocess.run([remap_oracle._CC] + _CFLAGS + ["-I", remap_oracle._ORACLE, "-shared", "-o", tmp] + _SOURCES + ["-lm"], check=True)
            os.replace(tmp, so)
        L = C.CDLL(so)
        dp, u8p = C.POINTER(C.c_double), C.POINTER(C.c_uint8)
        from oracle.oracle import Model
        mp = C.POINTER(Model)
        L.orc_remap_map_rotated.argtypes = [mp, mp, dp, dp]; L.orc_remap_map_rotated.restype = None
        L.orc_remap_rgb8_rotated.argtypes = [mp, mp, dp, u8p, u8p, C.c_int]; L.orc_remap_rgb8_rotated.restype = None
        _lib = L
    return _lib


def _rot(R) -> np.ndarray:
    R = np.ascontiguousarray(R, dtype=np.float64)
    assert R.shape == (3, 3)
    return R


def remap_map_rotated(mi, mo, R) -> np.ndarray:
    """(Ho, Wo, 2) source coordinates on the input camera's frame through ray_in = R^T ray_out, NaN where a step fails."""
    R = _rot(R)
    out = np.empty((mo.height, mo.width, 2))
    lib().orc_remap_map_rotated(C.byref(mi), C.byref(mo), R.ctypes.data_as(C.POINTER(C.c_double)), out.ctypes.data_as(C.POINTER(C.c_double)))
    return out


def remap_rgb8_rotated(mi, mo, R, img: np.ndarray, interp: int = 1) -> np.ndarray:
    R = _rot(R)
    img = np.ascontiguousarray(img, dtype=np.uint8); assert img.shape == (mi.height, mi.width, 3)
    out = np.empty((mo.height, mo.width, 3), np.uint8)
    u8p = C.POINTER(C.c_uint8)
    lib().orc_remap_rgb8_rotated(C.byref(mi), C.byref(mo), R.ctypes.data_as(C.POINTER(C.c_double)), img.ctypes.data_as(u8p),
                                 out.ctypes.data_as(u8p), interp)
    return out
