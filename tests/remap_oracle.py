"""ctypes loader of the remap oracle (tests/remap_oracle.c), built with the oracle's flags together with the oracle's
sources into a per-user temporary directory, so that the tree may stay read-only.  Test infrastructure only."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_ORACLE = os.path.join(os.path.dirname(_HERE), "oracle")
_SOURCES = [os.path.join(_ORACLE, f) for f in ("acm_oracle_models.c", "acm_oracle_solver.c", "acm_oracle_util.c", "acm_oracle_image.c")]
_SOURCES.append(os.path.join(_HERE, "remap_oracle.c"))
_CC = "/usr/bin/gcc" if os.access("/usr/bin/gcc", os.X_OK) else "gcc"
_CFLAGS = ["-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-fopenmp", "-Wall", "-Wextra", "-std=c11"]  # oracle/Makefile

_lib = None


def lib():
    global _lib
    if _lib is None:
        h = hashlib.sha256(" ".join(_CFLAGS).encode())
        for f in _SOURCES + [os.path.join(_ORACLE, "acm_oracle.h")]:
            with open(f, "rb") as fh:
                h.update(fh.read())
        out_dir = os.path.join(tempfile.gettempdir(), f"acm_remap_oracle_{os.getuid()}_{h.hexdigest()[:16]}")
        so = os.path.join(out_dir, "libremaporacle.so")
        if not os.path.exists(so):
            os.makedirs(out_dir, exist_ok=True)
            tmp = so + f".{os.getpid()}"
            subprocess.run([_CC] + _CFLAGS + ["-I", _ORACLE, "-shared", "-o", tmp] + _SOURCES + ["-lm"], check=True)
            os.replace(tmp, so)
        L = C.CDLL(so)
        dp, u8p = C.POINTER(C.c_double), C.POINTER(C.c_uint8)
        from oracle.oracle import Model
        mp = C.POINTER(Model)
        L.orc_remap_map.argtypes = [mp, mp, dp]; L.orc_remap_map.restype = None
        L.orc_remap_rgb8.argtypes = [mp, mp, u8p, u8p, C.c_int]; L.orc_remap_rgb8.restype = None
        L.orc_remap_apply_map.argtypes = [dp, C.c_uint32, C.c_uint32, u8p, C.c_uint32, C.c_uint32, C.c_int, u8p]
        L.orc_remap_apply_map.restype = None
        _lib = L
    return _lib


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def _u8p(a):
    return a.ctypes.data_as(C.POINTER(C.c_uint8))


def remap_map(mi, mo) -> np.ndarray:
    """(Ho, Wo, 2) source coordinates on the input camera's frame, NaN where a step fails."""
    out = np.empty((mo.height, mo.width, 2))
    lib().orc_remap_map(C.byref(mi), C.byref(mo), _dp(out))
    return out


def remap_rgb8(mi, mo, img: np.ndarray, interp: int = 1) -> np.ndarray:
    img = np.ascontiguousarray(img, dtype=np.uint8); assert img.shape == (mi.height, mi.width, 3)
    out = np.empty((mo.height, mo.width, 3), np.uint8)
    lib().orc_remap_rgb8(C.byref(mi), C.byref(mo), _u8p(img), _u8p(out), interp)
    return out


def remap_apply_map(src_xy: np.ndarray, img: np.ndarray, interp: int = 1) -> np.ndarray:
    src_xy = np.ascontiguousarray(src_xy, dtype=np.float64); img = np.ascontiguousarray(img, dtype=np.uint8)
    Ho, Wo, _ = src_xy.shape
    Hi, Wi, _ = img.shape
    out = np.empty((Ho, Wo, 3), np.uint8)
    lib().orc_remap_apply_map(_dp(src_xy), Wo, Ho, _u8p(img), Wi, Hi, interp, _u8p(out))
    return out
