"""ctypes loader of the triangulation oracle (tests/triangulate_oracle.c), built like remap_oracle.py: the oracle's sources
and triangulate_oracle.c with the oracle's flags, into a per-user temporary directory.  Test infrastructure only."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

import remap_oracle

_HERE = os.path.dirname(os.path.abspath(__file__))
_SOURCES = remap_oracle._SOURCES[:-1] + [os.path.join(_HERE, "triangulate_oracle.c")]
_CFLAGS = remap_oracle._CFLAGS

OK, UNPROJECT_FIRST, UNPROJECT_SECOND, PARALLEL, BEHIND, PROJECT = range(6)

_lib = None


def lib():
    global _lib
    if _lib is None:
        h = hashlib.sha256(" ".join(_CFLAGS).encode())
        for f in _SOURCES + [os.path.join(remap_oracle._ORACLE, "acm_oracle.h")]:
            with open(f, "rb") as fh:
                h.update(fh.read())
        out_dir = os.path.join(tempfile.gettempdir(), f"acm_triangulate_oracle_{os.getuid()}_{h.hexdigest()[:16]}")
        so = os.path.join(out_dir, "libtriangulateoracle.so")
        if not os.path.exists(so):
            os.makedirs(out_dir, exist_ok=True)
            tmp = so + f".{os.getpid()}"
            subprocess.run([remap_oracle._CC] + _CFLAGS + ["-I", remap_oracle._ORACLE, "-shared", "-o", tmp] + _SOURCES + ["-lm"], check=True)
            os.replace(tmp, so)
        L = C.CDLL(so)
        dp, u8p = C.POINTER(C.c_double), C.POINTER(C.c_uint8)
        from oracle.oracle import Model
        mp = C.POINTER(Model)
        L.orc_triangulate.argtypes = [mp, mp, dp, dp, dp, dp, C.c_size_t, C.c_int, dp, dp, u8p, C.c_int]
        L.orc_triangulate.restype = None
        L.orc_triangulate_residuals.argtypes = [mp, mp, dp, dp, dp, dp, dp, dp]
        L.orc_triangulate_residuals.restype = C.c_int
        _lib = L
    return _lib


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def _arr(a, shape):
    a = np.ascontiguousarray(a, dtype=np.float64)
    assert a.shape[1:] == shape[1:] or a.shape == shape, a.shape
    return a


def triangulate(ma, mb, R, t, uv1, uv2, max_iterations=10, nthreads=1):
    """(points (N,3), errors (N,2), status (N,) uint8) of the pairs uv1[i] <-> uv2[i]; x_cam2 = R x_cam1 + t."""
    R = _arr(R, (3, 3)).reshape(9)
    t = np.ascontiguousarray(t, dtype=np.float64).reshape(3)
    uv1 = np.ascontiguousarray(uv1, dtype=np.float64).reshape(-1, 2)
    uv2 = np.ascontiguousarray(uv2, dtype=np.float64).reshape(-1, 2)
    n = len(uv1)
    assert len(uv2) == n
    xyz, err, st = np.empty((n, 3)), np.empty((n, 2)), np.empty(n, np.uint8)
    lib().orc_triangulate(C.byref(ma), C.byref(mb), _dp(R), _dp(t), _dp(uv1), _dp(uv2), n, max_iterations, _dp(xyz), _dp(err),
                          st.ctypes.data_as(C.POINTER(C.c_uint8)), nthreads)
    return xyz, err, st


def residuals(ma, mb, R, t, uv1, uv2, X):
    """The four pixel residuals at X, or None where X does not project into both cameras."""
    R = np.ascontiguousarray(R, dtype=np.float64).reshape(9)
    t = np.ascontiguousarray(t, dtype=np.float64).reshape(3)
    a, b = np.ascontiguousarray(uv1, dtype=np.float64), np.ascontiguousarray(uv2, dtype=np.float64)
    X = np.ascontiguousarray(X, dtype=np.float64)
    r = np.empty(4)
    ok = lib().orc_triangulate_residuals(C.byref(ma), C.byref(mb), _dp(R), _dp(t), _dp(a), _dp(b), _dp(X), _dp(r))
    return r if ok else None
