"""Context and device point buffers (thin wrappers over the acm_ctx / acm_points handles)."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _native as N
from .errors import AcmError, raise_call_status

_lib = N.lib


class Context:
    """One CUDA device + one stream.  `stream` may be a raw cudaStream_t (e.g.
    torch.cuda.current_stream().cuda_stream) so that torch events see the work."""

    def __init__(self, device: int = 0, stream: int | None = None):
        self._h = C.c_void_p()
        rc = _lib.acm_ctx_create(device, C.c_void_p(stream) if stream else None, C.byref(self._h))
        if rc != N.OK:
            raise AcmError(f"acm_ctx_create({device}) failed ({rc}): {_lib.acm_last_error(None).decode()}")
        self.device = device
        self._pinned = []

    # -- plumbing ---------------------------------------------------------------------------
    @property
    def handle(self):
        return self._h

    def check(self, rc: int):
        if rc != N.OK:
            raise_call_status(rc, _lib.acm_last_error(self._h).decode())

    def sync(self):
        self.check(_lib.acm_ctx_sync(self._h))

    def close(self):
        if self._h:
            for ptr in getattr(self, "_pinned", []):
                _lib.acm_host_free_pinned(self._h, C.c_void_p(ptr))
            self._pinned = []
            _lib.acm_ctx_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def device_info(self) -> dict:
        info = (C.c_int64 * 4)()
        self.check(_lib.acm_ctx_device_info(self._h, info))
        return {"sm_count": info[0], "l2_bytes": info[1], "max_smem_per_block": info[2], "cc": info[3]}

    def kernel_launches(self) -> int:
        return int(_lib.acm_ctx_kernel_launches(self._h))

    def timer_start(self):
        self.check(_lib.acm_timer_start(self._h))

    def timer_stop(self) -> float:
        ms = C.c_float()
        self.check(_lib.acm_timer_stop(self._h, C.byref(ms)))
        return float(ms.value)

    # -- raw memory -------------------------------------------------------------------------
    def device_alloc(self, nbytes: int) -> int:
        p = C.c_void_p()
        self.check(_lib.acm_device_alloc(self._h, nbytes, C.byref(p)))
        return p.value

    def device_free(self, ptr: int):
        self.check(_lib.acm_device_free(self._h, C.c_void_p(ptr)))

    def staging(self) -> "Staging":
        """Owner of one call's device temporaries, freed when its `with` block ends."""
        return Staging(self)

    def pinned_empty(self, shape, dtype) -> np.ndarray:
        """numpy array backed by page-locked host memory owned by this context."""
        dtype = np.dtype(dtype)
        nbytes = int(np.prod(shape)) * dtype.itemsize
        p = C.c_void_p()
        self.check(_lib.acm_host_alloc_pinned(self._h, max(nbytes, 1), C.byref(p)))
        buf = (C.c_uint8 * max(nbytes, 1)).from_address(p.value)
        arr = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)
        self._pinned.append(p.value)  # released by close(); free earlier with pinned_free(arr)
        return arr

    def pinned_free(self, arr: np.ndarray):
        ptr = arr.ctypes.data
        if ptr in self._pinned:
            self._pinned.remove(ptr)
            _lib.acm_host_free_pinned(self._h, C.c_void_p(ptr))

    def h2d(self, dst_ptr: int, src: np.ndarray):
        self.check(_lib.acm_memcpy_h2d(self._h, C.c_void_p(dst_ptr), src.ctypes.data_as(C.c_void_p), src.nbytes))

    def d2h(self, dst: np.ndarray, src_ptr: int):
        self.check(_lib.acm_memcpy_d2h(self._h, dst.ctypes.data_as(C.c_void_p), C.c_void_p(src_ptr), dst.nbytes))

    def d2d(self, dst_ptr: int, src_ptr: int, nbytes: int):
        self.check(_lib.acm_memcpy_d2d(self._h, C.c_void_p(dst_ptr), C.c_void_p(src_ptr), nbytes))

    # -- multi-GPU ----------------------------------------------------------------------------
    @staticmethod
    def comm_unique_id() -> bytes:
        buf = (C.c_uint8 * 128)()
        rc = _lib.acm_comm_get_unique_id(buf)
        if rc != N.OK:
            raise AcmError(f"acm_comm_get_unique_id failed ({rc}): {_lib.acm_last_error(None).decode()}")
        return bytes(buf)

    def comm_init_rank(self, n_ranks: int, rank: int, unique_id: bytes):
        buf = (C.c_uint8 * 128).from_buffer_copy(unique_id)
        self.check(_lib.acm_comm_init_rank(self._h, n_ranks, rank, buf))

    def peer_export(self) -> bytes:
        buf = (C.c_uint8 * 64)()
        self.check(_lib.acm_peer_export(self._h, buf))
        return bytes(buf)

    def peer_attach(self, n_ranks: int, rank: int, handles: bytes):
        buf = (C.c_uint8 * (64 * n_ranks)).from_buffer_copy(handles)
        self.check(_lib.acm_peer_attach(self._h, n_ranks, rank, buf))

    def peer_detach(self):
        self.check(_lib.acm_peer_detach(self._h))

    def comm_size(self) -> int:
        return int(_lib.acm_comm_size(self._h))


_default_ctx = None


def default_context() -> Context:
    global _default_ctx
    if _default_ctx is None:
        _default_ctx = Context(0)
    return _default_ctx


class Points:
    """Device SoA point buffer (acm_points).  Host arrays are (N, dim) float64, C-contiguous: the
    memory order of nalgebra's Matrix3xX / Matrix2xX (reference src/util/point_sampling.rs:46-49)."""

    def __init__(self, ctx: Context, dim: int, n: int, dtype: int = N.F64, _handle=None):
        self.ctx = ctx
        if _handle is None:
            self._h = C.c_void_p()
            ctx.check(_lib.acm_points_create(ctx.handle, dim, n, dtype, C.byref(self._h)))
        else:
            self._h = _handle
        self.dim, self.dtype = dim, dtype

    @property
    def handle(self):
        return self._h

    def __len__(self):
        return int(_lib.acm_points_len(self._h))

    @classmethod
    def from_numpy(cls, ctx: Context, a, dtype: int = N.F64) -> "Points":
        a = np.ascontiguousarray(a, dtype=np.float64)
        if a.ndim != 2 or a.shape[1] not in (2, 3):
            raise ValueError("expected an (N, 2) or (N, 3) array")
        p = cls(ctx, a.shape[1], a.shape[0], dtype)
        p.upload(a)
        return p

    def upload(self, a: np.ndarray):
        a = np.ascontiguousarray(a, dtype=np.float64)
        self.ctx.check(_lib.acm_points_upload_aos_f64(self.ctx.handle, self._h, a.ctypes.data_as(C.c_void_p), a.shape[0]))
        self.ctx.sync()  # `a` may be a temporary

    def numpy(self) -> np.ndarray:
        n = len(self)
        out = np.empty((n, self.dim), dtype=np.float64)
        self.ctx.check(_lib.acm_points_download_aos_f64(self.ctx.handle, self._h, out.ctypes.data_as(C.c_void_p), n))
        return out

    def component_ptr(self, c: int) -> int:
        return _lib.acm_points_component(self._h, c)

    def free(self):
        if self._h:
            _lib.acm_points_destroy(self.ctx.handle, self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            if self.ctx.handle:
                self.free()
        except Exception:
            pass


class Staging:
    """The device temporaries of one call: raw buffers and `Points`.  Everything it owns is freed when its `with` block
    ends, whether the block returns or raises; `keep` hands objects to the caller instead."""

    def __init__(self, ctx: Context):
        self.ctx = ctx
        self._owned = []

    def alloc(self, nbytes: int) -> int:
        """A device buffer of max(nbytes, 1) bytes."""
        return self.own(self.ctx.device_alloc(max(nbytes, 1)))

    def points(self, a, dim: int, dtype: int = N.F64) -> Points:
        """`a` itself if it is `Points` (not owned), else `a` as (-1, dim) float64 uploaded to new owned `Points`."""
        if isinstance(a, Points):
            return a
        a = np.ascontiguousarray(a, dtype=np.float64).reshape(-1, dim)
        p = self.own(Points(self.ctx, dim, a.shape[0], dtype))
        p.upload(a)
        return p

    def own(self, obj):
        self._owned.append(obj)
        return obj

    def keep(self, *objs):
        """Releases `objs` to the caller and returns them."""
        for o in objs:
            self._owned.remove(o)
        return objs

    def close(self):
        """Frees everything owned, going on past a failed free; raises the first failure at the end."""
        owned, self._owned = self._owned, []
        err = None
        for o in owned:
            try:
                if isinstance(o, Points):
                    o.free()
                else:
                    self.ctx.device_free(o)
            except Exception as e:
                err = err or e
        if err is not None:
            raise err

    def __enter__(self):
        return self

    def __exit__(self, exc_type, exc, tb):
        try:
            self.close()
        except Exception:
            if exc_type is None:
                raise
