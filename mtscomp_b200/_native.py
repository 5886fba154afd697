# -*- coding: utf-8 -*-
"""ctypes binding of the C ABI in include/mtscomp_b200.h (libmtscomp_b200.so, built by mtscomp_b200/build.py).

There is no CPU fallback: if the shared library is missing, or no CUDA device is usable, the product path raises
`NativeUnavailable` with the reason.
"""

import ctypes as C
import os
import threading
from pathlib import Path

import numpy as np

_PKG = Path(__file__).resolve().parent
LIB_PATH = _PKG / '_build' / 'libmtscomp_b200.so'

TIME_DIFF, SPATIAL_DIFF, ORDER_C, FLOAT = 1, 2, 4, 8


def _fl(flags, dtype):
    """flags with the FLOAT bit set for floating point dtypes (the array-level helpers below add it themselves)."""
    return flags | FLOAT if np.dtype(dtype).kind == 'f' else flags
E_CORRUPT = -5

SYMBOLS = (
    'mtsb_version', 'mtsb_device_count', 'mtsb_create', 'mtsb_destroy', 'mtsb_last_error', 'mtsb_sync',
    'mtsb_set_param', 'mtsb_get_param', 'mtsb_compress_bound', 'mtsb_delta_transform', 'mtsb_inverse_transform',
    'mtsb_compress_chunks', 'mtsb_decompress_chunks', 'mtsb_verify_chunks', 'mtsb_recompress_chunks',
    'mtsb_last_timings', 'mtsb_last_launches',
    'mtsb_host_alloc', 'mtsb_host_free', 'mtsb_device_alloc', 'mtsb_device_free', 'mtsb_memcpy')


class NativeUnavailable(RuntimeError):
    pass


class NativeError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__('mtscomp_b200 native error %d: %s' % (code, msg))
        self.code = code


def _declare(lib):
    vp, ll, i = C.c_void_p, C.c_longlong, C.c_int
    pll = C.POINTER(C.c_longlong)
    lib.mtsb_version.restype = i
    lib.mtsb_device_count.restype = i
    lib.mtsb_create.restype = vp
    lib.mtsb_create.argtypes = [i, vp]
    lib.mtsb_destroy.argtypes = [vp]
    lib.mtsb_destroy.restype = None
    lib.mtsb_last_error.restype = C.c_char_p
    lib.mtsb_last_error.argtypes = [vp]
    lib.mtsb_sync.argtypes = [vp]
    lib.mtsb_set_param.argtypes = [vp, C.c_char_p, ll]
    lib.mtsb_get_param.argtypes = [vp, C.c_char_p]
    lib.mtsb_get_param.restype = ll
    lib.mtsb_compress_bound.argtypes = [vp, ll, ll, i, i, i]
    lib.mtsb_compress_bound.restype = ll
    lib.mtsb_delta_transform.argtypes = [vp, vp, i, ll, i, i, i, vp, i]
    lib.mtsb_inverse_transform.argtypes = [vp, vp, i, ll, i, i, i, vp, i, C.POINTER(C.c_uint32)]
    lib.mtsb_compress_chunks.argtypes = [vp, vp, i, i, pll, i, i, i, vp, i, ll, pll]
    lib.mtsb_decompress_chunks.argtypes = [vp, vp, i, pll, i, pll, i, i, i, vp, i, C.POINTER(C.c_int)]
    lib.mtsb_verify_chunks.argtypes = [vp, vp, i, pll, i, pll, i, i, i, vp, i, C.c_double, C.c_double, pll, pll,
                                       C.POINTER(C.c_int)]
    lib.mtsb_recompress_chunks.argtypes = [vp, vp, i, pll, i, pll, i, i, i, vp, i, ll, pll, C.POINTER(C.c_int)]
    lib.mtsb_last_timings.argtypes = [vp, C.POINTER(C.c_float), i]
    lib.mtsb_last_launches.argtypes = [vp]
    lib.mtsb_last_launches.restype = ll
    lib.mtsb_host_alloc.argtypes = [ll]
    lib.mtsb_host_alloc.restype = vp
    lib.mtsb_host_free.argtypes = [vp]
    lib.mtsb_host_free.restype = None
    lib.mtsb_device_alloc.argtypes = [vp, ll]
    lib.mtsb_device_alloc.restype = vp
    lib.mtsb_device_free.argtypes = [vp, vp]
    lib.mtsb_device_free.restype = None
    lib.mtsb_memcpy.argtypes = [vp, vp, vp, ll, i]
    return lib


class HostBuffer:
    """Pinned host memory from mtsb_host_alloc, visible as a NumPy uint8 array (`.array`) and a raw pointer (`.ptr`).
    Views of `.array` must not outlive the buffer."""

    def __init__(self, lib, nbytes):
        self.lib, self.nbytes = lib, int(nbytes)
        self.ptr = lib.mtsb_host_alloc(self.nbytes)
        if not self.ptr:
            raise MemoryError('mtsb_host_alloc(%d) failed' % self.nbytes)
        self.array = np.ctypeslib.as_array((C.c_ubyte * self.nbytes).from_address(self.ptr))

    def release(self):
        if self.ptr:
            self.array = None
            self.lib.mtsb_host_free(C.c_void_p(self.ptr))
            self.ptr = None

    def __del__(self):
        try:
            self.release()
        except Exception:
            pass


_lib = None
_lib_lock = threading.Lock()


def load_library(path=None):
    """dlopen the native library (no device needed).  `path` is for development tools only."""
    global _lib
    if path is not None:
        return _declare(C.CDLL(str(path)))
    with _lib_lock:
        if _lib is None:
            p = Path(os.environ.get('MTSCOMP_B200_LIB', LIB_PATH))
            if not p.exists():
                raise NativeUnavailable(
                    '%s not found: build it with `python -m mtscomp_b200.build` (nvcc, sm_100a). '
                    'mtscomp_b200 has no CPU fallback.' % p)
            _lib = _declare(C.CDLL(str(p)))
        return _lib


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def _i64(seq):
    return np.ascontiguousarray(np.asarray(seq, dtype=np.int64))


class Codec:
    """One native context (one CUDA device, one stream).  Thread-safe through an internal lock."""

    def __init__(self, device=0, stream=None, lib=None):
        self.lib = lib or load_library()
        if self.lib.mtsb_device_count() < 1:
            raise NativeUnavailable('no CUDA device visible; mtscomp_b200 has no CPU fallback.')
        self.ctx = self.lib.mtsb_create(int(device), C.c_void_p(stream) if stream else None)
        if not self.ctx:
            raise NativeUnavailable('mtsb_create failed: %s' % self.lib.mtsb_last_error(None).decode())
        self.device = int(device)
        self.lock = threading.Lock()
        self.stage_lock = threading.RLock()     # guards the named staging buffers below (one user at a time)
        self._staging = {}
        # tunables for experiments without touching code: MTSCOMP_B200_PARAMS="par_batch_bytes=4294967296,max_chain=8"
        for kv in filter(None, os.environ.get('MTSCOMP_B200_PARAMS', '').split(',')):
            k, v = kv.split('=')
            self.set_param(k.strip(), int(v))

    def close(self):
        if getattr(self, 'ctx', None):
            for b in self._staging.values():
                b.release()
            self._staging.clear()
            self.lib.mtsb_destroy(self.ctx)
            self.ctx = None

    # -- pinned staging and device memory (the Python layer's I/O buffers)
    def host_buffer(self, name, nbytes):
        """Named pinned buffer of at least `nbytes`, kept for reuse and grown on demand (hold `stage_lock` while the
        contents matter)."""
        b = self._staging.get(name)
        if b is None or b.nbytes < nbytes:
            if b is not None:
                b.release()
            # (pinning is slow: grow in large steps so that a Reader asked for ever wider windows re-pins rarely)
            b = self._staging[name] = HostBuffer(self.lib, max(2 * int(nbytes), 1 << 20))
        return b

    def device_alloc(self, nbytes):
        p = self.lib.mtsb_device_alloc(self.ctx, int(nbytes))
        if not p:
            raise MemoryError('mtsb_device_alloc(%d) failed' % nbytes)
        return p

    def device_free(self, ptr):
        if getattr(self, 'ctx', None) and ptr:
            self.lib.mtsb_device_free(self.ctx, C.c_void_p(ptr))

    def memcpy(self, dst, src, nbytes, kind):
        """kind 1: host -> device, 2: device -> host, 3: device -> device (synchronous)."""
        with self.lock:
            self._check(self.lib.mtsb_memcpy(self.ctx, C.c_void_p(dst), C.c_void_p(src), int(nbytes), int(kind)))

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            raise NativeError(rc, self.lib.mtsb_last_error(self.ctx).decode())

    # -- parameters
    def set_param(self, name, value):
        self._check(self.lib.mtsb_set_param(self.ctx, name.encode(), int(value)))

    def get_param(self, name):
        return int(self.lib.mtsb_get_param(self.ctx, name.encode()))

    def compress_bound(self, ns, nc, itemsize, flags):
        return int(self.lib.mtsb_compress_bound(self.ctx, int(ns) * nc * itemsize, int(ns), nc, itemsize, flags))

    def timings(self):
        buf = (C.c_float * 8)()
        n = self.lib.mtsb_last_timings(self.ctx, buf, 8)
        return [float(buf[i]) for i in range(n)]

    def launches(self):
        return int(self.lib.mtsb_last_launches(self.ctx))

    # -- raw-pointer entry points (host or device pointers; used by bench.py with resident buffers)
    def compress_ptr(self, src, src_is_device, chunk_rows, nc, itemsize, flags, dst, dst_is_device, dst_capacity):
        rows = _i64(chunk_rows)
        n = len(rows) - 1
        offs = np.zeros(n + 1, dtype=np.int64)
        pll = C.POINTER(C.c_longlong)
        with self.lock:
            self._check(self.lib.mtsb_compress_chunks(
                self.ctx, C.c_void_p(src), int(src_is_device), n, rows.ctypes.data_as(pll), nc, itemsize, flags,
                C.c_void_p(dst), int(dst_is_device), int(dst_capacity), offs.ctypes.data_as(pll)))
        return offs

    def decompress_ptr(self, comp, comp_is_device, comp_offsets, chunk_rows, nc, itemsize, flags, dst, dst_is_device):
        rows, offs = _i64(chunk_rows), _i64(comp_offsets)
        n = len(rows) - 1
        status = np.zeros(n, dtype=np.int32)
        pll = C.POINTER(C.c_longlong)
        with self.lock:
            rc = self.lib.mtsb_decompress_chunks(
                self.ctx, C.c_void_p(comp), int(comp_is_device), offs.ctypes.data_as(pll), n,
                rows.ctypes.data_as(pll), nc, itemsize, flags, C.c_void_p(dst), int(dst_is_device),
                status.ctypes.data_as(C.POINTER(C.c_int)))
            if rc != 0 and rc != E_CORRUPT:
                self._check(rc)
        return status

    def verify_ptr(self, comp, comp_is_device, comp_offsets, chunk_rows, nc, itemsize, flags, ref, ref_is_device,
                   rtol, atol):
        """Decode each chunk and compare it on the device with its rows of `ref` (mtsb_verify_chunks) ->
        (status int32[n], mismatches int64[n], first_mismatch int64[n]); -1 in both counters where a chunk is corrupt."""
        rows, offs = _i64(chunk_rows), _i64(comp_offsets)
        n = len(rows) - 1
        status = np.zeros(n, dtype=np.int32)
        mism, first = np.zeros(n, dtype=np.int64), np.zeros(n, dtype=np.int64)
        pll = C.POINTER(C.c_longlong)
        with self.lock:
            rc = self.lib.mtsb_verify_chunks(
                self.ctx, C.c_void_p(comp), int(comp_is_device), offs.ctypes.data_as(pll), n,
                rows.ctypes.data_as(pll), nc, itemsize, flags, C.c_void_p(ref), int(ref_is_device), float(rtol),
                float(atol), mism.ctypes.data_as(pll), first.ctypes.data_as(pll), status.ctypes.data_as(C.POINTER(C.c_int)))
            if rc != 0 and rc != E_CORRUPT:
                self._check(rc)
        return status, mism, first

    def recompress_ptr(self, comp, comp_is_device, comp_offsets, chunk_rows, nc, itemsize, flags, dst, dst_is_device,
                       dst_capacity):
        """Inflate each chunk to its transformed bytes and deflate them again with the codec's current parameters
        (mtsb_recompress_chunks) -> (out_offsets int64[n+1], status int32[n]).  Where a status is non-zero the output
        is undefined."""
        rows, offs = _i64(chunk_rows), _i64(comp_offsets)
        n = len(rows) - 1
        out = np.zeros(n + 1, dtype=np.int64)
        status = np.zeros(n, dtype=np.int32)
        pll = C.POINTER(C.c_longlong)
        with self.lock:
            rc = self.lib.mtsb_recompress_chunks(
                self.ctx, C.c_void_p(comp), int(comp_is_device), offs.ctypes.data_as(pll), n,
                rows.ctypes.data_as(pll), nc, itemsize, flags, C.c_void_p(dst), int(dst_is_device), int(dst_capacity),
                out.ctypes.data_as(pll), status.ctypes.data_as(C.POINTER(C.c_int)))
            if rc != 0 and rc != E_CORRUPT:
                self._check(rc)
        return out, status

    # -- NumPy conveniences (host arrays)
    def delta_transform(self, chunk, flags):
        chunk = np.ascontiguousarray(chunk)
        assert chunk.ndim == 2
        out = np.empty(chunk.nbytes, dtype=np.uint8)
        with self.lock:
            self._check(self.lib.mtsb_delta_transform(
                self.ctx, _ptr(chunk), 0, chunk.shape[0], chunk.shape[1], chunk.dtype.itemsize, _fl(flags, chunk.dtype),
                _ptr(out), 0))
        return out

    def inverse_transform(self, buf, ns, nc, dtype, flags, want_adler=False):
        dtype = np.dtype(dtype)
        src = np.frombuffer(buf, dtype=np.uint8)
        assert src.size == ns * nc * dtype.itemsize
        src = np.ascontiguousarray(src)
        out = np.empty((ns, nc), dtype=dtype)
        ad = C.c_uint32(0)
        with self.lock:
            self._check(self.lib.mtsb_inverse_transform(
                self.ctx, _ptr(src), 0, ns, nc, dtype.itemsize, _fl(flags, dtype), _ptr(out), 0,
                C.byref(ad) if want_adler else None))
        return (out, int(ad.value)) if want_adler else out

    def compress(self, data, chunk_rows, flags):
        """data: C-contiguous (n_samples, nc) array; returns (bytes-like uint8 array, offsets int64[n+1])."""
        data = np.ascontiguousarray(data)
        rows = _i64(chunk_rows)
        nc, isz = data.shape[1], data.dtype.itemsize
        flags = _fl(flags, data.dtype)
        cap = sum(self.compress_bound(int(rows[i + 1] - rows[i]), nc, isz, flags) for i in range(len(rows) - 1))
        dst = np.empty(cap, dtype=np.uint8)
        offs = self.compress_ptr(data.ctypes.data, 0, rows, nc, isz, flags, dst.ctypes.data, 0, cap)
        return dst[:int(offs[-1])], offs

    def decompress(self, comp, comp_offsets, chunk_rows, nc, dtype, flags):
        """comp: bytes-like; returns ((n_samples, nc) array, status int32[n])."""
        dtype = np.dtype(dtype)
        comp = np.frombuffer(comp, dtype=np.uint8)
        rows = _i64(chunk_rows)
        out = np.empty((int(rows[-1]), nc), dtype=dtype)
        status = self.decompress_ptr(comp.ctypes.data, 0, comp_offsets, rows, nc, dtype.itemsize, _fl(flags, dtype),
                                     out.ctypes.data, 0)
        return out, status


    def verify(self, comp, comp_offsets, chunk_rows, ref, flags, rtol=1e-5, atol=1e-16):
        """comp: bytes-like; ref: C-contiguous (n_samples, nc) array -> (status, mismatches, first_mismatch)."""
        ref = np.ascontiguousarray(ref)
        comp = np.frombuffer(comp, dtype=np.uint8)
        return self.verify_ptr(comp.ctypes.data, 0, comp_offsets, chunk_rows, ref.shape[1], ref.dtype.itemsize,
                               _fl(flags, ref.dtype), ref.ctypes.data, 0, rtol, atol)

    def recompress(self, comp, comp_offsets, chunk_rows, nc, dtype, flags):
        """comp: bytes-like -> (bytes-like uint8 array, offsets int64[n+1], status int32[n])."""
        dtype = np.dtype(dtype)
        comp = np.frombuffer(comp, dtype=np.uint8)
        rows = _i64(chunk_rows)
        flags = _fl(flags, dtype)
        cap = sum(self.compress_bound(int(rows[i + 1] - rows[i]), nc, dtype.itemsize, flags)
                  for i in range(len(rows) - 1))
        dst = np.empty(cap, dtype=np.uint8)
        offs, status = self.recompress_ptr(comp.ctypes.data, 0, comp_offsets, rows, nc, dtype.itemsize, flags,
                                           dst.ctypes.data, 0, cap)
        return dst[:int(offs[-1])], offs, status


_default = {}
_default_lock = threading.Lock()


def default_codec(device=None):
    """Process-wide codec for `device` (default: $LOCAL_RANK or 0), created on first use."""
    if device is None:
        device = int(os.environ.get('MTSCOMP_B200_DEVICE', os.environ.get('LOCAL_RANK', 0)))
    with _default_lock:
        if device not in _default:
            _default[device] = Codec(device)
        return _default[device]


def flags_of(do_time_diff, do_spatial_diff, chunk_order):
    assert chunk_order in ('F', 'C')
    return (TIME_DIFF if do_time_diff else 0) | (SPATIAL_DIFF if do_spatial_diff else 0) | \
        (ORDER_C if chunk_order == 'C' else 0)
