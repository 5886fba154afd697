"""Shared helpers of the recompress suites (tests/test_emu_recompress.py, tests/test_gpu_recompress.py), also used by the
misled-index cases (tests/misled_cases.py, tests/test_emu_verify.py)."""
import json
import struct
import zlib
from pathlib import Path

import numpy as np

from mtscomp_b200 import _native
from oracle import codec as ora

GOLDEN = Path(__file__).resolve().parent / 'golden'
MANIFEST = json.loads((GOLDEN / 'manifest.json').read_text())
INT_GOLDENS = sorted(MANIFEST['cases'])
FLOAT_GOLDENS = sorted(MANIFEST['float_cases'])
PLACEMENTS = [(0, 0), (0, 1), (1, 0), (1, 1)]     # (comp_is_device, dst_is_device)


def golden(name):
    """-> (manifest entry, .ch dict, raw rows, .cbin bytes, flags without MTSB_FLOAT)."""
    m = MANIFEST['cases'].get(name) or MANIFEST['float_cases'][name]
    meta = json.loads((GOLDEN / (name + '.ch')).read_text())
    raw = np.fromfile(GOLDEN / (name + '.bin'), dtype=meta['dtype']).reshape(-1, meta['n_channels'])
    flags = _native.flags_of(meta['do_time_diff'], meta['do_spatial_diff'], meta['chunk_order'])
    return m, meta, raw, (GOLDEN / (name + '.cbin')).read_bytes(), flags


def inflated(blob, offsets):
    """What CPython's zlib inflates each chunk to (it ignores the bytes after a stream)."""
    blob = bytes(blob)
    return [zlib.decompress(blob[int(offsets[i]):int(offsets[i + 1])]) for i in range(len(offsets) - 1)]


def reference_streams(data, rows, flags):
    """One zlib level-6 stream per chunk of the transformed rows, as the reference Writer writes them
    -> (bytes, offsets)."""
    kw = dict(do_time_diff=bool(flags & _native.TIME_DIFF), do_spatial_diff=bool(flags & _native.SPATIAL_DIFF),
              chunk_order='C' if flags & _native.ORDER_C else 'F')
    parts = [ora.encode_chunk(data[rows[i]:rows[i + 1]], **kw) for i in range(len(rows) - 1)]
    return b''.join(parts), np.concatenate(([0], np.cumsum([len(p) for p in parts]))).astype(np.int64)


def misleading_chunk(codec, data, flags):
    """One chunk: a zlib stream of the chunk's transformed bytes written by CPython's zlib, followed by the segment
    index of the GPU's own stream of the same rows, its last length adjusted so that the index passes every check of
    the decoder, yet does not describe that stream.  (The decoder takes the segments to end 2 bytes before the adler32
    trailer, where the GPU's own streams close with an empty final block.)"""
    rows = np.array([0, data.shape[0]], np.int64)
    gpu, _ = codec.compress(data, rows, flags)
    d = zlib.decompressobj()
    d.decompress(gpu.tobytes())
    index = d.unused_data
    foreign = zlib.compress(ora.transform_chunk(data), 1)
    sb, k, magic, total = struct.unpack('<4I', index[-16:])
    v2 = len(index) > 4 * k + 16
    lens_end = len(index) - 16 - (8 if v2 else 0)
    lens = list(struct.unpack('<%dI' % k, index[lens_end - 4 * k:lens_end]))
    body = len(foreign) - 8
    lens[-1] += body - sum(lens)
    assert lens[-1] > 0
    index = (index[:lens_end - 4 * k] + struct.pack('<%dI' % k, *lens) + index[lens_end:-4] + struct.pack('<I', body))
    return foreign + index


def recompress_at(codec, comp, offs, rows, nc, itemsize, flags, comp_dev, dst_dev):
    """codec.recompress_ptr with `comp` and the output in host or device memory -> (output bytes, offsets, status)."""
    comp = np.frombuffer(bytes(comp), np.uint8)
    cap = sum(codec.compress_bound(int(rows[i + 1] - rows[i]), nc, itemsize, flags) for i in range(len(rows) - 1))
    allocs = []
    try:
        src = comp.ctypes.data
        if comp_dev:
            src = codec.device_alloc(comp.nbytes + 256)
            allocs.append(src)
            codec.memcpy(src, comp.ctypes.data, comp.nbytes, 1)
        host = np.zeros(cap, np.uint8)
        dst = host.ctypes.data
        if dst_dev:
            dst = codec.device_alloc(cap + 256)
            allocs.append(dst)
        out, st = codec.recompress_ptr(src, comp_dev, offs, rows, nc, itemsize, flags, dst, dst_dev, cap)
        if dst_dev and not st.any():
            codec.memcpy(host.ctypes.data, dst, int(out[-1]), 2)
        return host[:int(out[-1])].tobytes(), out, st
    finally:
        for a in allocs:
            codec.device_free(a)
