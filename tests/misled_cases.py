"""Chunks whose trailing bytes pass every check of the segment index but do not describe the stream in front of them
(recompress_cases.misleading_chunk).  zlib ignores such bytes, so decompress, verify and recompress must decode each
such chunk again as a plain zlib stream inside its sub-batch, whether or not the caller asks for statuses.  Each case
runs through the host emulation (tests/test_emu_misled.py) and on the B200 (tests/test_gpu_misled.py), with a context
whose host-buffer sub-batches are 1 MiB (`small_batches`), so that a call with a host buffer has several.

With host buffers, decode sub-batches close only before a plain stream here, so the chunks fall in three sub-batches,
[0], [1, 6] and [7, 9], and recompress ones (by raw bytes) in [0, 4], [5, 7] and [8, 9]: misled chunks come first in
the call, as a pair inside one sub-batch, and last in the call."""
import ctypes as C

import numpy as np

from mtscomp_b200 import _native
from recompress_cases import PLACEMENTS, misleading_chunk, recompress_at, reference_streams

NC = 16
ROWS = np.cumsum([0, 3000, 11001, 10003, 2500, 3999, 14000, 3500, 11003, 9500, 2100]).astype(np.int64)
FLAGS = _native.TIME_DIFF
MISLED = (0, 3, 4, 9)
BROKEN = 6          # misled, and corrupt as a plain stream too
CORRUPT = 7         # an ordinary plain stream with a damaged byte


def small_batches(codec):
    codec.set_param('host_batch_bytes', 1 << 20)
    codec.set_param('par_batch_bytes', 1 << 20)
    return codec


def _flip(part, pos):
    b = bytearray(part)
    b[pos] ^= 0x5a
    return bytes(b)


def _join(parts):
    return b''.join(parts), np.concatenate(([0], np.cumsum([len(p) for p in parts]))).astype(np.int64)


def build(codec):
    """-> (data, (clean blob, offsets), (bad blob, offsets)): plain reference streams with misleading chunks at MISLED
    and BROKEN; in the bad blob BROKEN's foreign stream and CORRUPT are damaged."""
    rng = np.random.default_rng(21)
    data = np.cumsum(rng.integers(-40, 41, (int(ROWS[-1]), NC)), axis=0).astype(np.int16)
    comp, offs = reference_streams(data, ROWS, FLAGS)
    parts = [comp[offs[i]:offs[i + 1]] for i in range(len(ROWS) - 1)]
    for i in MISLED + (BROKEN,):
        parts[i] = misleading_chunk(codec, data[ROWS[i]:ROWS[i + 1]], FLAGS)
    bad = list(parts)
    bad[BROKEN] = _flip(bad[BROKEN], 30)
    bad[CORRUPT] = _flip(bad[CORRUPT], 20)
    return data, _join(parts), _join(bad)


def _at(codec, host, dev, allocs):
    """The address of `host`, or of a device copy of it (appended to allocs)."""
    if not dev:
        return host.ctypes.data
    p = codec.device_alloc(host.nbytes + 256)
    allocs.append(p)
    codec.memcpy(p, host.ctypes.data, host.nbytes, 1)
    return p


def _decompress_at(codec, blob, offs, comp_dev, dst_dev):
    comp, out = np.frombuffer(blob, np.uint8), np.zeros((int(ROWS[-1]), NC), np.int16)
    allocs = []
    try:
        dst = _at(codec, out, dst_dev, allocs)
        st = codec.decompress_ptr(_at(codec, comp, comp_dev, allocs), comp_dev, offs, ROWS, NC, 2, FLAGS, dst, dst_dev)
        if dst_dev:
            codec.memcpy(out.ctypes.data, dst, out.nbytes, 2)
        return out, st
    finally:
        for p in allocs:
            codec.device_free(p)


def _verify_at(codec, blob, offs, ref, comp_dev, ref_dev):
    comp = np.frombuffer(blob, np.uint8)
    allocs = []
    try:
        return codec.verify_ptr(_at(codec, comp, comp_dev, allocs), comp_dev, offs, ROWS, NC, 2, FLAGS,
                                _at(codec, ref, ref_dev, allocs), ref_dev, 0, 0)
    finally:
        for p in allocs:
            codec.device_free(p)


def _good(i):
    return i not in (BROKEN, CORRUPT)


def case_decompress(codec, built):
    data, _, (blob, offs) = built
    for comp_dev, dst_dev in PLACEMENTS:
        out, st = _decompress_at(codec, blob, offs, comp_dev, dst_dev)
        assert np.flatnonzero(st).tolist() == [BROKEN, CORRUPT], (comp_dev, dst_dev)
        for i in filter(_good, range(len(ROWS) - 1)):
            assert np.array_equal(out[ROWS[i]:ROWS[i + 1]], data[ROWS[i]:ROWS[i + 1]]), (i, comp_dev, dst_dev)


def case_verify(codec, built):
    data, _, (blob, offs) = built
    ref = data.copy()
    plant = [(ROWS[0], 0), (ROWS[3] + 17, 5), (ROWS[4] - 1, NC - 1), (ROWS[4] + 2, 3), (ROWS[5] + 9, 1),
             (ROWS[BROKEN] + 4, 4), (ROWS[-1] - 1, NC - 1)]
    for r, ch in plant:
        ref[r, ch] += 1
    want_m, want_f = [], []
    for i in range(len(ROWS) - 1):
        diff = (ref[ROWS[i]:ROWS[i + 1]] != data[ROWS[i]:ROWS[i + 1]]).ravel()
        want_m.append(int(diff.sum()) if _good(i) else -1)
        want_f.append(int(np.flatnonzero(diff)[0]) if _good(i) and diff.any() else -1)
    assert [want_m[i] for i in MISLED] == [1, 2, 1, 1]
    for comp_dev, ref_dev in PLACEMENTS:
        st, m, f = _verify_at(codec, blob, offs, ref, comp_dev, ref_dev)
        assert np.flatnonzero(st).tolist() == [BROKEN, CORRUPT], (comp_dev, ref_dev)
        assert (m.tolist(), f.tolist()) == (want_m, want_f), (comp_dev, ref_dev)


def case_recompress(codec, built):
    data, (blob, offs), _ = built
    for wi in (1, 0):
        codec.set_param('write_index', wi)
        try:
            want, want_offs = codec.compress(data, ROWS, FLAGS)
            for comp_dev, dst_dev in PLACEMENTS:
                out, new_offs, st = recompress_at(codec, blob, offs, ROWS, NC, 2, FLAGS, comp_dev, dst_dev)
                assert not st.any(), (wi, comp_dev, dst_dev)
                assert out == want.tobytes() and new_offs.tolist() == want_offs.tolist(), (wi, comp_dev, dst_dev)
        finally:
            codec.set_param('write_index', 1)


def case_decompress_without_status(codec, built):
    """mtsb_decompress_chunks with chunk_status NULL: misled chunks decode; a corrupt one fails the call."""
    data, clean, bad = built
    pll = C.POINTER(C.c_longlong)
    rows = np.ascontiguousarray(ROWS)
    for (blob, offs), want_rc in ((clean, 0), (bad, _native.E_CORRUPT)):
        comp, out = np.frombuffer(blob, np.uint8), np.zeros((int(ROWS[-1]), NC), np.int16)
        offs = np.ascontiguousarray(offs, np.int64)
        with codec.lock:
            rc = codec.lib.mtsb_decompress_chunks(
                codec.ctx, C.c_void_p(comp.ctypes.data), 0, offs.ctypes.data_as(pll), len(ROWS) - 1,
                rows.ctypes.data_as(pll), NC, 2, FLAGS, C.c_void_p(out.ctypes.data), 0, None)
        assert rc == want_rc
        if not rc:
            assert np.array_equal(out, data)


ALL_CASES = [case_decompress, case_verify, case_recompress, case_decompress_without_status]
