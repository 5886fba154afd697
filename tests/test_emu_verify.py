"""CPU: mtsb_verify_chunks (the integrity check's decode + compare) and check() through the host emulation of the
kernels.  Every verdict is compared with NumPy's on the rows mtsb_decompress_chunks decodes: `!=` for integers,
~np.isclose(decoded, ref, rtol, atol) for floats."""
import ctypes as C
import json
import zlib

import numpy as np
import pytest
from pytest import raises

import mtscomp_b200 as M
from mtscomp_b200 import _native
from mtscomp_b200.config import CHECK_ATOL
from mtscomp_b200.core import CHECK_RTOL
from recompress_cases import misleading_chunk

DTYPES = (np.uint8, np.int16, np.int32, np.int64, np.float32, np.float64)
ROWS = np.array([0, 301, 302, 1033, 1500, 2211, 2212, 2900], np.int64)   # ragged, with one-row chunks


@pytest.fixture(scope='module')
def emu():
    from mtscomp_b200 import build
    c = _native.Codec(0, lib=_native.load_library(build.build_emulation()))
    # the smallest host-buffer sub-batches (test_verify_several_sub_batches has enough chunks to fill several)
    c.set_param('host_batch_bytes', 1 << 20)
    c.set_param('par_batch_bytes', 1 << 20)
    yield c
    c.close()


def _data(dt, nc, seed, ns=int(ROWS[-1])):
    rng = np.random.default_rng(seed)
    walk = np.cumsum(rng.integers(-40, 41, (ns, nc)), axis=0)
    if np.dtype(dt).kind == 'f':
        return (walk / 7.3 + 20000.).astype(dt)
    return walk.astype(dt)


def _expected(dec, ref, rows):
    if dec.dtype.kind == 'f':
        bad = ~np.isclose(dec, ref, rtol=CHECK_RTOL, atol=CHECK_ATOL)
    else:
        bad = dec != ref
    m, f = [], []
    for i in range(len(rows) - 1):
        b = bad[rows[i]:rows[i + 1]].ravel()
        m.append(int(b.sum()))
        f.append(int(np.flatnonzero(b)[0]) if b.any() else -1)
    return m, f


def _verify(codec, comp, offs, rows, ref, flags):
    st, m, f = codec.verify(comp.tobytes(), offs, rows, ref, flags, CHECK_RTOL, CHECK_ATOL)
    return st, m.tolist(), f.tolist()


def _plant(ref, rows, nc):
    """Differences at chunk starts and ends (the borders of the sub-batches are chunk borders), first and last
    channel, and inside a chunk."""
    out = ref.copy()
    one = np.array(1, out.dtype)
    for r, ch in ((rows[1], 0), (rows[2] - 1, nc - 1), (rows[3], nc - 1), (rows[4] - 1, 0), (rows[5] + 7, nc // 2),
                  (rows[-1] - 1, nc - 1)):
        out[r, ch] = out[r, ch] + one
    return out


@pytest.mark.parametrize('dt', DTYPES, ids=lambda d: np.dtype(d).name)
@pytest.mark.parametrize('order', ['F', 'C'])
@pytest.mark.parametrize('spatial', [False, True], ids=['time', 'time+spatial'])
def test_verify_matches_numpy(emu, dt, order, spatial):
    nc = 37 if order == 'F' else 12
    flags = _native.flags_of(True, spatial, order)
    data = _data(dt, nc, 3)
    comp, offs = emu.compress(data, ROWS, flags)
    dec, st = emu.decompress(comp, offs, ROWS, nc, dt, flags)
    assert not st.any()
    for ref in (dec, data, _plant(dec, ROWS, nc)):
        st, m, f = _verify(emu, comp, offs, ROWS, ref, flags)
        assert not st.any()
        assert (m, f) == _expected(dec, ref, ROWS)
    assert emu.timings()[6] > 0 and emu.launches() > 0


@pytest.mark.parametrize('dt', [np.int16, np.float64], ids=['int16', 'float64'])
def test_verify_several_sub_batches(emu, dt):
    """Enough chunks (a sub-batch closes at 1 MB once it holds 8 streams per SM) for three sub-batches, so that the
    reference rows go up through both buffers of their pair, with differences at the sub-batches' borders."""
    nc, n = 40, 150
    rows = np.arange(n + 1, dtype=np.int64) * 200
    rows[-1] -= 13
    flags = _native.flags_of(True, False, 'F')
    data = _data(dt, nc, 12, int(rows[-1]))
    comp, offs = emu.compress(data, rows, flags)
    dec, _ = emu.decompress(comp, offs, rows, nc, dt, flags)
    ref = dec.copy()
    for i in (0, 63, 64, 65, 127, 128, 149):
        ref[rows[i], 0] += np.array(1, dt)
        ref[rows[i + 1] - 1, nc - 1] += np.array(1, dt)
    st, m, f = _verify(emu, comp, offs, rows, ref, flags)
    assert not st.any() and (m, f) == _expected(dec, ref, rows) and sum(m) == 14
    split = emu.launches()
    emu.set_param('host_batch_bytes', 1 << 40)
    try:
        assert _verify(emu, comp, offs, rows, ref, flags)[1:] == (m, f)
        assert emu.launches() < split                        # one sub-batch: fewer launches
    finally:
        emu.set_param('host_batch_bytes', 1 << 20)


def _tolerance_edges(y, dt):
    """Reference values one and two ulps either side of where |x - y| crosses atol + rtol * |y| (x fixed)."""
    dt = np.dtype(dt)
    edge = (y.astype(np.float64) * (1 + CHECK_RTOL)).astype(dt)
    cand = [edge]
    for k in (1, 2):
        up, down = edge, edge
        for _ in range(k):
            up = np.nextafter(up, dt.type(np.inf))
            down = np.nextafter(down, dt.type(-np.inf))
        cand += [up, down]
    return cand


@pytest.mark.parametrize('dt', (np.float32, np.float64), ids=lambda d: np.dtype(d).name)
@pytest.mark.parametrize('time_diff', [False, True])
def test_verify_float_edges_and_specials(emu, dt, time_diff):
    nc, rows = 16, np.array([0, 40, 97, 150], np.int64)
    dt = np.dtype(dt)
    flags = _native.flags_of(time_diff, False, 'F')
    fi = np.finfo(dt)
    specials = np.array([np.nan, np.inf, -np.inf, 0., -0., fi.max, -fi.max, fi.tiny, 1.], dt)
    data = (np.random.default_rng(5).normal(0, 1000, (150, nc)) + 3000).astype(dt)
    data[41, :len(specials)] = specials            # special values in the data ...
    data[149, -len(specials):] = specials[::-1]
    comp, offs = emu.compress(data, rows, flags)
    dec, st = emu.decompress(comp, offs, rows, nc, dt, flags)
    ref = dec.copy()
    for j in range(5):                                   # ... pairs at the tolerance's edge ...
        r0 = 2 + 10 * (j % 3)
        ref[r0:r0 + 10, 4 + j] = _tolerance_edges(dec[r0:r0 + 10, 4 + j], dt)[j]
    ref[100, :len(specials)] = specials                  # ... and in the reference, against finite and special data
    ref[41, 1:len(specials)] = specials[:-1]
    ref[149, -len(specials):] = specials
    ref[120, 0] = np.nextafter(dec[120, 0], dt.type(np.inf))
    ref[121, 0] = -dec[121, 0]
    with np.errstate(invalid='ignore', over='ignore'):
        want = _expected(dec, ref, rows)
        st, m, f = _verify(emu, comp, offs, rows, ref, flags)
    assert not st.any()
    assert (m, f) == want
    assert sum(want[0]) > 10


def _ref_arg_verify(emu, comp, offs, rows, ref, flags):
    """mtsb_verify_chunks called directly: (return code, status, mismatches, first_mismatch)."""
    n = len(rows) - 1
    st = np.zeros(n, np.int32)
    m, f = np.zeros(n, np.int64), np.zeros(n, np.int64)
    pll = C.POINTER(C.c_longlong)
    offs, rows = np.ascontiguousarray(offs, np.int64), np.ascontiguousarray(rows, np.int64)
    comp = np.frombuffer(comp, np.uint8)
    rc = emu.lib.mtsb_verify_chunks(
        emu.ctx, C.c_void_p(comp.ctypes.data), 0, offs.ctypes.data_as(pll), n, rows.ctypes.data_as(pll), ref.shape[1],
        ref.dtype.itemsize, _native._fl(flags, ref.dtype), C.c_void_p(ref.ctypes.data), 0, CHECK_RTOL, CHECK_ATOL,
        m.ctypes.data_as(pll), f.ctypes.data_as(pll), st.ctypes.data_as(C.POINTER(C.c_int)))
    return rc, st, m, f


def test_verify_corrupt_chunk(emu):
    nc, flags = 19, _native.flags_of(True, False, 'F')
    data = _data(np.int16, nc, 7)
    comp, offs = emu.compress(data, ROWS, flags)
    blob = bytearray(comp.tobytes())
    blob[int(offs[3]) + 40] ^= 0x5a
    ref = data.copy()
    ref[ROWS[5], 2] += 1
    rc, st, m, f = _ref_arg_verify(emu, bytes(blob), offs, ROWS, ref, flags)
    assert rc == _native.E_CORRUPT
    assert st[3] != 0 and m[3] == -1 and f[3] == -1
    good = [i for i in range(len(ROWS) - 1) if i != 3]
    assert not st[good].any()
    assert m[good].tolist() == [0, 0, 0, 0, 1, 0] and f[5] == 2


def test_verify_misleading_index_is_retried(emu):
    nc, flags = 19, _native.flags_of(True, False, 'F')
    data = _data(np.int16, nc, 8)[:2000]
    chunk = misleading_chunk(emu, data, flags)
    d = zlib.decompressobj()
    d.decompress(chunk)
    plain = chunk[:len(chunk) - len(d.unused_data)]          # the same stream without the bytes after it
    rows = [0, data.shape[0]]
    launches = {}
    for blob in (plain, chunk):
        offs = [0, len(blob)]
        dec, st = emu.decompress(blob, offs, rows, nc, np.int16, flags)
        assert not st.any() and np.array_equal(dec, data)
        n = emu.launches()
        assert _verify(emu, np.frombuffer(blob, np.uint8), offs, rows, data, flags) == (np.zeros(1, np.int32), [0], [-1])
        launches[blob] = (n, emu.launches())
    # the call decoded the misled chunk through its index, then again as a plain stream
    assert all(m > p for m, p in zip(launches[chunk], launches[plain])), launches.values()
    ref = data.copy()
    ref[1999, 18] += 3
    st, m, f = _verify(emu, np.frombuffer(chunk, np.uint8), [0, len(chunk)], rows, ref, flags)
    assert not st.any() and m == [1] and f == [1999 * nc + 18]


def test_verify_bad_arguments(emu):
    nc, flags = 4, _native.flags_of(True, False, 'F')
    data = _data(np.int16, nc, 9)[:100]
    comp, offs = emu.compress(data, [0, 100], flags)
    buf = np.zeros(data.nbytes + 1, np.uint8)
    odd = buf[1:].view(np.uint8)
    odd[:] = data.view(np.uint8).ravel()
    pll = C.POINTER(C.c_longlong)
    offs, rows = np.ascontiguousarray(offs, np.int64), np.array([0, 100], np.int64)
    m, f, st = np.zeros(1, np.int64), np.zeros(1, np.int64), np.zeros(1, np.int32)
    rc = emu.lib.mtsb_verify_chunks(
        emu.ctx, C.c_void_p(comp.ctypes.data), 0, offs.ctypes.data_as(pll), 1, rows.ctypes.data_as(pll), nc, 2, flags,
        C.c_void_p(odd.ctypes.data), 0, CHECK_RTOL, CHECK_ATOL, m.ctypes.data_as(pll), f.ctypes.data_as(pll),
        st.ctypes.data_as(C.POINTER(C.c_int)))
    assert rc == -2          # a reference that is not itemsize-aligned


@pytest.fixture
def emulated_default_codec(emu):
    saved = dict(_native._default)
    _native._default.clear()
    _native._default[0] = emu
    yield emu
    _native._default.clear()
    _native._default.update(saved)


@pytest.mark.parametrize('corrupt_first', [True, False])
def test_check_raises_for_the_first_failing_chunk(tmp_path, emulated_default_codec, corrupt_first):
    M.CONFIG_PATH = tmp_path / '.mtscomp'
    nc, sr = 11, 1000.
    data = _data(np.int16, nc, 10, 6500)
    path, out, outmeta = tmp_path / 'd.bin', tmp_path / 'd.cbin', tmp_path / 'd.ch'
    data.tofile(path)
    M.compress(path, out, outmeta, sample_rate=sr, n_channels=nc, dtype=np.int16, check_after_compress=False,
               quiet=True)
    o = json.loads(outmeta.read_text())['chunk_offsets']
    bad_chunk, diff_chunk = (2, 4) if corrupt_first else (4, 2)
    blob = bytearray(out.read_bytes())
    blob[o[bad_chunk] + 30] ^= 0xff
    out.write_bytes(bytes(blob))
    src = data.copy()
    src[diff_chunk * 1000 + 17, 5] += 1
    if corrupt_first:
        with raises(IOError, match='Compressed chunk #2 is corrupted'):
            M.check(src, out, outmeta)
    else:
        with raises(AssertionError, match=r'chunk #2 .* row 17 \(sample 2017\), channel 5'):
            M.check(src, out, outmeta)


def test_check_passes_and_names_the_mismatch(tmp_path, emulated_default_codec):
    M.CONFIG_PATH = tmp_path / '.mtscomp'
    nc = 7
    data = _data(np.float32, nc, 11)[:2600]
    path, out, outmeta = tmp_path / 'f.bin', tmp_path / 'f.cbin', tmp_path / 'f.ch'
    data.tofile(path)
    M.compress(path, out, outmeta, sample_rate=1000., n_channels=nc, dtype=np.float32, quiet=True)  # checks itself
    M.check(data, out, outmeta)
    src = data.copy()
    src[2599, 6] = np.float32(1.5)
    with raises(AssertionError, match=r'chunk #2 .*channel 6: decoded [0-9.e+]+, expected 1\.5'):
        M.check(src, out, outmeta)
