"""CPU: mtsb_recompress_chunks and recompress() through the host emulation of the kernels.  The encoder is
deterministic and a chunk's zlib stream inflates to its transformed bytes, so recompressing a reference-written integer
file must give exactly the bytes compress() writes from the raw samples; float files must inflate to the same bytes."""
import hashlib
import json
import shutil
import zlib

import numpy as np
import pytest
from pytest import raises

import mtscomp_b200 as M
from mtscomp_b200 import _native, core
from oracle.reader import PortReader
from recompress_cases import (
    FLOAT_GOLDENS, GOLDEN, INT_GOLDENS, PLACEMENTS, golden, inflated, misleading_chunk, recompress_at, reference_streams)

DTYPES = (np.uint8, np.int16, np.int32, np.int64, np.float32, np.float64)
ROWS = np.array([0, 301, 302, 1033, 1500, 2211, 2212, 2900], np.int64)   # ragged, with one-row chunks


@pytest.fixture(scope='module')
def emu():
    from mtscomp_b200 import build
    c = _native.Codec(0, lib=_native.load_library(build.build_emulation()))
    c.set_param('host_batch_bytes', 1 << 20)     # the smallest host-buffer sub-batches
    c.set_param('par_batch_bytes', 1 << 20)
    yield c
    c.close()


@pytest.fixture
def default_emu(emu, tmp_path, monkeypatch):
    """The emulated context where the package's CUDA one would be, a private config, and batches of two chunks in
    the Python pipeline (so that a golden file spans several)."""
    saved = dict(_native._default)
    _native._default.clear()
    _native._default[0] = emu
    M.CONFIG_PATH = tmp_path / '.mtscomp'
    monkeypatch.setattr(core, 'GPU_BATCH_CHUNKS', 2)
    yield emu
    _native._default.clear()
    _native._default.update(saved)


def _data(dt, nc, seed, ns=int(ROWS[-1])):
    rng = np.random.default_rng(seed)
    walk = np.cumsum(rng.integers(-40, 41, (ns, nc)), axis=0)
    if np.dtype(dt).kind == 'f':
        return (walk / 7.3 + 20000.).astype(dt)
    return walk.astype(dt)


def _copy_golden(name, dst):
    for ext in ('.cbin', '.ch'):
        shutil.copy(GOLDEN / (name + ext), dst / (name + ext))
    return dst / (name + '.cbin'), dst / (name + '.ch')


def _compress_raw(tmp_path, name, **kw):
    m, meta, raw, _, _ = golden(name)
    path = tmp_path / (name + '.bin')
    raw.tofile(path)
    out, outmeta = tmp_path / (name + '_c.cbin'), tmp_path / (name + '_c.ch')
    M.compress(path, out, outmeta, sample_rate=m['sample_rate'], n_channels=raw.shape[1], dtype=raw.dtype, quiet=True,
               **m['kwargs'], **kw)
    return out.read_bytes(), json.loads(outmeta.read_text())


@pytest.mark.parametrize('write_index', [True, False], ids=['indexed', 'plain'])
@pytest.mark.parametrize('name', INT_GOLDENS)
def test_integer_golden_equals_compress_of_raw(tmp_path, default_emu, name, write_index):
    src, src_ch = _copy_golden(name, tmp_path)
    out, outmeta = tmp_path / 'r.cbin', tmp_path / 'r.ch'
    ratio = M.recompress(src, src_ch, out, outmeta, write_index=write_index, quiet=True)
    want, want_meta = _compress_raw(tmp_path, name, write_index=write_index)
    assert out.read_bytes() == want
    meta = json.loads(outmeta.read_text())
    assert sorted(meta) == sorted(want_meta)
    for k in want_meta:
        assert meta[k] == want_meta[k], k
    assert ratio == len(want) / golden(name)[2].nbytes
    assert outmeta.read_text() == json.dumps(meta, indent=2, sort_keys=True)


@pytest.mark.parametrize('name', FLOAT_GOLDENS)
def test_float_golden_inflates_to_the_same_bytes(tmp_path, default_emu, name):
    m, meta, raw, cbin, _ = golden(name)
    src, src_ch = _copy_golden(name, tmp_path)
    out, outmeta = tmp_path / 'r.cbin', tmp_path / 'r.ch'
    M.recompress(src, src_ch, out, outmeta, quiet=True)
    new = json.loads(outmeta.read_text())
    assert inflated(out.read_bytes(), new['chunk_offsets']) == inflated(cbin, meta['chunk_offsets'])
    dec = np.fromfile(GOLDEN / (name + '.dec'), dtype=raw.dtype).reshape(raw.shape)
    r = M.decompress(out, outmeta)
    got = r[:]
    r.close()
    uint = np.dtype('u%d' % raw.dtype.itemsize)
    assert np.array_equal(got.view(uint), dec.view(uint))


@pytest.mark.parametrize('dt', [np.int16, np.float32], ids=['int16', 'float32'])
def test_fixed_points_and_the_other_direction(tmp_path, default_emu, dt):
    nc, sr = 13, 1000.
    data = _data(dt, nc, 4, 5300)
    path = tmp_path / 'd.bin'
    data.tofile(path)
    files = {}
    for wi in (True, False):
        files[wi] = (tmp_path / ('w%d.cbin' % wi), tmp_path / ('w%d.ch' % wi))
        M.compress(path, *files[wi], sample_rate=sr, n_channels=nc, dtype=dt, write_index=wi, quiet=True)
    indexed, plain = (files[w][0].read_bytes() for w in (True, False))
    assert indexed != plain
    M.recompress(*files[True], tmp_path / 'a.cbin', write_index=True, quiet=True)
    assert (tmp_path / 'a.cbin').read_bytes() == indexed
    M.recompress(*files[True], tmp_path / 'b.cbin', write_index=False, quiet=True)
    assert (tmp_path / 'b.cbin').read_bytes() == plain
    M.recompress(tmp_path / 'b.cbin', tmp_path / 'b.ch', tmp_path / 'c.cbin', quiet=True)
    assert (tmp_path / 'c.cbin').read_bytes() == indexed
    assert json.loads((tmp_path / 'c.ch').read_text()) == json.loads(files[True][1].read_text())


@pytest.mark.parametrize('dt', DTYPES, ids=lambda d: np.dtype(d).name)
@pytest.mark.parametrize('order', ['F', 'C'])
@pytest.mark.parametrize('diff', [(False, False), (True, False), (False, True), (True, True)],
                         ids=['nodiff', 'time', 'spatial', 'time+spatial'])
def test_cabi_matrix(emu, dt, order, diff):
    nc = 9 if order == 'F' else 5
    flags = _native.flags_of(diff[0], diff[1], order)
    data = _data(dt, nc, 5)
    comp, offs = reference_streams(data, ROWS, flags)
    flags = _native._fl(flags, dt)
    isz = np.dtype(dt).itemsize
    want = emu.compress(data, ROWS, flags)
    for comp_dev, dst_dev in PLACEMENTS:
        out, new_offs, st = recompress_at(emu, comp, offs, ROWS, nc, isz, flags, comp_dev, dst_dev)
        assert not st.any()
        if np.dtype(dt).kind == 'f':
            assert inflated(out, new_offs) == inflated(comp, offs)
        else:
            assert out == want[0].tobytes() and new_offs.tolist() == want[1].tolist(), (comp_dev, dst_dev)
        t = emu.timings()
        assert t[2] > 0 and t[4] > 0 and t[5] > 0 and t[7] > 0 and emu.launches() > 0


def test_several_sub_batches(emu):
    """Enough raw bytes for three 1 MB sub-batches, with a write_index change between calls."""
    nc, n = 40, 150
    rows = np.arange(n + 1, dtype=np.int64) * 200
    rows[-1] -= 13
    flags = _native.flags_of(True, False, 'F')
    data = _data(np.int16, nc, 12, int(rows[-1]))
    comp, offs = reference_streams(data, rows, flags)
    for wi in (1, 0):
        emu.set_param('write_index', wi)
        try:
            want, want_offs = emu.compress(data, rows, flags)
            for comp_dev, dst_dev in ((0, 0), (1, 1)):
                out, new_offs, st = recompress_at(emu, comp, offs, rows, nc, 2, flags, comp_dev, dst_dev)
                assert not st.any() and out == want.tobytes() and new_offs.tolist() == want_offs.tolist()
        finally:
            emu.set_param('write_index', 1)


def test_corrupt_chunk_status(emu):
    nc, flags = 11, _native.flags_of(True, False, 'F')
    data = _data(np.int16, nc, 7)
    comp, offs = reference_streams(data, ROWS, flags)
    blob = bytearray(comp)
    for i in (3, 5):
        blob[int(offs[i]) + 20] ^= 0x5a
    for comp_dev, dst_dev in ((0, 0), (1, 1)):
        _, _, st = recompress_at(emu, bytes(blob), offs, ROWS, nc, 2, flags, comp_dev, dst_dev)
        assert np.flatnonzero(st).tolist() == [3, 5]


def test_forged_index_is_recompressed_from_the_plain_stream(emu):
    nc, flags = 19, _native.flags_of(True, False, 'F')
    data = _data(np.int16, nc, 8)
    comp, plain_offs = reference_streams(data, ROWS, flags)
    parts = [comp[plain_offs[i]:plain_offs[i + 1]] for i in range(len(ROWS) - 1)]
    parts[3] = misleading_chunk(emu, data[ROWS[3]:ROWS[4]], flags)
    blob = b''.join(parts)
    offs = np.concatenate(([0], np.cumsum([len(p) for p in parts]))).astype(np.int64)
    want, want_offs = emu.compress(data, ROWS, flags)
    recompress_at(emu, comp, plain_offs, ROWS, nc, 2, flags, 0, 0)
    plain_launches = emu.launches()
    for comp_dev, dst_dev in PLACEMENTS:
        out, new_offs, st = recompress_at(emu, blob, offs, ROWS, nc, 2, flags, comp_dev, dst_dev)
        assert not st.any()
        assert out == want.tobytes() and new_offs.tolist() == want_offs.tolist()
        assert emu.launches() > plain_launches           # the misled chunk was inflated a second time


def test_recompress_corrupt_file_leaves_nothing(tmp_path, default_emu):
    src, src_ch = _copy_golden('ap_small', tmp_path)
    o = json.loads(src_ch.read_text())['chunk_offsets']
    blob = bytearray(src.read_bytes())
    blob[o[1] + 100] ^= 0xff
    src.write_bytes(bytes(blob))
    out, outmeta = tmp_path / 'r.cbin', tmp_path / 'r.ch'
    with raises(IOError, match=r'Compressed chunk #1 is corrupted\.'):
        M.recompress(src, src_ch, out, outmeta, quiet=True)
    assert not out.exists() and not outmeta.exists()


def test_metadata_is_carried_over(tmp_path, default_emu):
    src, src_ch = _copy_golden('ap_small', tmp_path)
    meta = json.loads(src_ch.read_text())
    meta['lab_notes'] = {'probe': 'np1.0', 'ok': [1, 2]}
    src_ch.write_text(json.dumps(meta, indent=2, sort_keys=True))
    out, outmeta = tmp_path / 'r.cbin', tmp_path / 'r.ch'
    M.recompress(src, src_ch, out, outmeta, quiet=True)
    new = json.loads(outmeta.read_text())
    assert new['lab_notes'] == meta['lab_notes']
    assert new['sha1_uncompressed'] == meta['sha1_uncompressed']
    assert new['sha1_compressed'] == hashlib.sha1(out.read_bytes()).hexdigest() != meta['sha1_compressed']
    assert {k for k in new if new[k] != meta[k]} == {'chunk_offsets', 'sha1_compressed'}
    pr = PortReader(out, outmeta)
    try:
        assert hashlib.sha1(np.ascontiguousarray(pr[:]).tobytes()).hexdigest() == golden('ap_small')[0]['sha1_decoded']
        assert np.array_equal(pr[123:456], golden('ap_small')[2][123:456])
    finally:
        pr.close()

    # a chopped source keeps `chopped` and its null sha1_uncompressed
    r = M.decompress(src, src_ch)
    r.chop(2, tmp_path / 'chop.cbin')
    r.close()
    M.recompress(tmp_path / 'chop.cbin', tmp_path / 'chop.ch', tmp_path / 'rc.cbin', quiet=True)
    new = json.loads((tmp_path / 'rc.ch').read_text())
    assert new['chopped'] is True and new['sha1_uncompressed'] is None
    assert new['sha1_compressed'] == hashlib.sha1((tmp_path / 'rc.cbin').read_bytes()).hexdigest()
    pr = PortReader(tmp_path / 'rc.cbin', tmp_path / 'rc.ch')
    try:
        assert np.array_equal(pr[:], golden('ap_small')[2][:new['chunk_bounds'][-1]])
    finally:
        pr.close()


def test_mtsrecomp(tmp_path, default_emu):
    src, src_ch = _copy_golden('lfp_spatial', tmp_path)
    before = src.read_bytes(), src_ch.read_text()
    out = tmp_path / 'r.cbin'
    M.mtsrecomp([str(src), '-o', str(out)])
    want, want_meta = _compress_raw(tmp_path, 'lfp_spatial')
    assert out.read_bytes() == want and json.loads((tmp_path / 'r.ch').read_text()) == want_meta
    M.mtsrecomp([str(src), str(src_ch), '-o', str(tmp_path / 'p.cbin'), '--outmeta', str(tmp_path / 'p.json'),
                 '--no-index', '-nc'])
    assert (tmp_path / 'p.cbin').read_bytes() == _compress_raw(tmp_path, 'lfp_spatial', write_index=False)[0]
    assert json.loads((tmp_path / 'p.json').read_text())['chunk_offsets'] != want_meta['chunk_offsets']
    with raises(ValueError, match='in place'):
        M.mtsrecomp([str(src), '-o', str(src), '-f'])
    with raises(ValueError, match='already exists, use --overwrite'):
        M.mtsrecomp([str(src), '-o', str(out)])
    assert (src.read_bytes(), src_ch.read_text()) == before
    out.write_bytes(b'old')
    M.mtsrecomp([str(src), '-o', str(out), '-f'])
    assert out.read_bytes() == want


def test_bad_arguments(emu):
    nc, flags = 4, _native.flags_of(True, False, 'F')
    data = _data(np.int16, nc, 9)[:100]
    comp, offs = reference_streams(data, [0, 100], flags)
    cap = emu.compress_bound(100, nc, 2, flags)
    dst = np.zeros(cap, np.uint8)
    with raises(_native.NativeError, match='dst_capacity'):
        emu.recompress_ptr(np.frombuffer(comp, np.uint8).ctypes.data, 0, offs, [0, 100], nc, 2, flags,
                           dst.ctypes.data, 0, cap - 1)
    with raises(_native.NativeError, match='bad compressed length'):
        emu.recompress_ptr(np.frombuffer(comp, np.uint8).ctypes.data, 0, [0, 0], [0, 100], nc, 2, flags,
                           dst.ctypes.data, 0, cap)
    assert zlib.decompress(comp) == zlib.decompress(bytes(emu.recompress(comp, offs, [0, 100], nc, np.int16, flags)[0]))
