"""GPU: mtsb_recompress_chunks at AP scale with every placement of the compressed input and the output, recompress()
on a reference-written file, and the misled-index and corrupt-chunk cases on the device."""
import json

import numpy as np
import pytest

import mtscomp_b200 as M
from mtscomp_b200 import _native, synth
from oracle import codec as ora
from recompress_cases import PLACEMENTS, inflated, misleading_chunk, recompress_at, reference_streams

pytestmark = pytest.mark.gpu
NS, NC, N_CHUNKS, DISTINCT = 30000, 385, 20, 4


@pytest.fixture(scope='module')
def small_batches():
    """A context of its own whose host-buffer sub-batches hold one AP chunk, so that a call has several."""
    c = _native.Codec(0)
    c.set_param('host_batch_bytes', 1 << 20)
    c.set_param('par_batch_bytes', 64 << 20)
    yield c
    c.close()


@pytest.fixture(scope='module', params=[np.int16, np.float32], ids=['int16', 'float32'])
def ap_source(request):
    """N_CHUNKS AP chunks tiled from DISTINCT synth chunks, and their reference-layout streams (zlib level 6)."""
    dt = request.param
    distinct = [synth.ap_chunk(NS, NC, seed=80 + i) for i in range(DISTINCT)]
    if dt == np.float32:
        distinct = [(d.astype(np.float64) / 7.3 + 20000.).astype(np.float32) for d in distinct]
    flags = _native.TIME_DIFF
    streams = [ora.encode_chunk(d) for d in distinct]
    data = np.concatenate([distinct[i % DISTINCT] for i in range(N_CHUNKS)])
    parts = [streams[i % DISTINCT] for i in range(N_CHUNKS)]
    comp = b''.join(parts)
    offs = np.concatenate(([0], np.cumsum([len(p) for p in parts]))).astype(np.int64)
    rows = np.arange(N_CHUNKS + 1, dtype=np.int64) * NS
    return data, rows, comp, offs, _native._fl(flags, dt)


@pytest.mark.parametrize('ctx', ['small_batches', 'codec'])
def test_ap_scale_every_placement(request, ap_source, ctx):
    c = request.getfixturevalue(ctx)
    data, rows, comp, offs, flags = ap_source
    isz = data.dtype.itemsize
    if data.dtype.kind != 'f':
        want, want_offs = c.compress(data, rows, flags)
    src_inflated = inflated(comp, offs[:DISTINCT + 1])
    for comp_dev, dst_dev in PLACEMENTS:
        out, new_offs, st = recompress_at(c, comp, offs, rows, NC, isz, flags, comp_dev, dst_dev)
        assert not st.any()
        t = c.timings()
        assert t[2] > 0 and t[4] > 0 and t[5] > 0
        if data.dtype.kind == 'f':
            assert inflated(out, new_offs[:DISTINCT + 1]) == src_inflated
            assert all(out[new_offs[i]:new_offs[i + 1]] == out[new_offs[i % DISTINCT]:new_offs[i % DISTINCT + 1]]
                       for i in range(N_CHUNKS))
            uint = np.uint32
            a, st1 = c.decompress(out, new_offs, rows, NC, data.dtype, flags)
            b, st2 = c.decompress(comp, offs, rows, NC, data.dtype, flags)
            assert not st1.any() and not st2.any() and np.array_equal(a.view(uint), b.view(uint))
        else:
            assert out == want.tobytes() and new_offs.tolist() == want_offs.tolist(), (comp_dev, dst_dev)


def test_recompress_reference_written_file(tmp_path, codec):
    M.CONFIG_PATH = tmp_path / '.mtscomp'
    sr = float(NS)
    data = np.concatenate([synth.ap_chunk(NS, NC, seed=90 + i) for i in range(3)])[:-1234]
    src, src_ch = tmp_path / 'ref.cbin', tmp_path / 'ref.ch'
    ora.write_file(data, sr, src, src_ch)
    out = tmp_path / 'gpu.cbin'
    ratio = M.recompress(src, src_ch, out, quiet=True)             # the check after writing runs by default
    assert 0.2 < ratio < 0.6
    r_src, r_new = M.decompress(src, src_ch), M.decompress(out, tmp_path / 'gpu.ch')
    try:
        for sl in (slice(None), slice(12345, 45678), slice(NS - 5, NS + 5), slice(-100, None)):
            assert np.array_equal(r_new[sl], r_src[sl])
        assert np.array_equal(r_new[:], data)
        # the new chunks take the indexed path: no block search
        for r, searched in ((r_new, False), (r_src, True)):
            block = np.empty_like(data)
            meta = r.cmeta
            blob = open(r.cdata.name, 'rb').read()
            st = codec.decompress_ptr(np.frombuffer(blob, np.uint8).ctypes.data, 0, meta.chunk_offsets,
                                      meta.chunk_bounds, NC, 2, _native.TIME_DIFF, block.ctypes.data, 0)
            assert not st.any() and np.array_equal(block, data)
            assert (codec.get_param('par_survivors') != 0) == searched
    finally:
        r_src.close()
        r_new.close()
    meta, want = json.loads((tmp_path / 'gpu.ch').read_text()), json.loads(src_ch.read_text())
    assert {k for k in want if meta[k] != want[k]} == {'chunk_offsets', 'sha1_compressed'}


def test_misled_index_and_corrupt_chunk_on_the_device(codec):
    rows = np.arange(6, dtype=np.int64) * 4000
    data = synth.ap_chunk(int(rows[-1]), 64, seed=5)
    flags = _native.TIME_DIFF
    comp, offs = reference_streams(data, rows, flags)
    parts = [comp[offs[i]:offs[i + 1]] for i in range(5)]
    parts[2] = misleading_chunk(codec, data[rows[2]:rows[3]], flags)
    blob = b''.join(parts)
    moffs = np.concatenate(([0], np.cumsum([len(p) for p in parts]))).astype(np.int64)
    want, want_offs = codec.compress(data, rows, flags)
    out, new_offs, st = recompress_at(codec, blob, moffs, rows, 64, 2, flags, 1, 1)
    assert not st.any() and out == want.tobytes() and new_offs.tolist() == want_offs.tolist()

    bad = bytearray(comp)
    bad[int(offs[3]) + 50] ^= 0x5a
    _, _, st = recompress_at(codec, bytes(bad), offs, rows, 64, 2, flags, 1, 1)
    assert np.flatnonzero(st).tolist() == [3]
