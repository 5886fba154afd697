"""GPU: mtsb_verify_chunks at AP scale with every placement of the compressed bytes and the reference rows, on
reference-written goldens, and the checks after Writer.write, Reader.tofile and a two-rank write_sharded."""
import json
import os
import socket

import numpy as np
import pytest
from pytest import raises

import mtscomp_b200 as M
from mtscomp_b200 import _native, synth
from mtscomp_b200.config import CHECK_ATOL
from mtscomp_b200.core import CHECK_RTOL

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(__file__), 'golden')
NS, NC = 30000, 385


@pytest.fixture(scope='module')
def small_batches():
    """A context of its own whose host-buffer sub-batches hold a few AP chunks, so that a call has several."""
    c = _native.Codec(0)
    c.set_param('host_batch_bytes', 1 << 20)
    c.set_param('par_batch_bytes', 64 << 20)
    yield c
    c.close()


def _expected(dec, ref, rows):
    bad = ~np.isclose(dec, ref, rtol=CHECK_RTOL, atol=CHECK_ATOL) if dec.dtype.kind == 'f' else dec != ref
    m = [int(bad[rows[i]:rows[i + 1]].sum()) for i in range(len(rows) - 1)]
    f = [int(np.flatnonzero(bad[rows[i]:rows[i + 1]].ravel())[0]) if m[i] else -1 for i in range(len(rows) - 1)]
    return m, f


def _to_device(codec, arr, shift=0):
    """Device copy of `arr` starting `shift` bytes into its allocation -> (allocation, pointer)."""
    p = codec.device_alloc(arr.nbytes + shift + 256)
    codec.memcpy(p + shift, arr.ctypes.data, arr.nbytes, 1)
    return p, p + shift


@pytest.mark.parametrize('dt', [np.int16, np.float32], ids=['int16', 'float32'])
@pytest.mark.parametrize('write_index', [1, 0], ids=['indexed', 'plain'])
def test_verify_ap_scale_every_placement(small_batches, dt, write_index):
    c = small_batches
    n_chunks = 20
    rows = np.arange(n_chunks + 1, dtype=np.int64) * NS
    rows[-1] -= 777                                                   # a ragged last chunk
    data = np.concatenate([synth.ap_chunk(NS, NC, seed=60 + i) for i in range(n_chunks)])[:rows[-1]]
    if dt == np.float32:
        data = (data.astype(np.float64) / 7.3 + 20000.).astype(np.float32)
    flags = _native._fl(_native.TIME_DIFF, data.dtype)
    c.set_param('write_index', write_index)
    try:
        comp, offs = c.compress(data, rows, flags)
    finally:
        c.set_param('write_index', 1)
    dec, st = c.decompress(comp, offs, rows, NC, dt, flags)
    assert not st.any()
    ref = dec.copy()
    for r, ch in ((rows[3], 0), (rows[4] - 1, NC - 1), (rows[11], 200), (rows[-1] - 1, NC - 1), (rows[15] + 12345, 1)):
        ref[r, ch] += np.array(3, dt)
    want = _expected(dec, ref, rows)
    assert sum(want[0]) == 5
    isz = data.dtype.itemsize
    allocs = []
    try:
        a, d_comp = _to_device(c, comp)
        allocs.append(a)
        a, d_ref = _to_device(c, ref)
        allocs.append(a)
        a, d_ref_odd = _to_device(c, ref, isz)                        # an odd element offset: phases of the two buffers differ
        allocs.append(a)
        for comp_ptr, comp_dev in ((comp.ctypes.data, 0), (d_comp, 1)):
            for ref_ptr, ref_dev in ((ref.ctypes.data, 0), (d_ref, 1), (d_ref_odd, 1)):
                st, m, f = c.verify_ptr(comp_ptr, comp_dev, offs, rows, NC, isz, flags, ref_ptr, ref_dev, CHECK_RTOL,
                                        CHECK_ATOL)
                assert not st.any()
                assert (m.tolist(), f.tolist()) == want, (comp_dev, ref_dev, ref_ptr == d_ref_odd)
                assert c.timings()[6] > 0
    finally:
        for a in allocs:
            c.device_free(a)


def _golden(name):
    meta = json.load(open(os.path.join(GOLDEN, name + '.ch')))
    dt = np.dtype(meta['dtype'])
    ref = np.fromfile(os.path.join(GOLDEN, name + '.bin'), dtype=dt).reshape(-1, meta['n_channels'])
    comp = open(os.path.join(GOLDEN, name + '.cbin'), 'rb').read()
    flags = _native.flags_of(meta['do_time_diff'], meta['do_spatial_diff'], meta['chunk_order'])
    return meta, ref, comp, flags


@pytest.mark.parametrize('name', ['float32_time', 'float64_spatial_c', 'float32_wild'])
def test_verify_reference_goldens(codec, name):
    meta, ref, comp, flags = _golden(name)
    rows = meta['chunk_bounds']
    st, m, f = codec.verify(comp, meta['chunk_offsets'], rows, ref, flags, CHECK_RTOL, CHECK_ATOL)
    assert not st.any()
    dec = np.fromfile(os.path.join(GOLDEN, name + '.dec'), dtype=ref.dtype).reshape(ref.shape)
    assert (m.tolist(), f.tolist()) == _expected(dec, ref, rows)
    if name == 'float32_wild':
        # the file the reference's own check refuses: np.isclose(dec, bin, atol=1e-16) fails 6363 times
        assert int(m.sum()) == 6363 and divmod(int(f[0]), meta['n_channels']) == (0, 5)
        r = M.decompress(os.path.join(GOLDEN, name + '.cbin'), os.path.join(GOLDEN, name + '.ch'))
        with raises(AssertionError, match=r'chunk #0 .*row 0 \(sample 0\), channel 5'):
            M.core._verify_range(r, ref, 0, r.n_chunks)
        r.close()
    else:
        assert not m.any()


def test_default_checks_of_writer_and_reader(tmp_path, codec):
    M.CONFIG_PATH = tmp_path / '.mtscomp'
    data = np.concatenate([synth.ap_chunk(NS, NC, seed=80 + i) for i in range(12)])
    path = tmp_path / 'ap.bin'
    data.tofile(path)
    M.compress(path, tmp_path / 'ap.cbin', tmp_path / 'ap.ch', sample_rate=30000., n_channels=NC, dtype=np.int16,
               quiet=True)
    M.decompress(tmp_path / 'ap.cbin', tmp_path / 'ap.ch', out=tmp_path / 'back.bin', quiet=True).close()
    assert (tmp_path / 'back.bin').read_bytes() == path.read_bytes()

    def corrupt(writer):                                      # a source row changes between the write and the check
        with open(path, 'r+b') as f:
            f.seek((7 * NS + 4321) * NC * 2 + 2 * 17)
            f.write(b'\x01\x7f')
    w = M.Writer(before_check=corrupt, quiet=True)
    w.open(path, sample_rate=30000., n_channels=NC, dtype=np.int16)
    with raises(RuntimeError, match='CRITICAL ERROR'):
        w.write(tmp_path / 'ap2.cbin', tmp_path / 'ap2.ch')
    w.close()


NCHUNK = 7


def _worker(rank, world, port, tmp, corrupt):
    import torch.distributed as dist
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    dist.init_process_group('gloo', rank=rank, world_size=world)
    import mtscomp_b200 as M
    from mtscomp_b200 import _native, sharding
    M.CONFIG_PATH = os.path.join(tmp, '.mtscomp')
    dev = rank % max(_native.load_library().mtsb_device_count(), 1)
    data_path = os.path.join(tmp, 'data.bin')

    def before_check(writer):
        if corrupt and rank == 1:                           # a row of chunk 5, inside rank 1's range [4, 7)
            with open(data_path, 'r+b') as f:
                f.seek((5 * 3000 + 10) * NC * 2)
                f.write(b'\x55\x55')
    try:
        sharding.write_sharded(data_path, os.path.join(tmp, 'sharded.cbin'), os.path.join(tmp, 'sharded.ch'), rank,
                               world, sample_rate=3000., n_channels=NC, dtype=np.int16, device=dev,
                               check_after_compress=True, before_check=before_check)
        verdict = 'ok'
    except Exception as e:
        verdict = '%s: %s' % (type(e).__name__, e)
    with open(os.path.join(tmp, 'rank%d.txt' % rank), 'w') as f:
        f.write(verdict)
    dist.destroy_process_group()


@pytest.mark.parametrize('corrupt', [False, True], ids=['clean', 'rank1_corrupt'])
def test_write_sharded_checks_every_rank(tmp_path, codec, corrupt):
    import torch.multiprocessing as mp
    data = np.concatenate([synth.ap_chunk(3000, NC, seed=90 + i) for i in range(NCHUNK)])[:3000 * NCHUNK - 1234]
    data.tofile(tmp_path / 'data.bin')
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    port = s.getsockname()[1]
    s.close()
    mp.spawn(_worker, args=(2, port, str(tmp_path), corrupt), nprocs=2, join=True)
    verdicts = [(tmp_path / ('rank%d.txt' % r)).read_text() for r in (0, 1)]
    if not corrupt:
        assert verdicts == ['ok', 'ok']
        r = M.decompress(tmp_path / 'sharded.cbin', tmp_path / 'sharded.ch')
        assert np.array_equal(r[:], data)
        r.close()
    else:
        for v in verdicts:
            assert v.startswith('RuntimeError: CRITICAL ERROR') and 'chunk #5' in v, v
