"""CPU: the batch pipeline of the whole-file operations (Writer.write, Reader.tofile, check, recompress) through the
host emulation of the kernels.  The output must not depend on how many chunks go to the GPU per batch, and a failure
in any step of a batch in the middle, with the batches around it in flight, must reach the caller as the operation's
own error, with no pipeline thread left and the staging lock free for the next operation."""
import hashlib
import json
import threading

import numpy as np
import pytest
from pytest import raises

import mtscomp_b200 as M
from mtscomp_b200 import _native, core

SR, NC, NS = 1000., 13, 7500           # 8 chunks of one second, the last one half as long


@pytest.fixture(scope='module')
def emu():
    from mtscomp_b200 import build
    c = _native.Codec(0, lib=_native.load_library(build.build_emulation()))
    yield c
    c.close()


@pytest.fixture
def default_emu(emu, tmp_path, monkeypatch):
    """The emulated context where the package's CUDA one would be, and a private config."""
    saved = dict(_native._default)
    _native._default.clear()
    _native._default[0] = emu
    monkeypatch.setattr(M, 'CONFIG_PATH', tmp_path / '.mtscomp')
    yield emu
    _native._default.clear()
    _native._default.update(saved)


def _data(dt, seed=3):
    walk = np.cumsum(np.random.default_rng(seed).integers(-40, 41, (NS, NC)), axis=0)
    return (walk / 7.3 + 20000.).astype(dt) if np.dtype(dt).kind == 'f' else walk.astype(dt)


def _compress(tmp_path, data, name='d', **kw):
    path = tmp_path / (name + '.bin')
    data.tofile(path)
    out, outmeta = tmp_path / (name + '.cbin'), tmp_path / (name + '.ch')
    w = M.Writer(quiet=True, check_after_compress=False, **kw)
    w.open(path, sample_rate=SR, n_channels=NC, dtype=data.dtype)
    w.write(out, outmeta)
    w.close()
    return out, outmeta


def _pipeline_threads():
    return [t.name for t in threading.enumerate() if t.name.startswith(('mtsb-stage', 'mtsb-finish'))]


def _lock_is_free(codec):
    got = []

    def take():
        ok = codec.stage_lock.acquire(blocking=False)
        got.append(ok)
        if ok:
            codec.stage_lock.release()
    t = threading.Thread(target=take)
    t.start()
    t.join()
    return got == [True]


@pytest.mark.parametrize('dt', [np.int16, np.float32], ids=['int16', 'float32'])
def test_batch_size_does_not_change_results(tmp_path, default_emu, monkeypatch, dt):
    data = _data(dt)
    bad = data.copy()
    bad[6000 + 17, 5] += 100                     # chunks 6 and 7: the last batch at every batch size below
    bad[7000 + 3, 2] += 100
    results = []
    for n in (1, 2, 3, 64):
        monkeypatch.setattr(core, 'GPU_BATCH_CHUNKS', n)
        d = tmp_path / str(n)
        d.mkdir()
        out, outmeta = _compress(d, data)
        meta = json.loads(outmeta.read_text())
        assert meta['sha1_compressed'] == hashlib.sha1(out.read_bytes()).hexdigest()
        assert meta['sha1_uncompressed'] == hashlib.sha1((d / 'd.bin').read_bytes()).hexdigest()
        assert len(meta['chunk_bounds']) == 9
        r = M.decompress(out, outmeta, out=d / 'dec.bin')
        r.close()
        assert (d / 'dec.bin').read_bytes() == (d / 'd.bin').read_bytes()
        M.check(data, out, outmeta)
        with raises(AssertionError, match=r'^chunk #6 does not match the data in 1 element\(s\); the first is row 17 '):
            M.check(bad, out, outmeta)
        M.recompress(out, outmeta, d / 'r.cbin', write_index=False, quiet=True)
        results.append((out.read_bytes(), outmeta.read_text(), (d / 'r.cbin').read_bytes(), (d / 'r.ch').read_text()))
    assert all(res == results[-1] for res in results)
    assert not _pipeline_threads()


def _tofile(cbin, ch, dst):
    r = M.Reader(quiet=True)
    r.open(cbin, ch)
    try:
        r.tofile(dst, overwrite=True)
    finally:
        r.close()


def _run_op(op, data, cbin, ch, tmp_path):
    if op == 'tofile':
        _tofile(cbin, ch, tmp_path / 'dec.bin')
    elif op == 'check':
        M.check(data, cbin, ch)
    else:
        M.recompress(cbin, ch, tmp_path / 'r.cbin', quiet=True)


def _after_failure(codec, op, data, good, tmp_path):
    assert not _pipeline_threads()
    assert _lock_is_free(codec)
    if op == 'recompress':
        assert not (tmp_path / 'r.cbin').exists() and not (tmp_path / 'r.ch').exists()
    _tofile(*good, tmp_path / 'again.bin')
    assert (tmp_path / 'again.bin').read_bytes() == data.tobytes()


@pytest.mark.parametrize('op', ['tofile', 'check', 'recompress'])
@pytest.mark.parametrize('step', ['stage', 'run'])
def test_failure_in_a_middle_batch(tmp_path, default_emu, monkeypatch, op, step):
    """Batch 2 of 8 fails in its stage step (the .cbin ends inside it) or in its run step (a corrupt chunk)."""
    monkeypatch.setattr(core, 'GPU_BATCH_CHUNKS', 1)
    data = _data(np.int16)
    good = _compress(tmp_path, data, 'good')
    cbin, ch = _compress(tmp_path, data)
    o = json.loads(ch.read_text())['chunk_offsets']
    blob = bytearray(cbin.read_bytes())
    if step == 'stage':
        del blob[o[2] + 10:]
        err, msg = AssertionError, 'unexpected end of the compressed file'
    else:
        blob[o[2] + 40] ^= 0x5a
        err, msg = IOError, r'Compressed chunk #2 is corrupted\.'
    cbin.write_bytes(bytes(blob))
    with raises(err, match=msg):
        _run_op(op, data, cbin, ch, tmp_path)
    _after_failure(default_emu, op, data, good, tmp_path)


class _Boom(Exception):
    pass


class _FailsOnSecondUpdate:
    def __init__(self):
        self.calls = 0

    def update(self, _):
        self.calls += 1
        if self.calls == 2:
            raise _Boom('second update')


def test_failure_in_a_finisher(tmp_path, default_emu, monkeypatch):
    """The raw SHA-1 of the Writer's batch 1 fails on its finisher lane while later batches are in flight."""
    monkeypatch.setattr(core, 'GPU_BATCH_CHUNKS', 1)
    data = _data(np.int16)
    good = _compress(tmp_path, data, 'good')
    (tmp_path / 'd.bin').write_bytes(data.tobytes())
    w = M.Writer(quiet=True, check_after_compress=False)
    w.open(tmp_path / 'd.bin', sample_rate=SR, n_channels=NC, dtype=data.dtype)
    w.sha1_uncompressed = _FailsOnSecondUpdate()
    with raises(_Boom, match='second update'):
        w.write(tmp_path / 'd.cbin', tmp_path / 'd.ch')
    w.close()
    assert not (tmp_path / 'd.ch').exists()
    _after_failure(default_emu, 'write', data, good, tmp_path)
    _compress(tmp_path, data)
    assert (tmp_path / 'd.cbin').read_bytes() == good[0].read_bytes()
