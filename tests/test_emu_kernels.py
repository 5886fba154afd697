"""CPU: kernel LOGIC through the host emulation build (csrc/emu/cuda_emu.h) against the oracle and the golden files.

This is a development aid that lets the CPU-only container exercise the exact kernel sources; it is not a product
path (mtscomp_b200/_native.py never loads the emulation library) and it says nothing about the GPU memory model —
the `-m gpu` tests do that on a B200."""
import json
import zlib

import numpy as np
import pytest

from conftest import GOLDEN
from oracle import codec as ora


@pytest.fixture(scope='module')
def emu():
    from mtscomp_b200 import _native, build
    return _native.Codec(0, lib=_native.load_library(build.build_emulation()))


def _flags(ch):
    from mtscomp_b200 import _native
    return _native.flags_of(ch['do_time_diff'], ch['do_spatial_diff'], ch['chunk_order'])


@pytest.mark.parametrize('name', ['lfp_spatial', 'order_c', 'fullrange', 'wrap_edges', 'tiny_1x1', 'tiny_chunks',
                                  'zeros_runs', 'spatial_only', 'nodiff', 'one_channel'])
def test_emulated_kernels_on_golden(emu, name):
    m = json.loads((GOLDEN / 'manifest.json').read_text())['cases'][name]
    ch = json.loads((GOLDEN / (name + '.ch')).read_text())
    raw = np.fromfile(GOLDEN / (name + '.bin'), dtype=m['dtype']).reshape(m['shape'])
    cbin = (GOLDEN / (name + '.cbin')).read_bytes()
    fl = _flags(ch)
    b, o = ch['chunk_bounds'], ch['chunk_offsets']
    # K1 vs the bytes the reference handed to zlib
    assert emu.delta_transform(raw[b[0]:b[1]], fl).tobytes() == (GOLDEN / (name + '.tr')).read_bytes()
    # decoder on the reference-written file
    out, st = emu.decompress(cbin, o, b, ch['n_channels'], ch['dtype'], fl)
    assert not st.any() and np.array_equal(out, raw)
    # encoder: zlib must accept every chunk and return the reference's transform bytes
    comp, offs = emu.compress(raw, b, fl)
    kw = dict(do_time_diff=ch['do_time_diff'], do_spatial_diff=ch['do_spatial_diff'], chunk_order=ch['chunk_order'])
    for i in range(len(b) - 1):
        assert zlib.decompress(bytes(comp[offs[i]:offs[i + 1]])) == ora.transform_chunk(raw[b[i]:b[i + 1]], **kw)
    out2, st2 = emu.decompress(comp, offs, b, ch['n_channels'], ch['dtype'], fl)
    assert not st2.any() and np.array_equal(out2, raw)


def test_emulated_corruption_is_reported(emu):
    ch = json.loads((GOLDEN / 'nodiff.ch').read_text())
    cbin = bytearray((GOLDEN / 'nodiff.cbin').read_bytes())
    o = ch['chunk_offsets']
    cbin[o[2] - 1] ^= 0x40          # adler32 of chunk 1
    cbin[o[2] + 40] ^= 0x10         # payload of chunk 2
    _, st = emu.decompress(bytes(cbin), o, ch['chunk_bounds'], ch['n_channels'], ch['dtype'], _flags(ch))
    assert st[0] == 0 and st[1] == 9 and st[2] != 0


def test_emulated_host_pipeline_many_sub_batches(emu):
    """Host-buffer path with several double-buffered sub-batches (H2D / kernels / D2H on separate streams)."""
    from mtscomp_b200 import synth, _native
    x = np.concatenate([synth.ap_chunk(ns=1500, nc=96, seed=80 + i) for i in range(3)] * 3)
    rows = np.arange(10) * 1500
    emu.set_param('host_batch_bytes', 1 << 20)
    emu.set_param('batch_bytes', 1 << 20)
    try:
        comp, offs = emu.compress(x, rows, _native.TIME_DIFF)
        for i in range(9):
            assert zlib.decompress(bytes(comp[offs[i]:offs[i + 1]])) == ora.transform_chunk(x[rows[i]:rows[i + 1]])
        out, st = emu.decompress(comp, offs, rows, 96, np.int16, _native.TIME_DIFF)
        assert not st.any() and np.array_equal(out, x)
    finally:
        emu.set_param('host_batch_bytes', 512 << 20)
        emu.set_param('batch_bytes', 2 << 30)


def test_emulated_block_parallel_inflate(emu):
    """Kernel logic of the block-parallel decoder on a reference-style zlib stream (several deflate blocks)."""
    from mtscomp_b200 import synth, _native
    x = synth.ap_chunk(ns=20000, nc=16, seed=33)
    good = ora.encode_chunk(x)
    for wide, cells in ((1, 0), (0, 0), (-1, 1), (-1, -1)):   # both chain-of-tiles shapes, the cells path, automatic
        emu.set_param('par_lz_wide', wide)
        emu.set_param('par_cells', cells)
        out, st = emu.decompress(good, [0, len(good)], [0, 20000], 16, np.int16, _native.TIME_DIFF)
        assert not st.any() and np.array_equal(out, x)
        assert emu.get_param('par_chained') >= 5 and emu.get_param('par_resumed') == 1
    bad = bytearray(good)
    bad[len(bad) // 2] ^= 0x33
    _, st = emu.decompress(bytes(bad), [0, len(bad)], [0, 20000], 16, np.int16, _native.TIME_DIFF)
    assert st[0] != 0


def test_emulated_marker_chains(emu):
    """Cells path of the block-parallel decoder on period-20 KB data: every block is made of references into the block
    before it, so markers have to be chased through several blocks."""
    from mtscomp_b200 import _native
    rng = np.random.default_rng(9)
    pat = rng.integers(-3000, 3000, 10000).astype(np.int16)
    x = np.tile(pat, 500).reshape(-1, 1)
    good = ora.encode_chunk(x)
    assert len(good) >= 65536
    try:
        emu.set_param('par_cells', 1)
        out, st = emu.decompress(good, [0, len(good)], [0, x.shape[0]], 1, np.int16, _native.TIME_DIFF)
        assert st[0] == 0 and np.array_equal(out, x)
        assert emu.get_param('par_resumed') == 1 and emu.get_param('par_chained') >= 3
    finally:
        emu.set_param('par_cells', -1)


def test_emulated_indexed_segments_both_decoders(emu):
    """GPU-written chunk (kernel logic under emulation): the indexed segments through the second-format kernels
    (seg_tokens / seg_resolve), through the block kernels and through the serial warp decoder give the same bytes; a
    segment stored uncompressed stays with the serial decoder."""
    from mtscomp_b200 import _native, synth
    rng = np.random.default_rng(2)
    x = np.concatenate([synth.ap_chunk(ns=4000, nc=48, seed=11),
                        rng.integers(-32768, 32767, (4000, 48)).astype(np.int16)])
    rows = [0, 4000, 8000]
    try:
        emu.set_param('seg_bytes', 65536)
        comp, offs = emu.compress(x, rows, _native.TIME_DIFF)
        outs = []
        for v2, indexed in ((1, 0), (0, 1), (0, 0)):
            emu.set_param('seg_v2', v2)
            emu.set_param('par_indexed', indexed)
            out, st = emu.decompress(comp, offs, rows, 48, np.int16, _native.TIME_DIFF)
            assert not st.any() and np.array_equal(out, x)
            outs.append(emu.get_param('par_resumed'))
        assert outs[0] >= 4 and outs[1] >= 4 and outs[2] == 0
    finally:
        emu.set_param('seg_bytes', 262144)
        emu.set_param('par_indexed', 1)
        emu.set_param('seg_v2', 1)


@pytest.mark.parametrize('name', sorted(json.loads((GOLDEN / 'manifest.json').read_text()).get('float_cases', {})))
def test_emulated_float_golden(emu, name):
    """float32 / float64 (kernel logic under emulation): decode of the reference-written file == the reference
    Reader's output bit for bit; the encoder's streams inflate to the reference's transform bytes."""
    from mtscomp_b200 import _native
    m = json.loads((GOLDEN / 'manifest.json').read_text())['float_cases'][name]
    ch = json.loads((GOLDEN / (name + '.ch')).read_text())
    raw = np.fromfile(GOLDEN / (name + '.bin'), dtype=m['dtype']).reshape(m['shape'])
    dec = np.fromfile(GOLDEN / (name + '.dec'), dtype=m['dtype']).reshape(m['shape'])
    cbin = (GOLDEN / (name + '.cbin')).read_bytes()
    fl = _flags(ch)
    out, st = emu.decompress(cbin, ch['chunk_offsets'], ch['chunk_bounds'], ch['n_channels'], raw.dtype, fl)
    assert not st.any() and out.tobytes() == dec.tobytes()
    comp, offs = emu.compress(raw, ch['chunk_bounds'], fl)
    b = ch['chunk_bounds']
    assert zlib.decompress(bytes(comp[offs[0]:offs[1]])) == (GOLDEN / (name + '.tr')).read_bytes()
    out2, st2 = emu.decompress(comp, offs, b, ch['n_channels'], raw.dtype, fl)
    assert not st2.any() and out2.tobytes() == dec.tobytes()


@pytest.mark.parametrize('nc,dtype', [(1, 'int16'), (31, 'uint8'), (447, 'int16'), (449, 'int16'), (449, 'int64'),
                                      (900, 'int32'), (1800, 'int16'), (2100, 'int16'), (450, 'uint8'),
                                      (190, 'float32'), (94, 'float64'), (1793, 'float32'), (1793, 'float64')])
def test_emulated_tile_kernels_channel_counts(emu, nc, dtype):
    """The channel-major tile kernels give a thread 1, 2 or 4 channels depending on n_channels and fall back to the
    generic kernels beyond that: every regime, ragged chunk lengths, all four difference settings.  Float arrays go
    through both orders: the generic forward kernel stages a tile of 65 rows in shared memory, more than the default
    48 KB from 190 float32 / 94 float64 channels on ('C'), and above 1792 channels in either order."""
    from mtscomp_b200 import _native
    rng = np.random.default_rng(nc)
    is_float = np.dtype(dtype).kind == 'f'
    ns = [70, 33, 5, 129] if not (is_float and nc > 1792) else [9, 1, 4]
    x = np.cumsum(rng.integers(-3, 4, (sum(ns), nc)), axis=0).astype(dtype)
    rows = np.concatenate(([0], np.cumsum(ns)))
    for order in ('F', 'C') if is_float else ('F',):
        for td, sd in ((True, False), (True, True), (False, True), (False, False)):
            fl = _native.flags_of(td, sd, order)
            kw = dict(do_time_diff=td, do_spatial_diff=sd, chunk_order=order)
            for i in range(len(ns)):
                assert emu.delta_transform(x[rows[i]:rows[i + 1]], fl).tobytes() == ora.transform_chunk(x[rows[i]:rows[i + 1]], **kw)
            comp = [ora.encode_chunk(x[rows[i]:rows[i + 1]], **kw) for i in range(len(ns))]
            offs = np.concatenate(([0], np.cumsum([len(c) for c in comp])))
            out, st = emu.decompress(b''.join(comp), offs, rows, nc, dtype, fl)
            assert not st.any() and out.tobytes() == x.tobytes(), (order, td, sd)


@pytest.mark.parametrize('dtype', ['float32', 'float64'])
@pytest.mark.parametrize('nc', [7, 449, 1793])
def test_emulated_float_special_values(emu, dtype, nc):
    """Signed zeros, subnormals, differences that overflow, inf - inf, quiet NaNs with payloads and signalling NaNs at
    the first and last row of every chunk and at the first and last column, through the forward and inverse kernels,
    compress and decompress, in both orders and all four difference settings.  The chunk's first row must be copied,
    not reduced by zero: that would quiet a signalling NaN there.  (The host emulation computes with the host's NaN
    rules, so it cannot show the device's; tests/test_gpu_transform_regimes.py checks those on a GPU.)"""
    from transform_cases import FLAG_SETS, NAN_PAYLOAD_SKIP, check_four_paths, float_data, nan_payloads_checked, \
        ragged_rows
    rows = ragged_rows(dtype, nc, tail=0 if nc > 1000 else 40)
    for kind in ('smooth', 'wild'):
        x = float_data(kind, dtype, rows, nc, seed=nc)
        for order in 'FC':
            for td, sd in FLAG_SETS:
                check_four_paths(emu, x, rows, td, sd, order)
    if not nan_payloads_checked():
        pytest.skip(NAN_PAYLOAD_SKIP)


def test_emulated_inverse_ragged_batches(emu):
    """The single-pass inverse over chunks of very different lengths in one launch (tickets of tiles past the end of a
    short chunk), ragged last tiles, tiles too small for a bulk store, every thread-per-channel regime, the 64-bit cells,
    spatial sums on top, the same cells used twice."""
    from mtscomp_b200 import _native
    rng = np.random.default_rng(3)
    for nc, dt, ns in ((40, 'int16', [300, 77, 31, 1, 1500]), (385, 'int16', [210, 64]), (9, 'int64', [130, 8]),
                       (33, 'uint8', [333, 2]), (3, 'int16', [1, 2, 700]), (900, 'int32', [50, 9]), (1800, 'int16', [70])):
        x = np.cumsum(rng.integers(-3, 4, (sum(ns), nc)), axis=0).astype(dt)
        rows = np.concatenate(([0], np.cumsum(ns)))
        for td, sd in ((True, False), (True, True), (False, True)):
            kw = dict(do_time_diff=td, do_spatial_diff=sd, chunk_order='F')
            comp = [ora.encode_chunk(x[rows[i]:rows[i + 1]], **kw) for i in range(len(ns))]
            offs = np.concatenate(([0], np.cumsum([len(c) for c in comp])))
            for rep in range(2):
                out, st = emu.decompress(b''.join(comp), offs, rows, nc, dt, _native.flags_of(td, sd, 'F'))
                assert not st.any() and np.array_equal(out, x), (nc, dt, td, sd)


def test_emulated_inverse_lookback_epochs(emu):
    """inv_tile_kernel tags its look-back cells with a launch epoch instead of clearing them: repeated launches over the
    same cells, other shapes in between, and the wrap of the epoch counter."""
    from mtscomp_b200 import _native
    rng = np.random.default_rng(5)
    cases = []
    for nc, dt, ns in ((40, 'int16', [300, 300, 77]), (40, 'int32', [500]), (7, 'int64', [260, 90]), (40, 'uint8', [333, 20])):
        x = np.cumsum(rng.integers(-3, 4, (sum(ns), nc)), axis=0).astype(dt)
        rows = np.concatenate(([0], np.cumsum(ns)))
        comp = [ora.encode_chunk(x[rows[i]:rows[i + 1]]) for i in range(len(ns))]
        cases.append((x, rows, b''.join(comp), np.concatenate(([0], np.cumsum([len(c) for c in comp]))), nc, dt))
    for rep in range(3):                                    # element sizes alternate: the cells are cleared in between
        for x, rows, comp, offs, nc, dt in cases:
            out, st = emu.decompress(comp, offs, rows, nc, dt, _native.TIME_DIFF)
            assert not st.any() and np.array_equal(out, x)
    x, rows, comp, offs, nc, dt = cases[0]
    seen = []
    for rep in range(8):                                    # same element size: epochs count up and wrap
        if rep == 2:
            emu.set_param('inv_epoch', 0x3ffc)
        out, st = emu.decompress(comp, offs, rows, nc, dt, _native.TIME_DIFF)
        assert not st.any() and np.array_equal(out, x)
        seen.append(emu.get_param('inv_epoch'))
    assert seen[1] == seen[0] + 1 and min(seen) == 1 and max(seen) == 0x3fff


def test_emulated_false_index_is_not_trusted(emu):
    """The host logic around the in-band index, without a GPU (the B200 version is in test_gpu_parity_holes.py): bytes
    behind a reference-written stream that pass every check of both index formats must not change what the chunk
    decodes to — zlib ignores them — while a damaged stream under a genuine index is still reported."""
    import struct
    from mtscomp_b200 import _native, synth
    ns, nc = 6000, 24
    x = synth.ap_chunk(ns, nc, seed=77)
    z = ora.encode_chunk(x)
    raw, seg = x.nbytes, 252000                                   # 21 channel runs of 12000 bytes
    k = (raw + seg - 1) // seg
    body = len(z) - 8
    lens = [body // k] * k
    lens[-1] += body - sum(lens)
    v1 = z + b''.join(struct.pack('<I', v) for v in lens) + struct.pack('<IIII', seg, k, 0x4253544D, sum(lens))
    n_sub = sum((min(seg, raw - j * seg) + 8191) // 8192 + (1 if min(seg, raw - j * seg) > 4096 else 0) for j in range(k))
    table = b''.join(struct.pack('<I', 20000 | (3 << 17)) for _ in range(n_sub))
    v2 = z + table + b''.join(struct.pack('<I', v) for v in lens) + struct.pack('<II', 8192, 1024) + \
        struct.pack('<IIII', seg, k, 0x3253544D, sum(lens))
    fl = _native.TIME_DIFF
    for forged in (v1, v2):
        assert zlib.decompress(forged) == ora.transform_chunk(x)
        out, st = emu.decompress(forged, [0, len(forged)], [0, ns], nc, np.int16, fl)
        assert not st.any() and np.array_equal(out, x)
    comp, offs = emu.compress(x, [0, ns], fl)
    bad = bytearray(comp)
    bad[len(bad) // 3] ^= 0x40
    try:
        _, st = emu.decompress(bytes(bad), offs, [0, ns], nc, np.int16, fl)
    except _native.NativeError:
        st = [1]
    assert st[0] != 0


def test_emulated_fuzz_of_valid_zlib_streams(emu):
    """A reduced form of the B200 fuzz (test_gpu_parity_holes.py): whatever zlib writes must decode — levels, strategies,
    window sizes, memLevels, on data with long runs (length-258 matches), far matches (distance 32768), periodic,
    low-entropy and incompressible content — through the block-parallel path (streams of 64 KB and more) and the
    serial decoder."""
    rng = np.random.default_rng(99)
    n = 90_000
    far = rng.integers(0, 256, 32768, dtype=np.uint8)
    inputs = [rng.integers(0, 256, n, dtype=np.uint8), rng.integers(0, 4, n, dtype=np.uint8),
              np.tile(np.arange(7, dtype=np.uint8), n // 7 + 1)[:n],
              np.repeat(rng.integers(0, 256, n // 300 + 1, dtype=np.uint8), 300)[:n],
              np.concatenate([far, far, far[:1000], rng.integers(0, 256, 5000, dtype=np.uint8), far])[:n]]
    strategies = [zlib.Z_DEFAULT_STRATEGY, zlib.Z_FILTERED, zlib.Z_HUFFMAN_ONLY, zlib.Z_RLE, zlib.Z_FIXED]
    for data in inputs:
        for level, strat, wbits, mem in [(0, 0, 15, 8), (6, 0, 15, 8), (9, 0, 15, 9), (6, 2, 15, 8), (6, 3, 15, 8), (6, 4, 15, 8),
                                         (9, 0, 9, 1), (2, 3, 10, 5)]:
            co = zlib.compressobj(level, zlib.DEFLATED, wbits, mem, strategies[strat])
            z = co.compress(data.tobytes()) + co.flush()
            out, st = emu.decompress(z, [0, len(z)], [0, len(data)], 1, np.uint8, 0)
            assert not st.any() and np.array_equal(out[:, 0], data), (level, strat, wbits, mem)


@pytest.mark.parametrize('shared', [False, True])
def test_emulated_contexts_from_several_threads(shared):
    """The reference calls its codec seam from n_threads pool threads at once (mtscomp.py:422, 648).  Here a context is
    one stream plus its scratch: callers either share one (calls are serialised by the binding's lock) or own one each
    (nothing is shared between contexts: no device globals, per-context scratch, staging and look-back cells)."""
    import threading
    from mtscomp_b200 import _native, build, synth
    lib = _native.load_library(build.build_emulation())
    codecs = [_native.Codec(0, lib=lib) for _ in range(1 if shared else 4)]
    res = {}

    def work(k):
        try:
            cd = codecs[0 if shared else k]
            x = synth.ap_chunk(2000, 40, seed=300 + k)
            rows = [0, 700, 2000]
            for rep in range(2):
                comp, offs = cd.compress(x, rows, _native.TIME_DIFF)
                for i in range(2):
                    assert zlib.decompress(bytes(comp[offs[i]:offs[i + 1]])) == ora.transform_chunk(x[rows[i]:rows[i + 1]])
                out, st = cd.decompress(comp, offs, rows, 40, np.int16, _native.TIME_DIFF)
                assert not st.any() and np.array_equal(out, x)
            res[k] = True
        except Exception as e:                      # noqa: BLE001 (reported below, from the main thread)
            res[k] = repr(e)

    th = [threading.Thread(target=work, args=(k,)) for k in range(4)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    for cd in codecs:
        cd.close()
    assert res == {k: True for k in range(4)}, res


def test_emulated_plain_stream_checksum_from_the_resolve_kernel(emu):
    """For a reference-written (index-less) stream that par_lz_kernel produces completely, the adler32 compared with the
    stream's trailer is the one that kernel sums from the bytes it stores: a wrong trailer, and any bit flipped in the
    body that zlib objects to, must still be reported — per chunk, the neighbours untouched."""
    from mtscomp_b200 import _native, synth
    fl = _native.TIME_DIFF
    xs = [synth.ap_chunk(3000, 40, seed=s) for s in range(4)]
    zs = [ora.encode_chunk(x) for x in xs]
    rows = np.arange(5) * 3000
    for pos, bit in ((-1, 1), (-4, 0x80), (-2, 4)):
        b = bytearray(zs[2])
        b[pos] ^= bit
        parts = [zs[0], zs[1], bytes(b), zs[3]]
        offs = np.concatenate(([0], np.cumsum([len(c) for c in parts])))
        out, st = emu.decompress(b''.join(parts), offs, rows, 40, np.int16, fl)
        assert st[2] != 0 and not st[[0, 1, 3]].any()
        for k in (0, 1, 3):
            assert np.array_equal(out[rows[k]:rows[k + 1]], xs[k])
    rng = np.random.default_rng(0)
    z = zs[0]
    for t in range(12):
        b = bytearray(z)
        b[int(rng.integers(2, len(z) - 4))] ^= 1 << int(rng.integers(0, 8))
        try:
            zlib.decompress(bytes(b))
            accepted = True
        except zlib.error:
            accepted = False
        out, st = emu.decompress(bytes(b), [0, len(b)], [0, 3000], 40, np.int16, fl)
        assert (st[0] == 0) == accepted
