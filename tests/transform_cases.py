"""Shared by the transform-stage tests (GPU and host emulation): ragged chunk batches, float arrays with IEEE special
values planted where the kernels' edge cases are, and the four-path check of a codec against oracle/codec.py.

Every comparison is of bit patterns: `np.array_equal` treats NaN != NaN and would hide a wrong payload.

NaN contract: the reference is NumPy in the array's own dtype on an x86-64 host, where a difference or sum with a NaN
operand returns that operand quieted (the first one if both are NaN) and inf - inf gives the default NaN 0xffc00000
(float64: 0xfff8000000000000).  On x86-64 the NaNs must match bit for bit; elsewhere the NaN positions must match and
only the payloads go unchecked (`nan_payloads_checked()`)."""
import platform
import zlib

import numpy as np

from oracle import codec as ora

IS_X86_64 = platform.machine().lower() in ('x86_64', 'amd64')
NAN_PAYLOAD_SKIP = ('NaN payloads are only compared on x86-64 hosts, where NumPy gives the NaNs that the files '
                    'written and read by the reference hold; NaN positions and every other bit were compared')
FLAG_SETS = ((True, False), (True, True), (False, True), (False, False))   # (time difference, spatial difference)
INV_TILE_MAXT = 448                                                         # transform.cuh


def nan_payloads_checked():
    return IS_X86_64


def tile_rows_f(nc, itemsize):
    """Rows TT = G * R of a tile of the channel-major tile kernels at this width (R = 32 / itemsize rows per run,
    G = 4, 2, 1 for 1, 2, 4 channels per thread); past 4 * 448 channels the generic kernels take over (G = 4 here)."""
    R = 32 // itemsize
    G = 4 if nc <= INV_TILE_MAXT else 2 if nc <= 2 * INV_TILE_MAXT else 1 if nc <= 4 * INV_TILE_MAXT else 4
    return G * R


def ragged_rows(dtype, nc, tail=300):
    """Chunk bounds of a batch whose chunks are 1 row, 7 rows, a run (R) -1 / exact / +1, two tiles + 3 and `tail`
    rows: ragged runs and tiles at every start alignment the row pitch allows."""
    isz = np.dtype(dtype).itemsize
    R, TT = 32 // isz, tile_rows_f(nc, isz)
    ns = [1, 7, R - 1, R, R + 1, 2 * TT + 3] + ([tail] if tail else [])
    return np.concatenate(([0], np.cumsum(ns))).astype(np.int64)


def int_data(kind, dtype, n, nc, seed):
    rng = np.random.default_rng(seed)
    info = np.iinfo(dtype)
    if kind == 'random':                            # full range: every difference wraps somewhere
        return rng.integers(info.min, info.max, (n, nc), dtype=dtype, endpoint=True)
    return np.cumsum(rng.integers(-40, 41, (n, nc)), axis=0).astype(dtype)   # smooth: the encoder finds matches


def _bits(dtype, *words):
    u = np.uint32 if np.dtype(dtype).itemsize == 4 else np.uint64
    return np.array(words, dtype=u).view(dtype)


def special_stamps(dtype):
    """2 x 2 blocks of special values; placed in a chunk, each value has a neighbour in time and in space."""
    dt = np.dtype(dtype)
    fi = np.finfo(dt)
    tiny = dt.type(1e-45) if dt.itemsize == 4 else dt.type(5e-324)             # smallest subnormal
    if dt.itemsize == 4:
        qnan, qnan2, nqnan, snan, nsnan = _bits(dt, 0x7fc00456, 0x7fc7abcd, 0xffc01234, 0x7f800001, 0xff812345)
    else:
        qnan, qnan2, nqnan, snan, nsnan = _bits(dt, 0x7ff8000000000456, 0x7ff80000abcdef01, 0xfff8000000001234,
                                                 0x7ff0000000000001, 0xfff0000000012345)
    inf, mx = dt.type(np.inf), fi.max
    one = dt.type(1)
    return [np.array(s, dtype=dt) for s in (
        [[0.0, -0.0], [-0.0, 0.0]],                 # signed zeros
        [[tiny, -tiny], [tiny, 0.0]],               # subnormals
        [[mx, -mx], [-mx, mx]],                     # differences overflow to +-inf
        [[inf, inf], [inf, -inf]],                  # inf - inf
        [[qnan, one], [qnan2, nqnan]],              # quiet NaNs with payloads (two in a row: NaN - NaN)
        [[snan, 2 * one], [nsnan, qnan]],           # signalling NaNs
    )]


def float_data(kind, dtype, rows, nc, seed):
    """A smooth signal or a wide-dynamic-range array (differences not exact), with the special stamps planted at the
    first and the last row of every chunk (so at row 0 and the last row of the batch), at column 0, the last column and
    columns in between."""
    dt = np.dtype(dtype)
    rng = np.random.default_rng(seed)
    n = int(rows[-1])
    if kind == 'smooth':
        x = np.cumsum(rng.normal(0, 1, (n, nc)), axis=0)
    else:
        x = rng.normal(0, 1, (n, nc)) * 10. ** rng.integers(-30, 30, (n, nc))
    x = x.astype(dt)
    stamps = special_stamps(dt)
    anchors = sorted({int(r) for i in range(len(rows) - 1) for r in (rows[i], rows[i + 1] - 1)})
    cols = sorted(set(range(0, nc, max(2, nc // 6))) | {nc - 1})
    for a, r in enumerate(anchors):
        r0 = min(r, n - 2) if n > 1 else 0
        for ci, c in enumerate(cols):
            c0 = min(c, nc - 2) if nc > 1 else 0
            s = stamps[(a + ci) % len(stamps)]
            blk = x[r0:r0 + 2, c0:c0 + 2]
            blk[...] = s[:blk.shape[0], :blk.shape[1]]
    return x


def assert_same_bits(got, want, dtype, what):
    """got / want: arrays or bytes of elements of `dtype`; equal bit for bit (NaN payloads: see the module's doc)."""
    dt = np.dtype(dtype)
    u = np.dtype('u%d' % dt.itemsize)
    g = np.frombuffer(np.ascontiguousarray(got).tobytes(), dtype=u)
    w = np.frombuffer(np.ascontiguousarray(want).tobytes(), dtype=u)
    assert g.size == w.size, '%s: %d elements, want %d' % (what, g.size, w.size)
    bad = g != w
    if dt.kind == 'f' and not nan_payloads_checked():
        gn, wn = np.isnan(g.view(dt)), np.isnan(w.view(dt))
        bad = (gn != wn) | (~wn & bad)
    if bad.any():
        i = np.flatnonzero(bad)[:6]
        raise AssertionError('%s: %d of %d elements differ, e.g. at %s: got %s, want %s' % (
            what, int(bad.sum()), g.size, i.tolist(), [hex(v) for v in g[i]], [hex(v) for v in w[i]]))


def check_four_paths(cd, x, rows, td, sd, order):
    """The codec `cd` against the reference on the batch x[rows[i]:rows[i + 1]]: forward transform, inverse transform
    (with its adler32), compress (zlib must return the reference's transform bytes; the codec decodes its own streams)
    and decompress of reference-written streams."""
    with np.errstate(all='ignore'):                 # overflow and inf - inf are what these arrays are for
        _check_four_paths(cd, x, rows, td, sd, order)


def _check_four_paths(cd, x, rows, td, sd, order):
    from mtscomp_b200 import _native
    fl = _native.flags_of(td, sd, order)
    kw = dict(do_time_diff=td, do_spatial_diff=sd, chunk_order=order)
    dt, nc = x.dtype, x.shape[1]
    tag = '%s nc=%d td=%d sd=%d %s' % (dt.name, nc, td, sd, order)
    chunks = [x[rows[i]:rows[i + 1]] for i in range(len(rows) - 1)]
    want_t = [ora.transform_chunk(c, **kw) for c in chunks]
    want_x = [ora.untransform_bytes(t, len(c), nc, dt, **kw) for t, c in zip(want_t, chunks)]
    for i, (c, t, u) in enumerate(zip(chunks, want_t, want_x)):
        assert_same_bits(cd.delta_transform(c, fl), t, dt, '%s chunk %d: delta_transform' % (tag, i))
        back, ad = cd.inverse_transform(t, len(c), nc, dt, fl, want_adler=True)
        assert_same_bits(back, u, dt, '%s chunk %d: inverse_transform' % (tag, i))
        assert ad == zlib.adler32(t), '%s chunk %d: adler32' % (tag, i)
    comp, offs = cd.compress(x, rows, fl)
    for i, t in enumerate(want_t):
        assert_same_bits(zlib.decompress(bytes(comp[offs[i]:offs[i + 1]])), t, dt, '%s chunk %d: compress' % (tag, i))
    out, st = cd.decompress(comp, offs, rows, nc, dt, fl)
    assert not st.any(), tag
    assert_same_bits(out, np.concatenate(want_x), dt, '%s: decompress of own streams' % tag)
    parts = [ora.encode_chunk(c, **kw) for c in chunks]
    roffs = np.concatenate(([0], np.cumsum([len(p) for p in parts])))
    ref = [ora.decode_chunk(p, len(c), nc, dt, **kw) for p, c in zip(parts, chunks)]
    out2, st2 = cd.decompress(b''.join(parts), roffs, rows, nc, dt, fl)
    assert not st2.any(), tag
    assert_same_bits(out2, np.concatenate(ref), dt, '%s: decompress of reference streams' % tag)
