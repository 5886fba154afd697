"""CPU: the match finder's output pinned byte for byte under the host emulation of the kernels.  A step whose positions
all have 258 + 16 bytes of input after them runs a body compiled without bounds tests, the last step or two of a
segment the guarded one; the split must not change one byte.  The inputs cover both strides (int16: 2 bytes per
position, else 1), segments of more than 65 536 positions (16-bit position numbers wrap), hash-bucket collisions of
whole steps (runs, plateaus, zeros: the settle pass, 258-byte matches), a last step shorter than 258 bytes, chunks too
small for an index, and the spatial difference; each with and without the index."""
import hashlib
import zlib

import numpy as np
import pytest

from oracle import codec as ora


def _cases():
    rng = np.random.default_rng(11)         # integer generators only: the same arrays on every platform
    walk = np.cumsum(rng.integers(-3, 4, (40000, 24)), axis=0)

    def ap(ns, nc):                          # AP-like: smooth common signal + per-channel noise, int16
        common = np.cumsum(rng.integers(-4, 5, ns))[:, None]
        return (common // 4 + rng.integers(-12, 13, (ns, nc))).astype(np.int16)

    runs = np.zeros((2000, 16), dtype=np.int16); runs[:, 3] = 17; runs[1000:, 5] = -3
    return [   # name, array, chunk rows, time difference, spatial difference
        ('ap_int16', ap(8000, 64), [0, 5000, 8000], True, False),
        ('walk_uint8', (walk & 0xff).astype(np.uint8), [0, 40000], True, False),
        ('walk_int8', (walk % 100).astype(np.int8), [0, 25000, 40000], False, False),
        ('walk_float32', (walk[:10000] * 0.25).astype(np.float32), [0, 10000], True, False),
        ('runs_int16', runs, [0, 1000, 2000], True, False),
        ('plateaus_int16', np.repeat(rng.integers(-200, 200, (40, 12)), 100, axis=0).astype(np.int16), [0, 4000], True,
         False),
        ('zeros_uint8', np.zeros((300000, 1), dtype=np.uint8), [0, 300000], False, False),
        # one segment whose last step holds 100 bytes: 3 * 1024 + 100 int16 bytes, 5 * 512 + 100 uint8 bytes
        ('short_last_step_int16', ap(793, 2), [0, 793], True, False),
        ('short_last_step_uint8', rng.integers(0, 3, (5 * 512 + 100, 1)).astype(np.uint8), [0, 5 * 512 + 100], True,
         False),
        ('tiny_chunks_int16', ap(1400, 3), [0, 200, 1400], True, False),
        ('spatial_int16', ap(1000, 385), [0, 1000], True, True),
    ]


CASES = _cases()
# sha256 of (chunk offsets as int64 | compressed bytes), index on / off
DIGESTS = {
    'ap_int16': ('e2b9bb5a0e445a027dd162c1f8e582dbf2554f1ec24723c938cef597f017323a',
                 '0e79ec82d02c53b3a3a959f164a2b798addf64beb54197f37d7cdfb4a6c88a17'),
    'walk_uint8': ('091d993a984149223058cbfe212189031bba95ac5895e32acc9fa856fd2d8729',
                   '723c82d89bd059e8f32ec6d1150c4955f15058edf918879c8cae0162c9252835'),
    'walk_int8': ('5c8227c4982153c9ed93ef9f464215bb15a7752e25063d5ed98055b0f056a303',
                  '3499ec10b209b3caa2cc8fe4215c1a0b348858f55a9ab4ec9c268940f12d4d8f'),
    'walk_float32': ('6a726d9ed5decaac14bd3ffed8c726d452d9c9c0f861a05946aa6a2ac5fd8e27',
                     'eb3bdf62d2167c35498a1ed5d6656e1892951cba8eb52f63f259bd3f77373954'),
    'runs_int16': ('bd15d918e5adecc615b202906fdfe8c5a9ed3c84f282dd4043d65a377870e142',
                   'c07c92e5740f818ee3149ae95cf6ba691c6cf0b775142a5c5ab2e4c093772feb'),
    'plateaus_int16': ('412d3c199ad4d88df1e559c250c496c837cb6d84d75211198769016c9ccbb8bf',
                       '62131d3d0aa74476170d04d81a8d2ea00e59d26c8d1af276ced931824c9c8e0c'),
    'zeros_uint8': ('ea6bd281813627ea9be7a161fb32564b15cf96368d069219462da2c415bd0cb5',
                    '9acc713e741c80066a2b8de6b9ee91cdcb4adac933bfbf57f787944a8ca3af94'),
    'short_last_step_int16': ('a90991841444791efb695126b9d6a6b396c66c326712c3f6bbd6bc019e21b891',
                              '68928c803b52a7962980e3bcea1b8150c0fd629512cdbe84257e58dc28b80e71'),
    'short_last_step_uint8': ('6fa66bcb23653f9ff8ca7327b5f339b6f781ce300b844007ee3cedfdb39d339b',
                              '2718bfba83c095bcd0d12e7e508047882a1ba30e62cecbeab6e6d65848ce4bf8'),
    'tiny_chunks_int16': ('5ab3640ef89b80a76219715780ac90dd7051f0397fca034face5e7fff9af5869',
                          'd70688a0eaadafe1fbc8020bda94cb7a8d66d17817a95420e6d23bbd1acf657c'),
    'spatial_int16': ('134c7983661954cf4b7cae56c9295c040d4a0caad1dc631444f5d68171a50fce',
                      '358827813d35921359264e849e472d879b0c91a2153822a6f779355d604a0667'),
}


@pytest.fixture(scope='module')
def emu():
    from mtscomp_b200 import _native, build
    c = _native.Codec(0, lib=_native.load_library(build.build_emulation()))
    yield c
    c.close()


def compress(codec, x, rows, td, sd, write_index):
    from mtscomp_b200 import _native
    saved = codec.get_param('write_index')
    codec.set_param('write_index', write_index)
    try:
        comp, offs = codec.compress(x, rows, _native.flags_of(td, sd, 'F'))
    finally:
        codec.set_param('write_index', saved)
    return bytes(comp), np.asarray(offs, dtype=np.int64)


@pytest.mark.parametrize('write_index', [1, 0])
@pytest.mark.parametrize('case', CASES, ids=[c[0] for c in CASES])
def test_match_finder_output_is_pinned(emu, case, write_index):
    name, x, rows, td, sd = case
    comp, offs = compress(emu, x, rows, td, sd, write_index)
    for i in range(len(rows) - 1):           # a valid zlib stream of the transformed chunk
        assert zlib.decompress(comp[offs[i]:offs[i + 1]]) == ora.transform_chunk(x[rows[i]:rows[i + 1]], td, sd)
    assert hashlib.sha256(offs.tobytes() + comp).hexdigest() == DIGESTS[name][1 - write_index]
