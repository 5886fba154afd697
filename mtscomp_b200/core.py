# -*- coding: utf-8 -*-
"""Writer / Reader / compress / decompress / check with mtscomp's API and file format, on the B200 codec.

Behavioural mirror of the reference's low- and high-level API (mtscomp.py:216-997): same constructor options,
attributes, return values, file layout (.cbin = concatenated per-chunk zlib streams, .ch = sorted indented JSON with the
same keys) and error behaviour.  The per-chunk codec — `Writer._compress_chunk` (mtscomp.py:375-397) and
`Reader.read_chunk` (mtscomp.py:602-635) — does not run NumPy/zlib here: whole batches of chunks go through the C ABI
(`_native.Codec`) to the sm_100a kernels.  There is no CPU codec path.

Differences that do not change results: a batch is one GPU call instead of `n_threads` zlib threads; the thread-pool
methods are kept as no-op compatible shims; GPU-written chunks carry a small segment index after each zlib stream (zlib
ignores trailing bytes), which lets the GPU Reader decode a chunk's segments in parallel.
"""

import bisect
from collections import OrderedDict
from functools import lru_cache, partial
import contextlib
import hashlib
import json
from concurrent import futures
from concurrent.futures import ThreadPoolExecutor
import os
import os.path as op
from pathlib import Path
from threading import Lock

import numpy as np
from tqdm import tqdm

from . import _native
from .config import Bunch, CHECK_ATOL, FORMAT_VERSION, clip, logger, read_config
from .rawio import load_raw_data

_seek_lock = Lock()
CRITICAL_ERROR_URL = "https://github.com/int-brain-lab/mtscomp/issues/new?title=Critical+error"
CRITICAL_CHECK_FAILED = ("CRITICAL ERROR: automatic check failed when compressing the data. "
                         "Report immediately to " + CRITICAL_ERROR_URL)
CHECK_RTOL = 1e-5            # np.allclose's default, which the reference's check() uses for floats
GPU_BATCH_CHUNKS = 64        # chunks handed to the GPU per call by Writer.write / Reader.tofile ...
GPU_BATCH_BYTES = 256 << 20  # ... and at most this many raw bytes: the pinned staging (two raw + two compressed buffers in
                             # the Writer) stays near 1 GB -- pinning host memory costs about 0.7 s per GB on the B200 box
MAX_CHUNK_BYTES = 0x7fffffff  # the kernels index a chunk with 32 bits


def _require_integer_dtype(dtype):
    """dtypes the CUDA codec handles: int8..int64 / uint8..uint64 (modular arithmetic, as NumPy's) and float32 /
    float64 (IEEE differences, sequential sums in np.cumsum's order: the decoded values equal the reference Reader's
    bit for bit, which — as in the reference — are close to, not identical with, what was written)."""
    dtype = np.dtype(dtype)
    if dtype.byteorder not in ('=', '|', '<' if np.little_endian else '>'):
        raise NotImplementedError("mtscomp_b200 works on native-endian data; dtype %s is not supported." % dtype.str)
    ok_int = np.issubdtype(dtype, np.integer) and dtype.itemsize in (1, 2, 4, 8)
    ok_float = dtype.kind == 'f' and dtype.itemsize in (4, 8)
    if not (ok_int or ok_float):
        raise NotImplementedError(
            "mtscomp_b200 implements the codec for int8..int64 and float32/float64; dtype %s is not "
            "supported and there is no CPU fallback." % dtype)
    return dtype


@contextlib.contextmanager
def _codec_param(codec, name, value):
    """Set a codec tunable for the duration of a block (None: leave it alone)."""
    if value is None:
        yield
        return
    old = codec.get_param(name)
    codec.set_param(name, int(bool(value)))
    try:
        yield
    finally:
        codec.set_param(name, old)


def _codec_for(config):
    dev = config.get('device', None)
    return _native.default_codec(dev)


_READ_POOL = None


def _read_pool():
    global _READ_POOL
    if _READ_POOL is None:
        _READ_POOL = ThreadPoolExecutor(4)
    return _READ_POOL


def _batch_ranges(bounds, row_bytes, first, last):
    """[lo, hi) chunk ranges covering [first, last): at most GPU_BATCH_CHUNKS chunks and GPU_BATCH_BYTES raw bytes each
    (a single chunk larger than that forms its own batch)."""
    lo = first
    while lo < last:
        hi = lo + 1
        while hi < last and hi - lo < GPU_BATCH_CHUNKS and (bounds[hi + 1] - bounds[lo]) * row_bytes <= GPU_BATCH_BYTES:
            hi += 1
        yield lo, hi
        lo = hi


def _pipeline(n, stage, run, finish=None, lanes=0, desc=None, quiet=False):
    """Run batches 0..n-1 of a whole-file operation, the caller holding codec.stage_lock.  Batch k uses the pinned
    buffers of slot k & 1.  stage(k, slot) fills them with host reads on a stager thread, one batch ahead; run(k, slot,
    staged) makes the GPU call and raises the operation's own errors; finish(k, slot, result) returns the batch's
    finisher work, whose callable i runs on lane i: one thread per lane keeps each lane in batch order (the updates of
    one SHA-1), and the lanes run side by side.  stage(k) waits for batch k-2's finisher work, which shares its slot.
    On an error every worker is done before it propagates, and the earliest failing batch's error is raised."""
    fins = []                                   # fins[k]: batch k's finisher futures

    def stage_after(k):
        for f in fins[k - 2] if k >= 2 else ():
            f.result()                          # batch k-2 shares the slot; its failure stops the pipeline here
        return stage(k, k & 1)

    with ThreadPoolExecutor(1, 'mtsb-stage') as stager, contextlib.ExitStack() as stack:
        pools = [stack.enter_context(ThreadPoolExecutor(1, 'mtsb-finish')) for _ in range(lanes)]
        k, nxt = 0, (stager.submit(stage_after, 0) if n else None)
        try:
            for k in tqdm(range(n), desc=desc, disable=quiet):
                staged = nxt.result()
                nxt = stager.submit(stage_after, k + 1) if k + 1 < n else None
                result = run(k, k & 1, staged)
                work = finish(k, k & 1, result) if finish else ()
                fins.append([pool.submit(fn) for pool, fn in zip(pools, work)])
            for fs in fins:
                for f in fs:
                    f.result()
        except BaseException as e:
            futures.wait(([nxt] if nxt else []) + [f for fs in fins for f in fs])
            earlier = [f.exception() for fs in fins[:k] for f in fs if f.exception() is not None]
            if earlier and earlier[0] is not e:
                raise earlier[0] from None
            raise


def _check_chunk_limits(bounds, n_channels, itemsize):
    big = max(bounds[i + 1] - bounds[i] for i in range(len(bounds) - 1)) * n_channels * itemsize
    if big > MAX_CHUNK_BYTES:
        raise NotImplementedError(
            "a chunk of %d bytes exceeds the %d bytes the CUDA codec handles per chunk; use a shorter chunk_duration."
            % (big, MAX_CHUNK_BYTES))


# ------------------------------------------------------------------------------------------------------------------
# Standalone transforms (reference mtscomp.py:143-169), executed by the K1 / K4 kernels
# ------------------------------------------------------------------------------------------------------------------

def diff_along_axis(chunk, axis=None):
    """np.diff along `axis` keeping the first row/column (reference mtscomp.py:143-159), on the GPU."""
    if axis is None:
        return chunk
    assert 0 <= axis < chunk.ndim
    dtype = _require_integer_dtype(chunk.dtype)
    flags = (_native.TIME_DIFF if axis == 0 else _native.SPATIAL_DIFF) | _native.ORDER_C
    out = _native.default_codec().delta_transform(np.ascontiguousarray(chunk), flags)
    return out.view(dtype).reshape(chunk.shape)


def cumsum_along_axis(chunk, axis=None):
    """np.cumsum along `axis` in the array's own dtype (reference mtscomp.py:162-169), on the GPU."""
    if axis is None:
        return chunk
    assert 0 <= axis < chunk.ndim
    dtype = _require_integer_dtype(chunk.dtype)
    flags = (_native.TIME_DIFF if axis == 0 else _native.SPATIAL_DIFF) | _native.ORDER_C
    c = np.ascontiguousarray(chunk)
    return _native.default_codec().inverse_transform(c.tobytes(), c.shape[0], c.shape[1], dtype, flags)


# ------------------------------------------------------------------------------------------------------------------
# Writer
# ------------------------------------------------------------------------------------------------------------------

class Writer:
    """Compress a raw (memory-mapped) recording into `.cbin` + `.ch` (reference mtscomp.py:216-511).

    Options: chunk_duration, algorithm ('zlib'), comp_level (recorded only, as in the reference: SURVEY G1),
    do_time_diff, do_spatial_diff, chunk_order, n_threads (batch size attribute), check_after_compress,
    before_check (callback), quiet; plus `device` (CUDA device index) and `write_index` (False: no in-band index after
    the chunks' zlib streams, i.e. the reference's exact .cbin layout; default: the codec's setting, on).
    """

    def __init__(self, before_check=None, **kwargs):
        self.pool = None
        self.quiet = kwargs.pop('quiet', False)
        cfg = read_config(**kwargs)
        self.config = cfg
        assert cfg.algorithm == 'zlib', "Only zlib is currently supported."
        for key in ('chunk_duration', 'algorithm', 'comp_level', 'do_time_diff', 'do_spatial_diff', 'n_threads',
                    'check_after_compress', 'chunk_order'):
            setattr(self, key, cfg[key])
        self.before_check = before_check or (lambda x: None)

    # -- opening --------------------------------------------------------------------------------------------------
    def open(self, data_path, sample_rate=None, n_channels=None, dtype=None, offset=None, mmap=True):
        """Open the raw file (flat binary or .npy) and compute the chunk layout (reference mtscomp.py:257-339)."""
        self.data_path = Path(data_path)
        sample_rate = sample_rate or self.config.get('sample_rate', None)
        if not sample_rate:
            raise ValueError("Please provide a sample rate (-s option in the command-line).")
        if str(data_path).endswith('.npy'):
            self.data = np.load(data_path, mmap_mode='r')
            self.shape = self.data.shape
            if self.data.ndim >= 3:
                self.data = np.reshape(self.data, (-1, self.data.shape[-1]))
            self.dtype = dtype = self.data.dtype
            self.n_channels = n_channels = self.data.shape[1]
        else:
            n_channels = n_channels or self.config.get('n_channels', None)
            if not n_channels:
                raise ValueError("Please provide n_channels (-n option in the command-line).")
            dtype = dtype or self.config.get('dtype', None)
            if not dtype:
                raise ValueError("Please provide a dtype (-d option in the command-line).")
            self.dtype = np.dtype(dtype)
            self.data = load_raw_data(data_path, n_channels=n_channels, dtype=self.dtype)
            self.shape = self.data.shape
        self.sample_rate = float(sample_rate)
        assert sample_rate > 0
        assert n_channels > 0
        self.file_size = self.data.size * self.data.itemsize
        assert self.data.ndim == 2
        self.n_samples, self.n_channels = self.data.shape
        assert self.n_samples > 0
        assert self.n_channels > 0
        assert n_channels == self.n_channels
        logger.info("Opening %s, duration %.1fs, %d channels.", data_path,
                    self.n_samples / self.sample_rate, self.n_channels)
        self._compute_chunk_bounds()
        _check_chunk_limits(self.chunk_bounds, self.n_channels, np.dtype(self.dtype).itemsize)
        self.sha1_compressed = hashlib.sha1()
        self.sha1_uncompressed = hashlib.sha1()

    def _compute_chunk_bounds(self):
        chunk_size = int(np.round(self.chunk_duration * self.sample_rate))
        bounds = list(range(0, self.n_samples, chunk_size))
        if bounds[-1] < self.n_samples:
            bounds.append(self.n_samples)
        self.chunk_bounds = bounds
        self.n_chunks = len(bounds) - 1
        assert bounds[0] == 0 and bounds[-1] == self.n_samples
        self.batch_size = self.n_threads
        self.n_batches = int(np.ceil(self.n_chunks / self.batch_size))

    def get_cmeta(self):
        """Contents of the `.ch` file (reference mtscomp.py:341-358)."""
        return {
            'version': FORMAT_VERSION,
            'algorithm': self.algorithm,
            'comp_level': self.comp_level,
            'do_time_diff': self.do_time_diff,
            'do_spatial_diff': self.do_spatial_diff,
            'dtype': str(np.dtype(self.dtype)),
            'n_channels': self.n_channels,
            'sample_rate': self.sample_rate,
            'chunk_bounds': self.chunk_bounds,
            'chunk_offsets': self.chunk_offsets,
            'chunk_order': self.chunk_order,
            'sha1_compressed': self.sha1_compressed.hexdigest(),
            'sha1_uncompressed': self.sha1_uncompressed.hexdigest(),
            'shape': self.shape,
        }

    def get_chunk(self, chunk_idx):
        assert 0 <= chunk_idx <= self.n_chunks - 1
        return self.data[self.chunk_bounds[chunk_idx]:self.chunk_bounds[chunk_idx + 1], :]

    # -- the codec seam ---------------------------------------------------------------------------------------------
    def _flags(self):
        return _native.flags_of(self.do_time_diff, self.do_spatial_diff, self.chunk_order)

    def compress_batch(self, first_chunk, last_chunk):
        """{chunk_idx: (uncompressed_chunk, compressed_bytes)} for chunks [first_chunk, last_chunk)
        (reference mtscomp.py:399-423); one batched GPU call instead of pool.map(_compress_chunk)."""
        assert 0 <= first_chunk < last_chunk <= self.n_chunks
        _require_integer_dtype(self.dtype)
        b = self.chunk_bounds
        block = np.ascontiguousarray(self.data[b[first_chunk]:b[last_chunk], :])
        rows = np.asarray(b[first_chunk:last_chunk + 1], dtype=np.int64) - b[first_chunk]
        comp, offs = _codec_for(self.config).compress(block, rows, self._flags())
        out = {}
        for k, idx in enumerate(range(first_chunk, last_chunk)):
            raw = block[rows[k]:rows[k + 1]]
            cbytes = comp[offs[k]:offs[k + 1]].tobytes()
            logger.debug("Chunk %d/%d: -%.3f%%.", idx + 1, self.n_chunks, 100 - 100 * len(cbytes) / max(raw.nbytes, 1))
            out[idx] = (raw, cbytes)
        return out

    def _compress_chunk(self, chunk_idx):
        """Single-chunk form of the seam, same return shape as the reference's (mtscomp.py:375-397)."""
        return chunk_idx, self.compress_batch(chunk_idx, chunk_idx + 1)[chunk_idx]

    def _compress_range(self, first, last, finish, lanes):
        """Compress chunks [first, last) on the _pipeline: stage reads a batch's rows from the memory map straight into
        pinned w_raw%d, run packs them into pinned w_comp%d, and finish(raw, offsets, comp) gets views of both buffers
        and the batch's chunk offsets and returns the batch's finisher work."""
        dtype = _require_integer_dtype(self.dtype)
        codec = _codec_for(self.config)
        flags = _native._fl(self._flags(), dtype)
        nc, isz, b = self.n_channels, dtype.itemsize, self.chunk_bounds
        ranges = list(_batch_ranges(b, nc * isz, first, last))

        def stage(k, slot):
            lo, hi = ranges[k]
            raw = raw_bufs[slot].array[:(b[hi] - b[lo]) * nc * isz]
            np.copyto(raw.view(dtype).reshape(-1, nc), self.data[b[lo]:b[hi], :])
            return raw

        def run(k, slot, raw):
            lo, hi = ranges[k]
            rows = np.asarray(b[lo:hi + 1], dtype=np.int64) - b[lo]
            offs = codec.compress_ptr(raw_bufs[slot].ptr, 0, rows, nc, isz, flags, comp_bufs[slot].ptr, 0, caps[k])
            return raw, offs, comp_bufs[slot].array[:int(offs[-1])]

        # write_index=False (Writer / compress() keyword, or "write_index" in ~/.mtscomp) gives exactly the reference's
        # .cbin layout, one zlib stream per chunk and nothing else; the default appends the in-band index to each chunk.
        with codec.stage_lock, _codec_param(codec, 'write_index', self.config.get('write_index')):
            # (the bound depends on write_index: computed with it set)
            caps = [sum(codec.compress_bound(b[i + 1] - b[i], nc, isz, flags) for i in range(lo, hi)) for lo, hi in ranges]
            raw_bufs = [codec.host_buffer('w_raw%d' % i, max((b[hi] - b[lo]) * nc * isz for lo, hi in ranges)) for i in (0, 1)]
            comp_bufs = [codec.host_buffer('w_comp%d' % i, max(caps)) for i in (0, 1)]
            _pipeline(len(ranges), stage, run, lambda k, slot, res: finish(*res), lanes, 'Compressing', self.quiet)

    def write(self, out, outmeta):
        """Write `.cbin` and `.ch`; returns csize / raw size (reference mtscomp.py:425-507, SURVEY G7)."""
        if not out:
            out = self.data_path.with_suffix('.c' + self.data_path.suffix[1:])
        if not outmeta:
            outmeta = self.data_path.with_suffix('.ch')
        Path(out).parent.mkdir(exist_ok=True, parents=True)
        self.chunk_offsets = [0]
        logger.info("Starting compression on the GPU.")

        # while the GPU works on batch k+1, two lanes finish batch k: one feeds the raw bytes to its SHA-1, the other
        # writes and hashes the compressed bytes.  The two digests the .ch format demands run at 1-2 GB/s per core and
        # are the ceiling of this method.
        def write_and_hash(comp):
            fb.write(comp)
            self.sha1_compressed.update(comp)

        def finish(raw, offs, comp):
            base = self.chunk_offsets[-1]
            self.chunk_offsets.extend(int(base + o) for o in offs[1:])
            return partial(self.sha1_uncompressed.update, raw), partial(write_and_hash, comp)

        with open(out, 'wb') as fb:
            self._compress_range(0, self.n_chunks, finish, 2)
            csize = fb.tell()
        assert self.chunk_offsets[-1] == csize
        ratio = csize / self.file_size
        logger.info("Wrote %s (%.1f GB, -%.3f%%).", out, csize / 1024 ** 3, 100 - 100 * ratio)
        with open(outmeta, 'w') as f:
            json.dump(self.get_cmeta(), f, indent=2, sort_keys=True)
        if self.check_after_compress:
            self.before_check(self)
            try:
                check(self.data, out, outmeta)
            except AssertionError:
                raise RuntimeError(CRITICAL_CHECK_FAILED)
            logger.debug("Automatic integrity check after compression PASSED.")
        return ratio

    def close(self):
        mm = getattr(self.data, '_mmap', None)
        if mm is not None:
            mm.close()


# ------------------------------------------------------------------------------------------------------------------
# Reader
# ------------------------------------------------------------------------------------------------------------------

class _SerialPool:
    """Stand-in returned by Reader.start_thread_pool(): the GPU call is already batched."""

    def map(self, fn, it):
        return [fn(x) for x in it]

    def close(self):
        pass

    def join(self):
        pass


class _DeviceBlock:
    """Device memory holding the decoded rows of one or more consecutive chunks.  Freed blocks go to a small per-codec
    pool instead of back to the driver: cudaMalloc / cudaFree cost 0.3 - 13 ms each on the B200 box (and cudaFree
    synchronises the device), which would dominate a 3 ms random access."""
    POOL_BLOCKS = 4

    def __init__(self, codec, nbytes):
        self.codec, self.nbytes = codec, int(nbytes)
        pool = codec.__dict__.setdefault('_block_pool', [])
        best = None
        for k, (cap, _) in enumerate(pool):
            if self.nbytes <= cap <= 2 * self.nbytes + (1 << 20) and (best is None or cap < pool[best][0]):
                best = k
        if best is not None:
            self.cap, self.ptr = pool.pop(best)
        else:
            self.cap = self.nbytes
            self.ptr = codec.device_alloc(self.cap)

    def __del__(self):
        try:
            pool = self.codec.__dict__.setdefault('_block_pool', [])
            if len(pool) < self.POOL_BLOCKS and getattr(self.codec, 'ctx', None):
                pool.append((self.cap, self.ptr))
            else:
                self.codec.device_free(self.ptr)
        except Exception:  # pragma: no cover
            pass


class _DeviceChunkCache:
    """LRU of decoded chunks kept IN DEVICE MEMORY (the reference keeps host arrays, mtscomp.py:582-588): a repeated or
    overlapping read costs one device-to-host copy of the rows asked for instead of a decode.
    Entry: chunk_idx -> (block, byte offset of the chunk in the block, bytes)."""

    def __init__(self, capacity):
        self.capacity = max(int(capacity), 1)
        self.entries = OrderedDict()

    def get(self, idx):
        e = self.entries.get(idx)
        if e is not None:
            self.entries.move_to_end(idx)
        return e

    def put(self, idx, entry):
        self.entries[idx] = entry
        self.entries.move_to_end(idx)
        while len(self.entries) > self.capacity:
            self.entries.popitem(last=False)

    def clear(self):
        self.entries.clear()


class Reader:
    """Random-access reader of `.cbin` + `.ch` (reference mtscomp.py:514-859), decoding on the GPU."""

    def __init__(self, **kwargs):
        self.pool = None
        self.cdata = None
        self.quiet = kwargs.pop('quiet', False)
        self.config = read_config(**kwargs)
        self.cache_size = self.config.cache_size
        self.check_after_decompress = self.config.check_after_decompress

    def open(self, cdata, cmeta=None):
        if cmeta is None:
            cmeta = Path(cdata).with_suffix('.ch')
        if not isinstance(cmeta, dict):
            with open(cmeta, 'r') as f:
                cmeta = json.load(f)
        assert isinstance(cmeta, dict)
        self.cmeta = Bunch(cmeta)
        m = self.cmeta
        self.n_channels = m.n_channels
        self.sample_rate = m.sample_rate
        self.dtype = np.dtype(m.dtype)
        self.chunk_offsets = m.chunk_offsets
        self.chunk_bounds = m.chunk_bounds
        self.chunk_order = m.chunk_order
        self.n_samples = self.chunk_bounds[-1]
        self.n_chunks = len(self.chunk_bounds) - 1
        self.shape = (self.n_samples, self.n_channels)
        self.ndim = 2
        self.batch_size = self.config.n_threads
        self.n_batches = int(np.ceil(self.n_chunks / self.batch_size))
        if isinstance(cdata, (str, Path)):
            if Path(cdata).suffix in ('.bin', '.dat'):  # pragma: no cover
                logger.error("File to decompress has unexpected extension %s.", Path(cdata).suffix)
            cdata = open(cdata, 'rb')
        self.cdata = cdata
        try:
            self._fd = cdata.fileno()
        except Exception:
            self._fd = None
        _check_chunk_limits(self.chunk_bounds, self.n_channels, self.dtype.itemsize)
        self._dev_cache = _DeviceChunkCache(self.cache_size)
        self.set_cache_size()

    def set_cache_size(self, cache_size=None):
        """(Re)wrap read_chunk in an LRU cache (reference mtscomp.py:582-588)."""
        if cache_size != self.cache_size:
            cache_size = cache_size or self.cache_size
            assert cache_size > 0
            self.read_chunk = lru_cache(maxsize=cache_size)(self.read_chunk)
            self.cache_size = cache_size
            if getattr(self, '_dev_cache', None) is not None:
                self._dev_cache.capacity = cache_size

    def iter_chunks(self, first_chunk=0, last_chunk=None):
        """Yield (chunk_idx, chunk_start, chunk_length) (reference mtscomp.py:590-600)."""
        last_chunk = last_chunk if last_chunk is not None else self.n_chunks - 1
        offs = self.chunk_offsets
        for idx in range(first_chunk, last_chunk + 1):
            yield idx, offs[idx], offs[idx + 1] - offs[idx]

    # -- the codec seam ---------------------------------------------------------------------------------------------
    def _flags(self):
        return _native.flags_of(self.cmeta.do_time_diff, self.cmeta.do_spatial_diff, self.chunk_order)

    def _pread(self, length, start):
        if self._fd is not None and hasattr(os, 'pread'):
            buf = os.pread(self._fd, length, start)
        else:  # pragma: no cover
            with _seek_lock:
                self.cdata.seek(start)
                buf = self.cdata.read(length)
        assert len(buf) == length
        return buf

    def _pread_into(self, view, start):
        """Fill the uint8 array `view` (pinned staging) from the .cbin at `start`, without intermediate bytes objects."""
        n = view.shape[0]
        if self._fd is not None and hasattr(os, 'preadv'):
            mv = memoryview(view)

            def part(lo, hi):
                got = lo
                while got < hi:
                    k = os.preadv(self._fd, [mv[got:hi]], start + got)
                    assert k > 0, "unexpected end of the compressed file"
                    got += k
            if n >= (4 << 20):
                # a chunk's ~9 MB come out of the page cache at memcpy speed: split the copy over a few threads
                # (preadv releases the GIL)
                nt = 4
                step = -(-n // nt)
                list(_read_pool().map(lambda a: part(a, min(a + step, n)), range(0, n, step)))
            else:
                part(0, n)
        else:
            view[:] = np.frombuffer(self._pread(n, start), dtype=np.uint8)

    def _stage_compressed(self, codec, spans, name='r_comp'):
        """Read the .cbin ranges `spans` [(start, length)] back to back into the pinned buffer `name` (one read per
        run of adjacent ranges) -> (buffer, offsets)."""
        offs = np.concatenate(([0], np.cumsum([length for _, length in spans]))).astype(np.int64)
        buf = codec.host_buffer(name, int(offs[-1]) + 64)
        k = 0
        while k < len(spans):
            j = k
            while j + 1 < len(spans) and spans[j][0] + spans[j][1] == spans[j + 1][0]:
                j += 1
            self._pread_into(buf.array[int(offs[k]):int(offs[j + 1])], spans[k][0])
            k = j + 1
        return buf, offs

    def _rows_of(self, chunk_ids):
        sizes = [self.chunk_bounds[i + 1] - self.chunk_bounds[i] for i in chunk_ids]
        return np.concatenate(([0], np.cumsum(sizes))).astype(np.int64)

    def _raise_if_corrupt(self, status, chunk_ids):
        bad = np.flatnonzero(status)
        if len(bad):
            raise IOError("Compressed chunk #%d is corrupted." % chunk_ids[int(bad[0])])

    def _decode_into(self, chunk_ids, spans, dst_ptr, dst_is_device):
        """One GPU call: chunks `chunk_ids` (compressed bytes at `spans`) decoded back to back at `dst_ptr`."""
        dtype = _require_integer_dtype(self.dtype)
        codec = _codec_for(self.config)
        with codec.stage_lock:
            buf, offs = self._stage_compressed(codec, spans)
            rows = self._rows_of(chunk_ids)
            status = codec.decompress_ptr(buf.ptr, 0, offs, rows, self.n_channels, dtype.itemsize,
                                          _native._fl(self._flags(), dtype), dst_ptr, int(dst_is_device))
        self._raise_if_corrupt(status, chunk_ids)
        return rows

    def _decode_block(self, chunk_ids, spans):
        """Decode several chunks in one GPU call -> (fresh host array of all their rows, row offsets)."""
        rows = self._rows_of(chunk_ids)
        out = np.empty((int(rows[-1]), self.n_channels), dtype=self.dtype)
        self._decode_into(chunk_ids, spans, out.ctypes.data, False)
        return out, rows

    def _decode(self, chunk_ids, spans):
        """Decode several chunks in one GPU call -> list of per-chunk arrays (views of one block)."""
        out, rows = self._decode_block(chunk_ids, spans)
        return [out[rows[k]:rows[k + 1]] for k in range(len(chunk_ids))]

    def _span(self, idx):
        return self.chunk_offsets[idx], self.chunk_offsets[idx + 1] - self.chunk_offsets[idx]

    def _device_chunks(self, first, last):
        """Make chunks first..last resident in device memory (decoding the missing ones, a run of consecutive misses
        per GPU call) and yield (chunk_idx, device pointer of its first row)."""
        codec = _codec_for(self.config)
        row_bytes = self.n_channels * self.dtype.itemsize
        idx = first
        while idx <= last:
            e = self._dev_cache.get(idx)
            if e is not None:
                yield idx, e[0].ptr + e[1], e
                idx += 1
                continue
            hi = idx + 1
            while hi <= last and hi - idx < GPU_BATCH_CHUNKS and self._dev_cache.entries.get(hi) is None and \
                    (self.chunk_bounds[hi + 1] - self.chunk_bounds[idx]) * row_bytes <= GPU_BATCH_BYTES:
                hi += 1
            ids = list(range(idx, hi))
            block = _DeviceBlock(codec, (self.chunk_bounds[hi] - self.chunk_bounds[idx]) * row_bytes + 256)
            rows = self._decode_into(ids, [self._span(i) for i in ids], block.ptr, True)
            for k, i in enumerate(ids):
                e = (block, int(rows[k]) * row_bytes, int(rows[k + 1] - rows[k]) * row_bytes)
                self._dev_cache.put(i, e)
                yield i, block.ptr + e[1], e
            idx = hi

    def _read_rows(self, i0, i1):
        """Rows [i0, i1) as a fresh C-contiguous host array: the chunks they touch are decoded into (or found in) the
        device-side cache and only the rows asked for cross the bus."""
        codec = _codec_for(self.config)
        row_bytes = self.n_channels * self.dtype.itemsize
        out = np.empty((i1 - i0, self.n_channels), dtype=self.dtype)
        first, last = self._chunks_for_interval(i0, i1)
        # consecutive chunks of one device block are fetched with a single copy
        run_ptr = run_dst = run_len = None
        keep = []                                     # the blocks stay alive until their rows have been copied
        for idx, ptr, entry in self._device_chunks(first, last):
            keep.append(entry)
            c0, c1 = self.chunk_bounds[idx], self.chunk_bounds[idx + 1]
            a, b = max(i0, c0), min(i1, c1)
            if b <= a:
                continue
            src, dst, n = ptr + (a - c0) * row_bytes, (a - i0) * row_bytes, (b - a) * row_bytes
            if run_ptr is not None and run_ptr + run_len == src and run_dst + run_len == dst:
                run_len += n
                continue
            if run_ptr is not None:
                codec.memcpy(out.ctypes.data + run_dst, run_ptr, run_len, 2)
            run_ptr, run_dst, run_len = src, dst, n
        if run_ptr is not None:
            codec.memcpy(out.ctypes.data + run_dst, run_ptr, run_len, 2)
        return out

    def read_chunk(self, chunk_idx, chunk_start, chunk_length):
        """Read + decode one chunk -> C-contiguous (n_samples_chunk, n_channels) (reference mtscomp.py:602-635)."""
        logger.debug("Reading compressed chunk %d, %d, %d", chunk_idx, chunk_start, chunk_length)
        chunk = self._decode([chunk_idx], [(chunk_start, chunk_length)])[0]
        i0, i1 = self.chunk_bounds[chunk_idx:chunk_idx + 2]
        assert chunk.shape == (i1 - i0, self.n_channels) and chunk.dtype == self.dtype
        return np.ascontiguousarray(chunk)

    def _decompress_chunk(self, chunk_idx):
        assert 0 <= chunk_idx <= self.n_chunks - 1
        start = self.chunk_offsets[chunk_idx]
        return chunk_idx, self.read_chunk(chunk_idx, start, self.chunk_offsets[chunk_idx + 1] - start)

    def decompress_chunks(self, chunk_ids, pool=None):
        """{chunk_idx: array} for `chunk_ids` (reference mtscomp.py:645-650), as one batched GPU call."""
        ids = list(chunk_ids)
        spans = [(self.chunk_offsets[i], self.chunk_offsets[i + 1] - self.chunk_offsets[i]) for i in ids]
        for i in ids:
            assert 0 <= i <= self.n_chunks - 1
        out = dict(zip(ids, self._decode(ids, spans))) if ids else {}
        assert set(out.keys()) == set(ids)
        return out

    def start_thread_pool(self):
        if not self.pool:
            self.pool = _SerialPool()
        return self.pool

    def stop_thread_pool(self):
        self.pool = None

    # -- indexing ---------------------------------------------------------------------------------------------------
    def _validate_index(self, i, value_for_none=0):
        if i is None:
            i = value_for_none
        elif i < 0:
            i += self.n_samples
        return int(clip(i, 0, self.n_samples))

    def _chunks_for_interval(self, i0, i1):
        """First and last chunk needed for samples [i0, i1] (reference mtscomp.py:661-684, pinned by its tests)."""
        i0 = clip(i0, 0, self.n_samples - 1)
        i1 = clip(i1, i0, self.n_samples - 1)
        first = clip(bisect.bisect_right(self.chunk_bounds, i0) - 1, 0, self.n_chunks - 1)
        last = clip(bisect.bisect_right(self.chunk_bounds, i1, lo=first) - 1, 0, self.n_chunks - 1)
        assert self.chunk_bounds[first] <= i0 < self.chunk_bounds[first + 1]
        assert self.chunk_bounds[last] <= i1 <= self.chunk_bounds[last + 1]
        assert 0 <= first <= last <= self.n_chunks - 1
        return first, last

    def __getitem__(self, item):
        """NumPy-style slicing returning in-memory arrays (reference mtscomp.py:798-856)."""
        empty = np.zeros((0, self.n_channels), dtype=self.dtype)
        if isinstance(item, slice):
            i0 = self._validate_index(item.start, 0)
            i1 = self._validate_index(item.stop, self.n_samples)
            if i1 <= i0:
                return empty
            # the chunks the slice touches are decoded into (or found in) the device-side LRU and only rows i0..i1
            # are copied to the host (the reference decodes and concatenates whole chunks, mtscomp.py:810-856)
            arr = self._read_rows(i0, i1)
            out = arr[::item.step, :] if item.step not in (None, 1) else arr
            assert out.shape[0] == len(range(i0, i1, item.step or 1))
            return out
        if isinstance(item, tuple):
            if len(item) == 1:
                return self[item[0]]
            if len(item) == 2 and np.isscalar(item[0]):
                return self[item[0]][item[1]]
            if len(item) == 2:
                return self[item[0]][:, item[1]]
        elif isinstance(item, (int, np.integer)):
            item = int(item)
            if item < 0:
                item += self.n_samples * -int(np.floor(item / self.n_samples))
                assert 0 <= item < self.n_samples
            if not 0 <= item < self.n_samples:  # pragma: no cover
                raise IndexError(
                    "index %d is out of bounds for axis 0 with size %d" % (item, self.n_samples))
            return self[item:item + 1][0]
        elif isinstance(item, (list, np.ndarray)):  # pragma: no cover
            raise NotImplementedError("Indexing with multiple values is currently unsupported.")
        return empty  # pragma: no cover

    # -- whole-file operations --------------------------------------------------------------------------------------
    def tofile(self, out, overwrite=False):
        """Write the decompressed array to `out` (reference mtscomp.py:701-743)."""
        if out is None:
            out = Path(self.cdata.name).with_suffix('.bin')
        out = Path(out)
        if not overwrite and out.exists():  # pragma: no cover
            raise ValueError(
                "The output file %s already exists, use --overwrite or specify another output path." % out)
        elif overwrite and out.exists():
            out.unlink()
        dtype = _require_integer_dtype(self.dtype)
        codec = _codec_for(self.config)
        row_bytes = self.n_channels * dtype.itemsize
        flags = _native._fl(self._flags(), dtype)
        b = self.chunk_bounds
        ranges = list(_batch_ranges(b, row_bytes, 0, self.n_chunks))

        def stage(k, slot):
            lo, hi = ranges[k]
            return self._stage_compressed(codec, [self._span(i) for i in range(lo, hi)], 'w_comp%d' % slot)

        def run(k, slot, staged):
            (cbuf, offs), (lo, hi) = staged, ranges[k]
            status = codec.decompress_ptr(cbuf.ptr, 0, offs, self._rows_of(range(lo, hi)), self.n_channels,
                                          dtype.itemsize, flags, bufs[slot].ptr, 0)
            self._raise_if_corrupt(status, list(range(lo, hi)))

        def finish(k, slot, _):
            lo, hi = ranges[k]
            pos, n, src = b[lo] * row_bytes, (b[hi] - b[lo]) * row_bytes, bufs[slot].array
            step = max(-(-n // 8), 1 << 20)
            return [partial(np.copyto, mm[pos + a:pos + min(a + step, n)], src[a:min(a + step, n)])
                    for a in range(0, n, step)]

        # two pinned output buffers: the GPU decodes batch k+1 into one while eight lanes copy batch k from the other
        # into a shared mapping of the output file.  (write() and pwrite() serialise on the file's write lock and run
        # at the speed of one page-cache copy — 3.5 GB/s on the bench box's tmpfs, four pwrite threads 4.3, four
        # mapping threads 5.6, eight 6.8 (tools/file_write_probe.py);
        # stores through a mapping only take per-page locks.  As with write(), nothing is fsync'ed.)
        total = b[-1] * row_bytes
        with codec.stage_lock, open(out, 'w+b') as fb:
            fb.truncate(total)
            mm = np.memmap(fb, dtype=np.uint8, mode='r+', shape=(total,)) if total else None
            n_max = max((b[hi] - b[lo]) * row_bytes for lo, hi in ranges)
            bufs = [codec.host_buffer('r_out%d' % i, n_max) for i in (0, 1)]
            _pipeline(len(ranges), stage, run, finish, 8, 'Decompressing', self.quiet)
            del mm
        logger.info("Wrote %s (%.1f GB).", out, total / 1024 ** 3)
        if self.check_after_decompress:
            decompressed = load_raw_data(out, n_channels=self.n_channels, dtype=self.dtype)
            check(decompressed, self.cdata, self.cmeta)
            logger.debug("Automatic integrity check after decompression PASSED.")

    def close(self):
        if getattr(self, '_dev_cache', None) is not None:
            self._dev_cache.clear()
        if self.cdata:
            self.cdata.close()

    def chop(self, n_chunks, out=None):
        """Copy the first `n_chunks` compressed chunks into a new .cbin/.ch pair (reference mtscomp.py:750-796)."""
        assert n_chunks > 0
        if n_chunks >= self.n_chunks:  # pragma: no cover
            logger.warning("Cannot chop more chunks than there are in the original file.")
            return
        assert out is not None, "The output path must be specified."
        out = Path(out)
        assert out.suffix == '.cbin'
        if out.exists():  # pragma: no cover
            raise IOError("File %s already exists." % out)
        out.parent.mkdir(exist_ok=True, parents=True)
        end = self.chunk_offsets[n_chunks]
        with open(out, 'wb') as f:
            for i in tqdm(range(n_chunks), desc='Chopping %d chunks' % n_chunks):
                start = self.chunk_offsets[i]
                f.write(self._pread(self.chunk_offsets[i + 1] - start, start))
            assert f.tell() == end
        outmeta = out.with_suffix('.ch')
        if outmeta.exists():  # pragma: no cover
            raise IOError("File %s already exists." % out)
        cmeta = Bunch(self.cmeta.copy())
        cmeta['chunk_bounds'] = cmeta['chunk_bounds'][:n_chunks + 1]
        cmeta['chunk_offsets'] = cmeta['chunk_offsets'][:n_chunks + 1]
        cmeta['sha1_compressed'] = None
        cmeta['sha1_uncompressed'] = None
        cmeta['chopped'] = True
        with open(outmeta, 'w') as f:
            json.dump(cmeta, f, indent=2, sort_keys=True)

    def __del__(self):
        try:
            self.close()
        except Exception:  # pragma: no cover
            pass


# ------------------------------------------------------------------------------------------------------------------
# High-level API
# ------------------------------------------------------------------------------------------------------------------

def _copy_rows(dst, src):
    """dst[...] = src (same shape) with a few threads: np.copyto releases the GIL, and the source is usually a memory
    map whose pages fault in as they are read."""
    n = src.shape[0]
    step = max(-(-n // 4), 1)
    if src.nbytes < (4 << 20):
        np.copyto(dst, src)
        return
    list(_read_pool().map(lambda a: np.copyto(dst[a:a + step], src[a:a + step]), range(0, n, step)))


def _verify_range(reader, data, first, last):
    """Check chunks [first, last) of the open `reader` against the rows of `data` on the GPU (mtsb_verify_chunks):
    batches of _batch_ranges, whose compressed bytes and source rows are staged into pinned memory for batch k+1 while
    the GPU verifies batch k.  Integers must be equal, floats np.isclose(rtol=CHECK_RTOL, atol=CHECK_ATOL).  Raises
    IOError for a corrupt chunk or AssertionError for a mismatching one, whichever comes first in chunk order."""
    dtype = _require_integer_dtype(reader.dtype)
    codec = _codec_for(reader.config)
    nc, b = reader.n_channels, reader.chunk_bounds
    row_bytes = nc * dtype.itemsize
    flags = _native._fl(reader._flags(), dtype)
    ranges = list(_batch_ranges(b, row_bytes, first, last))

    def stage(k, slot):
        # the Writer's staging buffers: pinned already when the check follows a write
        lo, hi = ranges[k]
        cbuf, offs = reader._stage_compressed(codec, [reader._span(i) for i in range(lo, hi)], 'w_comp%d' % slot)
        n = (b[hi] - b[lo]) * row_bytes
        rbuf = codec.host_buffer('w_raw%d' % slot, n)
        _copy_rows(rbuf.array[:n].view(dtype).reshape(-1, nc), data[b[lo]:b[hi]])
        return cbuf, offs, rbuf

    def run(k, slot, staged):
        (lo, hi), (cbuf, offs, rbuf) = ranges[k], staged
        status, mism, at = codec.verify_ptr(cbuf.ptr, 0, offs, reader._rows_of(range(lo, hi)), nc, dtype.itemsize,
                                            flags, rbuf.ptr, 0, CHECK_RTOL, CHECK_ATOL)
        bad = np.flatnonzero((status != 0) | (mism != 0))
        if len(bad):
            i = int(bad[0])
            if status[i]:
                raise IOError("Compressed chunk #%d is corrupted." % (lo + i))
            raise AssertionError(_mismatch_message(reader, data, lo + i, int(mism[i]), int(at[i])))

    with codec.stage_lock:
        _pipeline(len(ranges), stage, run, desc='Checking')


def _mismatch_message(reader, data, idx, n_bad, at):
    row, ch = divmod(at, reader.n_channels)
    sample = reader.chunk_bounds[idx] + row
    got = reader._decode([idx], [reader._span(idx)])[0][row, ch]
    return ("chunk #%d does not match the data in %d element(s); the first is row %d (sample %d), channel %d: "
            "decoded %r, expected %r" % (idx, n_bad, row, sample, ch, got.item(), data[sample, ch].item()))


def check(data, out, outmeta):
    """Decode every chunk and compare it with `data` on the GPU (reference mtscomp.py:866-888): IOError for a corrupt
    chunk, AssertionError for a mismatch, whichever chunk comes first."""
    unc = decompress(out, outmeta)
    try:
        dtype = _require_integer_dtype(unc.dtype)
        assert tuple(data.shape) == tuple(unc.shape) and data.dtype == dtype
        _verify_range(unc, data, 0, unc.n_chunks)
    finally:
        unc.close()


def compress(path, out=None, outmeta=None, sample_rate=None, n_channels=None, dtype=None, **kwargs):
    """Compress a raw binary file into `out` (.cbin) + `outmeta` (.ch); returns compressed/raw size ratio
    (reference mtscomp.py:891-958)."""
    w = Writer(**kwargs)
    w.open(path, sample_rate=sample_rate, n_channels=n_channels, dtype=dtype)
    ratio = w.write(out, outmeta)
    w.close()
    return ratio


def _recompress_batches(r, fb, ranges, flags, write_index, quiet):
    """Recompress the open Reader `r` batch by batch into the file `fb` -> (chunk_offsets, SHA-1 of the written bytes).
    While the GPU recompresses batch k, a worker stages batch k+1's .cbin bytes into pinned memory and another writes
    and hashes batch k-1's output."""
    codec = _codec_for(r.config)
    nc, b, isz = r.n_channels, r.chunk_bounds, r.dtype.itemsize
    sha1 = hashlib.sha1()
    offsets = [0]

    def stage(k, slot):
        lo, hi = ranges[k]
        return r._stage_compressed(codec, [r._span(i) for i in range(lo, hi)], 'rc_in%d' % slot)

    def run(k, slot, staged):
        (lo, hi), (cbuf, coffs) = ranges[k], staged
        offs, status = codec.recompress_ptr(cbuf.ptr, 0, coffs, r._rows_of(range(lo, hi)), nc, isz, flags,
                                            out_bufs[slot].ptr, 0, caps[k])
        r._raise_if_corrupt(status, list(range(lo, hi)))
        return offs

    def write_and_hash(comp):
        fb.write(comp)
        sha1.update(comp)

    def finish(k, slot, offs):
        base = offsets[-1]
        offsets.extend(int(base + o) for o in offs[1:])
        return partial(write_and_hash, out_bufs[slot].array[:int(offs[-1])]),

    with codec.stage_lock, _codec_param(codec, 'write_index', write_index):
        # (the bound depends on write_index: computed with it set)
        caps = [sum(codec.compress_bound(b[i + 1] - b[i], nc, isz, flags) for i in range(lo, hi)) for lo, hi in ranges]
        out_bufs = [codec.host_buffer('rc_out%d' % i, max(caps)) for i in (0, 1)]
        _pipeline(len(ranges), stage, run, finish, 1, 'Recompressing', quiet)
    return offsets, sha1


def _check_recompressed(src, new, ranges, quiet):
    """Both Readers' chunks decode to the same bits: each batch of `src` is decoded into device memory and `new`'s
    chunks are verified against it (mtsb_verify_chunks, reference on the device).  Both calls use the integer flags
    of the element width: the modular inverse transform is a bijection, so equal integer decodes mean equal inflated
    bytes, which makes the check exact for floats too (NaN payloads included)."""
    codec = _codec_for(src.config)
    nc, b, isz = src.n_channels, src.chunk_bounds, src.dtype.itemsize
    row_bytes = nc * isz
    flags = src._flags()                          # no MTSB_FLOAT
    block = _DeviceBlock(codec, max((b[hi] - b[lo]) * row_bytes for lo, hi in ranges) + 256)

    def stage(k, slot):
        lo, hi = ranges[k]
        ids = range(lo, hi)
        return (src._stage_compressed(codec, [src._span(i) for i in ids], 'rc_in%d' % slot),
                new._stage_compressed(codec, [new._span(i) for i in ids], 'rc_chk%d' % slot))

    def run(k, slot, staged):
        ids, ((sbuf, soffs), (nbuf, noffs)) = list(range(*ranges[k])), staged
        rows = src._rows_of(ids)
        src._raise_if_corrupt(codec.decompress_ptr(sbuf.ptr, 0, soffs, rows, nc, isz, flags, block.ptr, 1), ids)
        status, mism, _ = codec.verify_ptr(nbuf.ptr, 0, noffs, rows, nc, isz, flags, block.ptr, 1, 0., 0.)
        bad = np.flatnonzero((status != 0) | (mism != 0))
        if len(bad):
            raise RuntimeError("recompressed chunk #%d does not decode to what the source chunk decodes to"
                               % ids[int(bad[0])])

    with codec.stage_lock:
        _pipeline(len(ranges), stage, run, desc='Checking', quiet=quiet)


def recompress(cdata, cmeta=None, out=None, outmeta=None, write_index=True, overwrite=False, quiet=False, **kwargs):
    """Re-encode a compressed dataset on the GPU into `out` (.cbin) + `outmeta` (.ch, default: next to `out`), with
    (write_index=True) or without the in-band segment index; returns compressed/raw size ratio.

    Every chunk's zlib stream is inflated to its transformed bytes and deflated again; the samples are never
    reconstructed, so the new file decodes to exactly what the source decodes to, for floats too.  The .ch keeps every
    key of the source's but `chunk_offsets` and `sha1_compressed`.  Unless check_after_compress is off, every new chunk
    is then checked against its source chunk on the GPU.  On failure the new .cbin is removed and no .ch is written."""
    if out is None:
        raise ValueError("The output path must be specified.")
    out = Path(out)
    outmeta = Path(outmeta) if outmeta else out.with_suffix('.ch')
    r = Reader(quiet=quiet, **kwargs)
    r.open(cdata, cmeta)
    try:
        src_cbin = Path(r.cdata.name)
        src_ch = Path(cmeta) if isinstance(cmeta, (str, Path)) else src_cbin.with_suffix('.ch')
        for p, s in ((out, src_cbin), (outmeta, src_ch)):
            if p.resolve() == s.resolve() or (p.exists() and s.exists() and op.samefile(p, s)):
                raise ValueError("Cannot recompress %s in place: %s is a source file." % (src_cbin, p))
        for p in (out, outmeta):
            if p.exists() and not overwrite:
                raise ValueError(
                    "The output file %s already exists, use --overwrite or specify another output path." % p)
        dtype = _require_integer_dtype(r.dtype)
        flags = _native._fl(r._flags(), dtype)
        ranges = list(_batch_ranges(r.chunk_bounds, r.n_channels * dtype.itemsize, 0, r.n_chunks))
        for p in (out, outmeta):
            if p.exists():
                p.unlink()
        out.parent.mkdir(exist_ok=True, parents=True)
        try:
            with open(out, 'wb') as fb:
                offsets, sha1 = _recompress_batches(r, fb, ranges, flags, write_index, quiet)
                csize = fb.tell()
            assert offsets[-1] == csize
            meta = dict(r.cmeta)
            meta['chunk_offsets'] = offsets
            meta['sha1_compressed'] = sha1.hexdigest()
            if r.config.check_after_compress:
                new = Reader(quiet=quiet, **kwargs)
                new.open(out, meta)
                try:
                    _check_recompressed(r, new, ranges, quiet)
                finally:
                    new.close()
                logger.debug("Automatic integrity check after recompression PASSED.")
        except BaseException:
            if out.exists():
                out.unlink()
            raise
        with open(outmeta, 'w') as f:
            json.dump(meta, f, indent=2, sort_keys=True)
        ratio = csize / (r.n_samples * r.n_channels * dtype.itemsize)
        logger.info("Wrote %s (%.1f GB, -%.3f%%).", out, csize / 1024 ** 3, 100 - 100 * ratio)
        return ratio
    finally:
        r.close()


def decompress(cdata, cmeta=None, out=None, write_output=False, overwrite=False, **kwargs):
    """Open a compressed dataset, optionally writing the decompressed file; returns the Reader
    (reference mtscomp.py:961-997)."""
    if out:
        write_output = True
    r = Reader(**kwargs)
    r.open(cdata, cmeta)
    if write_output:
        r.tofile(out, overwrite=overwrite)
    return r
