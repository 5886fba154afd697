# -*- coding: utf-8 -*-
"""Chunk-range sharding across GPUs (SURVEY §8e): contiguous ranges per rank, host-side gather of compressed sizes.

Chunks are independent zlib streams, so there is no collective on the data path.  The only cross-rank datum is the
per-chunk compressed size, gathered as Python objects over whatever process group exists (gloo on CPU, nccl ranks use
the default group's object collectives) and prefix-summed into the reference's `chunk_offsets` (mtscomp.py:453-480).
"""

import hashlib
import json
import os
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

import numpy as np


def shard_range(n_chunks, rank, world):
    """Chunks [first, last) of rank `rank`: contiguous, in file order, sizes differ by at most ceil/floor."""
    per = -(-n_chunks // world)
    return min(rank * per, n_chunks), min((rank + 1) * per, n_chunks)


def assemble_offsets(sizes_by_rank):
    """sizes_by_rank: list (rank order) of per-chunk compressed sizes -> global chunk_offsets (n_chunks + 1)."""
    sizes = [int(s) for part in sizes_by_rank for s in part]
    return [0] + np.cumsum(sizes, dtype=np.int64).tolist() if sizes else [0]


def rank_base_offsets(sizes_by_rank):
    """Byte offset in the .cbin at which each rank's packed output starts."""
    totals = [int(np.sum(p, dtype=np.int64)) if len(p) else 0 for p in sizes_by_rank]
    return [0] + np.cumsum(totals, dtype=np.int64).tolist()[:-1]


def gather_sizes(local_sizes, group=None):
    """All ranks get every rank's per-chunk sizes (torch.distributed object all-gather; works on gloo and nccl)."""
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()):
        return [list(map(int, local_sizes))]
    out = [None] * dist.get_world_size(group)
    dist.all_gather_object(out, list(map(int, local_sizes)), group=group)
    return out


def compress_sharded(codec, data, chunk_bounds, flags, rank, world, group=None):
    """Compress this rank's chunk range of `data` (rows chunk_bounds[first]..chunk_bounds[last]) and return
    (packed bytes of this rank, global chunk_offsets, byte offset of this rank's part in the .cbin)."""
    first, last = shard_range(len(chunk_bounds) - 1, rank, world)
    if last > first:
        b0 = chunk_bounds[first]
        rows = np.asarray(chunk_bounds[first:last + 1], dtype=np.int64) - b0
        comp, offs = codec.compress(data[b0:chunk_bounds[last]], rows, flags)
        sizes = np.diff(offs).tolist()
    else:
        comp, sizes = np.zeros(0, np.uint8), []
    all_sizes = gather_sizes(sizes, group)
    return comp, assemble_offsets(all_sizes), rank_base_offsets(all_sizes)[rank] if world > 1 else 0


def gather_objects(obj, group=None):
    """Every rank's `obj`, in rank order, on all ranks (one object all-gather; [obj] without a process group)."""
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()):
        return [obj]
    out = [None] * dist.get_world_size(group)
    dist.all_gather_object(out, obj, group=group)
    return out


def _barrier(group=None):
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized():
        dist.barrier(group=group)


def write_sharded(data_path, out, outmeta, rank, world, sample_rate=None, n_channels=None, dtype=None, group=None,
                  hash_raw=True, check_after_compress=False, before_check=None, **config):
    """ONE `.cbin` + `.ch` written by `world` ranks (one GPU each): every rank memory-maps the raw file, compresses its
    contiguous chunk range (shard_range) on its GPU, the per-chunk sizes are gathered on the host, and each rank writes
    its packed streams at its base offset with pwrite (reference mtscomp.py:453-486 builds the same offset table
    sequentially).  Rank 0 computes the two SHA-1 digests the format records — they are sequential passes over the raw
    and the compressed file — and writes the `.ch`.  Returns (chunk_offsets, seconds spent compressing on this rank).
    The rank's range goes through the Writer's own batching, on the rank's `_native.Codec`.

    check_after_compress (off by default here): once the file is complete, each rank calls `before_check(writer)` and
    verifies its own chunk range of the written .cbin against its memory map on its GPU.  The verdicts are gathered, so
    that every rank raises the same error when any rank's check failed: the CRITICAL ERROR RuntimeError of
    Writer.write for a mismatch, IOError for a corrupt chunk (the first failure in chunk order decides)."""
    import time
    from .core import Writer, _require_integer_dtype
    w = Writer(quiet=True, check_after_compress=check_after_compress, before_check=before_check, **config)
    w.open(data_path, sample_rate=sample_rate, n_channels=n_channels, dtype=dtype)
    nc, isz = w.n_channels, _require_integer_dtype(w.dtype).itemsize
    first, last = shard_range(w.n_chunks, rank, world)
    raw_sha = None
    pool = ThreadPoolExecutor(1)
    if rank == 0 and hash_raw:
        def _hash_all():
            h = hashlib.sha1()
            step = max(1, (64 << 20) // max(nc * isz, 1))
            for r0 in range(0, w.n_samples, step):
                h.update(np.ascontiguousarray(w.data[r0:r0 + step]))
            return h.hexdigest()
        raw_sha = pool.submit(_hash_all)
    parts, sizes = [], []

    def finish(raw, offs, comp):
        sizes.extend(np.diff(offs).tolist())
        return (lambda: parts.append(comp.copy()),)

    t0 = time.perf_counter()
    if last > first:
        w._compress_range(first, last, finish, 1)
    secs = time.perf_counter() - t0
    all_sizes = gather_sizes(sizes, group)
    offsets = assemble_offsets(all_sizes)
    base = rank_base_offsets(all_sizes)[rank] if world > 1 else 0
    out, outmeta = Path(out), Path(outmeta)
    if rank == 0:
        out.parent.mkdir(exist_ok=True, parents=True)
        with open(out, 'wb') as f:
            f.truncate(offsets[-1])
    _barrier(group)
    fd = os.open(out, os.O_WRONLY)
    try:
        pos = base
        for p in parts:
            mv, done = memoryview(p), 0
            while done < len(mv):
                done += os.pwrite(fd, mv[done:], pos + done)
            pos += len(mv)
    finally:
        os.close(fd)
    _barrier(group)
    if rank == 0:
        h = hashlib.sha1()
        with open(out, 'rb') as f:
            for blk in iter(lambda: f.read(64 << 20), b''):
                h.update(blk)
        w.chunk_offsets = offsets
        meta = w.get_cmeta()
        meta['sha1_compressed'] = h.hexdigest()
        meta['sha1_uncompressed'] = raw_sha.result() if raw_sha is not None else None   # (None: as after a chop)
        with open(outmeta, 'w') as f:
            json.dump(meta, f, indent=2, sort_keys=True)
    pool.shutdown()
    _barrier(group)
    if check_after_compress:
        _check_shard(w, out, outmeta, first, last, group)
    w.close()
    return offsets, secs


def _check_shard(w, out, outmeta, first, last, group=None):
    """The post-write check of write_sharded on chunks [first, last): every rank takes part in the gather whatever its
    own check did, so no rank waits in a collective for a rank that raised."""
    from .core import CRITICAL_CHECK_FAILED, Reader, _verify_range
    verdict = None
    try:
        w.before_check(w)
        r = Reader(quiet=True, device=w.config.get('device', None))
        r.open(out, outmeta)
        try:
            _verify_range(r, w.data, first, last)
        finally:
            r.close()
    except AssertionError as e:
        verdict = ('mismatch', str(e))
    except IOError as e:
        verdict = ('corrupt', str(e))
    except Exception as e:
        verdict = ('error', '%s: %s' % (type(e).__name__, e))
    failed = [v for v in gather_objects(verdict, group) if v is not None]
    if not failed:
        return
    kind, msg = failed[0]
    if kind == 'mismatch':
        raise RuntimeError(CRITICAL_CHECK_FAILED + " (" + msg + ")")
    if kind == 'corrupt':
        raise IOError(msg)
    raise RuntimeError("the check after a sharded write failed on a rank: " + msg)
