"""CPU, world_size 2 over gloo: the multi-GPU host logic — contiguous chunk ranges, size gather, offset assembly.
compress_sharded's per-chunk codec is stood in for by the oracle; write_sharded runs the host emulation of the kernels."""
import os
import socket

import numpy as np
import pytest

from mtscomp_b200 import sharding


def test_shard_range_partitions():
    for n in (0, 1, 2, 7, 60, 600, 3600):
        for world in (1, 2, 3, 4, 8):
            rs = [sharding.shard_range(n, r, world) for r in range(world)]
            assert rs[0][0] == 0 and rs[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(rs, rs[1:]))
            assert all(0 <= a <= b for a, b in rs)
    assert sharding.shard_range(3600, 3, 8) == (1350, 1800)


class _OracleCodec:
    def compress(self, data, rows, flags):
        from oracle import codec as ora
        parts = [ora.encode_chunk(data[rows[i]:rows[i + 1]]) for i in range(len(rows) - 1)]
        offs = np.concatenate(([0], np.cumsum([len(p) for p in parts]))).astype(np.int64)
        return np.frombuffer(b''.join(parts), np.uint8), offs


def _worker(rank, world, port, tmp):
    import torch.distributed as dist
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    dist.init_process_group('gloo', rank=rank, world_size=world)
    rng = np.random.default_rng(0)
    data = np.cumsum(rng.integers(-9, 10, (7000, 12)), axis=0).astype(np.int16)
    bounds = list(range(0, 7000, 1000)) + [7000]
    comp, offsets, base = sharding.compress_sharded(_OracleCodec(), data, bounds, 1, rank, world)
    np.save(os.path.join(tmp, 'comp%d.npy' % rank), comp)
    if rank == 0:
        np.save(os.path.join(tmp, 'offsets.npy'), np.asarray(offsets))
    np.save(os.path.join(tmp, 'base%d.npy' % rank), np.asarray([base]))
    dist.barrier()
    dist.destroy_process_group()


def test_two_ranks_reassemble_the_sequential_file(tmp_path):
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    port = s.getsockname()[1]
    s.close()
    mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    rng = np.random.default_rng(0)
    data = np.cumsum(rng.integers(-9, 10, (7000, 12)), axis=0).astype(np.int16)
    bounds = list(range(0, 7000, 1000)) + [7000]
    want, woffs = _OracleCodec().compress(data, np.asarray(bounds), 1)
    parts = [np.load(tmp_path / ('comp%d.npy' % r)) for r in range(2)]
    bases = [int(np.load(tmp_path / ('base%d.npy' % r))[0]) for r in range(2)]
    offsets = np.load(tmp_path / 'offsets.npy')
    assert offsets.tolist() == woffs.tolist()
    assert bases == [0, len(parts[0])]
    assert np.array_equal(np.concatenate(parts), want)


def _file_worker(rank, world, port, tmp, emu_lib):
    import torch.distributed as dist
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    dist.init_process_group('gloo', rank=rank, world_size=world)
    import mtscomp_b200 as M
    from mtscomp_b200 import _native
    M.CONFIG_PATH = os.path.join(tmp, '.mtscomp')
    _native._default[0] = _native.Codec(0, lib=_native.load_library(emu_lib))   # the emulated kernels as the rank's codec
    sharding.write_sharded(os.path.join(tmp, 'data.bin'), os.path.join(tmp, 'data.cbin'), os.path.join(tmp, 'data.ch'),
                           rank, world, sample_rate=1000., n_channels=12, dtype=np.int16)
    dist.destroy_process_group()


def test_two_ranks_write_one_file_through_the_writer(tmp_path):
    """write_sharded at world size 2 (offsets, pwrite at the rank bases, digests, .ch), each rank compressing through
    the Writer's batches on the host emulation of the kernels, gives a file for which the reference's own Reader
    semantics hold (zlib per chunk, SHA-1s)."""
    import hashlib
    import json
    import zlib
    import torch.multiprocessing as mp
    from mtscomp_b200 import build
    from oracle import codec as ora
    emu_lib = str(build.build_emulation())     # once here, not by both ranks at the same time
    rng = np.random.default_rng(3)
    data = np.cumsum(rng.integers(-9, 10, (7300, 12)), axis=0).astype(np.int16)
    data.tofile(tmp_path / 'data.bin')
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    port = s.getsockname()[1]
    s.close()
    mp.spawn(_file_worker, args=(2, port, str(tmp_path), emu_lib), nprocs=2, join=True)
    meta = json.loads((tmp_path / 'data.ch').read_text())
    blob = (tmp_path / 'data.cbin').read_bytes()
    b, o = meta['chunk_bounds'], meta['chunk_offsets']
    assert b == list(range(0, 7300, 1000)) + [7300] and o[-1] == len(blob)
    assert meta['sha1_compressed'] == hashlib.sha1(blob).hexdigest()
    assert meta['sha1_uncompressed'] == hashlib.sha1(data.tobytes()).hexdigest()
    for i in range(len(b) - 1):
        assert zlib.decompress(blob[o[i]:o[i + 1]]) == ora.transform_chunk(data[b[i]:b[i + 1]])
