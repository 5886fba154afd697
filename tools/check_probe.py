"""What the integrity check costs: check() on the GPU against the host compare it replaced, and the device-resident
verify rate.  Prints one JSON line (with the card's name and power limit).

Files: 128 one-second AP chunks (385 x int16, synth.ap_chunk), and the same chunks as float32 (/ 7.3 + 20000, as
case_float_dtypes writes them: the offset makes the reference's np.allclose pass), written with the default writer
and checked against their memory maps with the page cache warm.  `host_check` is the previous check() body, verbatim:
decode each batch to pinned memory and compare on one CPU thread.  The two alternate, three runs each.

Device-resident: 600 AP chunks (8 distinct ones tiled) with the compressed bytes and the reference rows in HBM;
GB/s of raw bytes and the compare stage's ms (mtsb_last_timings slot 6).

    python tools/check_probe.py [--chunks 128] [--reps 3] [--dev-chunks 600] [--dir /dev/shm]
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
import mtscomp_b200 as M                                                       # noqa: E402
from mtscomp_b200 import _native, synth                                        # noqa: E402
from mtscomp_b200.config import CHECK_ATOL                                     # noqa: E402
from mtscomp_b200.core import (_batch_ranges, _codec_for, _require_integer_dtype, decompress,  # noqa: E402
                               CHECK_RTOL)
from tqdm import tqdm                                                          # noqa: E402

NS, NC = 30000, 385


def host_check(data, out, outmeta):
    """Decode every chunk and compare with `data` (reference mtscomp.py:866-888); AssertionError on mismatch."""
    unc = decompress(out, outmeta)
    try:
        dtype = _require_integer_dtype(unc.dtype)
        codec = _codec_for(unc.config)
        row_bytes = unc.n_channels * dtype.itemsize
        assert tuple(data.shape) == tuple(unc.shape) and data.dtype == dtype
        with codec.stage_lock:
            for lo, hi in tqdm(list(_batch_ranges(unc.chunk_bounds, row_bytes, 0, unc.n_chunks)), desc='Checking'):
                ids = list(range(lo, hi))
                buf = codec.host_buffer('r_out0', (unc.chunk_bounds[hi] - unc.chunk_bounds[lo]) * row_bytes)
                rows = unc._decode_into(ids, [unc._span(i) for i in ids], buf.ptr, False)
                got = buf.array[:int(rows[-1]) * row_bytes].view(dtype).reshape(-1, unc.n_channels)
                expected = data[unc.chunk_bounds[lo]:unc.chunk_bounds[hi]]
                assert got.shape == expected.shape
                if np.issubdtype(dtype, np.integer):
                    assert np.array_equal(got, expected)
                else:
                    assert np.allclose(got, expected, atol=CHECK_ATOL)
    finally:
        unc.close()


def card():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=60).stdout.strip()
        name, power = [s.strip() for s in q.split(',')]
        return name, power
    except Exception as e:  # pragma: no cover
        return 'unknown (%s)' % e, 'unknown'


def time_checks(tmp, chunks, reps, dtype):
    base = np.concatenate([synth.ap_chunk(NS, NC, seed=200 + i) for i in range(8)])
    tile = np.concatenate([base] * (-(-chunks // 8)))[:chunks * NS]
    if dtype == np.float32:
        tile = (tile.astype(np.float64) / 7.3 + 20000.).astype(np.float32)
    path = tmp / ('ap_%s.bin' % np.dtype(dtype).name)
    tile.tofile(path)
    del tile
    out, outmeta = path.with_suffix('.cbin'), path.with_suffix('.ch')
    M.compress(path, out, outmeta, sample_rate=30000., n_channels=NC, dtype=dtype, check_after_compress=False,
               quiet=True)
    data = np.memmap(path, dtype=dtype, mode='r').reshape(-1, NC)
    np.asarray(data).sum(dtype=np.float64)                   # page cache warm
    M.check(data, out, outmeta)                              # warm-up of the GPU path (pinning, modules)
    res = {'gpu': [], 'host': []}
    for _ in range(reps):
        for name, fn in (('gpu', M.check), ('host', host_check)):
            t = time.perf_counter()
            fn(data, out, outmeta)
            res[name].append(time.perf_counter() - t)
    gb = data.nbytes / 1e9
    del data
    for p in (path, out, outmeta):
        p.unlink()
    return {'raw_gb': round(gb, 3),
            'gpu_check_s': [round(x, 3) for x in res['gpu']], 'host_check_s': [round(x, 3) for x in res['host']],
            'gpu_check_gbps': round(gb / min(res['gpu']), 3), 'host_check_gbps': round(gb / min(res['host']), 3),
            'speedup': round(min(res['host']) / min(res['gpu']), 2)}


def device_verify(n_chunks, reps):
    codec = _native.default_codec(0)
    flags = _native.TIME_DIFF
    distinct = [synth.ap_chunk(NS, NC, seed=300 + i) for i in range(8)]
    comps = [codec.compress(x, [0, NS], flags)[0] for x in distinct]
    sizes = [len(comps[i % 8]) for i in range(n_chunks)]
    offs = np.concatenate(([0], np.cumsum(sizes))).astype(np.int64)
    rows = np.arange(n_chunks + 1, dtype=np.int64) * NS
    chunk_bytes = NS * NC * 2
    d_comp = codec.device_alloc(int(offs[-1]) + 256)
    d_ref = codec.device_alloc(n_chunks * chunk_bytes + 256)
    try:
        for i in range(n_chunks):
            codec.memcpy(d_comp + int(offs[i]), comps[i % 8].ctypes.data, sizes[i], 1)
            codec.memcpy(d_ref + i * chunk_bytes, distinct[i % 8].ctypes.data, chunk_bytes, 1)
        ts, cmp_ms, tot_ms = [], [], []
        for r in range(reps + 1):
            t = time.perf_counter()
            st, m, f = codec.verify_ptr(d_comp, 1, offs, rows, NC, 2, flags, d_ref, 1, CHECK_RTOL, CHECK_ATOL)
            dt = time.perf_counter() - t
            assert not st.any() and not m.any()
            tm = codec.timings()
            if r:                                                   # (the first call is the warm-up)
                ts.append(dt)
                cmp_ms.append(tm[6])
                tot_ms.append(tm[7])
    finally:
        codec.device_free(d_comp)
        codec.device_free(d_ref)
    gb = n_chunks * chunk_bytes / 1e9
    return {'chunks': n_chunks, 'raw_gb': round(gb, 3), 'verify_s': [round(x, 3) for x in ts],
            'verify_gbps': round(gb / min(ts), 2), 'compare_ms': [round(x, 2) for x in cmp_ms],
            'device_total_ms': [round(x, 1) for x in tot_ms],
            'compare_share': round(min(cmp_ms) / (min(ts) * 1e3), 4),
            'compare_gbps_hbm': round(2 * gb / (min(cmp_ms) / 1e3), 1)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--chunks', type=int, default=128)
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--dev-chunks', type=int, default=600)
    ap.add_argument('--dir', default=None, help='where the files go (default: /dev/shm when it has room)')
    args = ap.parse_args()
    name, power = card()
    need = args.chunks * NS * NC * 2 * 4                  # the float32 file and its .cbin, with room to spare
    if args.dir is None and os.path.isdir('/dev/shm') and shutil.disk_usage('/dev/shm').free > need:
        args.dir = '/dev/shm'
    tmp = Path(tempfile.mkdtemp(prefix='check_probe_', dir=args.dir))
    try:
        M.CONFIG_PATH = tmp / '.mtscomp'
        res = {'card': name, 'power_limit': power,
               'int16': time_checks(tmp, args.chunks, args.reps, np.int16),
               'float32': time_checks(tmp, args.chunks, args.reps, np.float32),
               'device_resident': device_verify(args.dev_chunks, args.reps)}
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    print(json.dumps(res))


if __name__ == '__main__':
    main()
