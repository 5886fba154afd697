"""What recompress() costs and what it buys.  Prints one JSON line (with the card's name and power limit).

(a) Device-resident: 600 reference-written AP chunks (385 x int16, 8 distinct synth.ap_chunk chunks tiled, as bench.py
    builds them) recompressed in HBM (mtsb_recompress_chunks), against decompress_ptr followed by compress_ptr on the
    same device buffers.  The two alternate; their outputs are compared byte for byte.  GB/s of raw bytes (host clock
    around the synchronous calls) and the per-stage ms of mtsb_last_timings.
(b) File to file on /dev/shm: 128 reference-written chunks, recompress() against decompress(write_output=True)
    followed by compress(), each with its check after writing on and off, alternating.
(c) The payoff: device-resident decode GB/s of the reference-written source and of the recompressed file, and the p50
    of a random 10 ms window (Reader, cache_size 1) on both files.

    python tools/recompress_probe.py [--dev-chunks 600] [--file-chunks 128] [--reps 3] [--dir /dev/shm]
"""
import argparse
import hashlib
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

import numpy as np

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
import mtscomp_b200 as M                                                       # noqa: E402
from mtscomp_b200 import _native, synth                                        # noqa: E402
from mtscomp_b200.config import FORMAT_VERSION                                 # noqa: E402
from oracle import codec as ora                                                # noqa: E402

NS, NC, DISTINCT = 30000, 385, 8
CHUNK_BYTES = NS * NC * 2
STAGES = ['h2d', 'plan', 'inflate', 'adler', 'lz77', 'huffman_scan_encode', 'unused', 'total']


def card():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=60).stdout.strip()
        name, power = [s.strip() for s in q.split(',')]
        return name, power
    except Exception as e:  # pragma: no cover
        return 'unknown (%s)' % e, 'unknown'


def sources():
    """The distinct chunks (bench.py's seeds) and their reference-written streams (zlib level 6)."""
    base = [synth.ap_chunk(NS, NC, seed=1234 + i, t0=i * NS) for i in range(DISTINCT)]
    with ThreadPoolExecutor(DISTINCT) as ex:
        streams = list(ex.map(ora.encode_chunk, base))
    return base, streams


def tiled(streams, n):
    parts = [streams[i % DISTINCT] for i in range(n)]
    offs = np.concatenate(([0], np.cumsum([len(p) for p in parts]))).astype(np.int64)
    return parts, offs


def device_resident(cd, base, streams, n, reps):
    fl = _native.TIME_DIFF
    parts, offs = tiled(streams, n)
    rows = np.arange(n + 1, dtype=np.int64) * NS
    cap = n * cd.compress_bound(NS, NC, 2, fl)
    raw_bytes = n * CHUNK_BYTES
    bufs = {'src': int(offs[-1]), 'raw': raw_bytes, 'out_r': cap, 'out_c': cap}
    d = {k: cd.device_alloc(v + 256) for k, v in bufs.items()}
    try:
        for i, p in enumerate(parts):
            a = np.frombuffer(p, np.uint8)
            cd.memcpy(d['src'] + int(offs[i]), a.ctypes.data, a.nbytes, 1)

        def recompress():
            o, st = cd.recompress_ptr(d['src'], 1, offs, rows, NC, 2, fl, d['out_r'], 1, cap)
            assert not st.any()
            return o

        def composed():
            st = cd.decompress_ptr(d['src'], 1, offs, rows, NC, 2, fl, d['raw'], 1)
            assert not st.any()
            return cd.compress_ptr(d['raw'], 1, rows, NC, 2, fl, d['out_c'], 1, cap)

        res = {'recompress': [], 'composed': []}
        stages = []
        recompress(), composed()                                 # warm-up
        for _ in range(reps):
            for name, fn in (('recompress', recompress), ('composed', composed)):
                t = time.perf_counter()
                o = fn()
                res[name].append(time.perf_counter() - t)
                if name == 'recompress':
                    stages.append(cd.timings())
                    o_r = o
                else:
                    o_c = o
        same_offsets = o_r.tolist() == o_c.tolist()
        size = int(o_r[-1])
        a, b = np.empty(size, np.uint8), np.empty(size, np.uint8)
        cd.memcpy(a.ctypes.data, d['out_r'], size, 2)
        cd.memcpy(b.ctypes.data, d['out_c'], size, 2)
        identical = same_offsets and np.array_equal(a, b)
        del a, b
        # (c) device-resident decode of the source and of the recompressed chunks
        dec = {'reference_written': [], 'recompressed': []}
        for _ in range(reps + 1):
            for name, ptr, o in (('reference_written', d['src'], offs), ('recompressed', d['out_r'], o_r)):
                t = time.perf_counter()
                st = cd.decompress_ptr(ptr, 1, o, rows, NC, 2, fl, d['raw'], 1)
                dec[name].append(time.perf_counter() - t)
                assert not st.any()
    finally:
        for p in d.values():
            cd.device_free(p)
    gb = raw_bytes / 1e9
    best = min(range(reps), key=lambda k: stages[k][7])
    return {
        'chunks': n, 'raw_gb': round(gb, 3),
        'recompress_s': [round(x, 3) for x in res['recompress']], 'composed_s': [round(x, 3) for x in res['composed']],
        'recompress_gbps': round(gb / min(res['recompress']), 2), 'composed_gbps': round(gb / min(res['composed']), 2),
        'recompress_stage_ms': {s: round(v, 1) for s, v in zip(STAGES, stages[best])},
        'outputs_identical': bool(identical), 'compressed_gb': round(int(o_r[-1]) / 1e9, 3),
        'decode_gbps': {k: round(gb / min(v[1:]), 2) for k, v in dec.items()},
    }


def write_reference_file(d, base, streams, n):
    """A .cbin / .ch pair as the reference Writer writes it, tiled from the distinct chunks' streams."""
    raw = np.concatenate([base[i % DISTINCT] for i in range(n)])
    raw.tofile(d / 'src.bin')
    parts, offs = tiled(streams, n)
    sha_c = hashlib.sha1()
    with open(d / 'src.cbin', 'wb') as f:
        for p in parts:
            f.write(p)
            sha_c.update(p)
    meta = {'version': FORMAT_VERSION, 'algorithm': 'zlib', 'comp_level': -1, 'do_time_diff': True,
            'do_spatial_diff': False, 'dtype': 'int16', 'n_channels': NC, 'sample_rate': float(NS),
            'chunk_bounds': [i * NS for i in range(n + 1)], 'chunk_offsets': offs.tolist(), 'chunk_order': 'F',
            'sha1_compressed': sha_c.hexdigest(), 'sha1_uncompressed': hashlib.sha1(raw.tobytes()).hexdigest(),
            'shape': list(raw.shape)}
    (d / 'src.ch').write_text(json.dumps(meta, indent=2, sort_keys=True))
    return raw


def file_to_file(d, raw, reps):
    def recompress(check):
        M.recompress(d / 'src.cbin', d / 'src.ch', d / 'rc.cbin', overwrite=True, quiet=True, check_after_compress=check)

    def composed(check):
        M.decompress(d / 'src.cbin', d / 'src.ch', out=d / 'dec.bin', overwrite=True, quiet=True,
                     check_after_decompress=check).close()
        M.compress(d / 'dec.bin', d / 'cc.cbin', d / 'cc.ch', sample_rate=float(NS), n_channels=NC, dtype=np.int16,
                   quiet=True, check_after_compress=check)

    out = {}
    for check in (False, True):
        recompress(check), composed(check)                     # warm-up (pinning, modules)
        ts = {'recompress': [], 'composed': []}
        for _ in range(reps):
            for name, fn in (('recompress', recompress), ('composed', composed)):
                t = time.perf_counter()
                fn(check)
                ts[name].append(time.perf_counter() - t)
        gb = raw.nbytes / 1e9
        out['check_on' if check else 'check_off'] = {
            'recompress_s': [round(x, 3) for x in ts['recompress']], 'composed_s': [round(x, 3) for x in ts['composed']],
            'recompress_gbps': round(gb / min(ts['recompress']), 3), 'composed_gbps': round(gb / min(ts['composed']), 3)}
    same = (d / 'rc.cbin').read_bytes() == (d / 'cc.cbin').read_bytes()
    out['outputs_identical'] = same
    out['raw_gb'] = round(raw.nbytes / 1e9, 3)
    return out


def window_p50(d, raw, n=40, seed=11):
    w = NS // 100
    res = {}
    for name, cbin in (('reference_written', 'src'), ('recompressed', 'rc')):
        r = M.decompress(d / (cbin + '.cbin'), d / (cbin + '.ch'), cache_size=1)
        r[0:300]
        rng = np.random.default_rng(seed)
        ts = []
        for _ in range(n):
            t0 = int(rng.integers(0, raw.shape[0] - w))
            t = time.perf_counter()
            a = r[t0:t0 + w, :]
            ts.append((time.perf_counter() - t) * 1e3)
            assert np.array_equal(a, raw[t0:t0 + w])
        r.close()
        res[name] = {'p50_ms': round(float(np.percentile(ts, 50)), 3), 'n': n}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--dev-chunks', type=int, default=600)
    ap.add_argument('--file-chunks', type=int, default=128)
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--dir', default=None, help='where the files go (default: /dev/shm when it has room)')
    args = ap.parse_args()
    name, power = card()
    cd = _native.default_codec(0)
    base, streams = sources()
    res = {'card': name, 'power_limit': power,
           'device_resident': device_resident(cd, base, streams, args.dev_chunks, args.reps)}
    need = args.file_chunks * CHUNK_BYTES * 4
    if args.dir is None and os.path.isdir('/dev/shm') and shutil.disk_usage('/dev/shm').free > need:
        args.dir = '/dev/shm'
    tmp = Path(tempfile.mkdtemp(prefix='recompress_probe_', dir=args.dir))
    try:
        M.CONFIG_PATH = tmp / '.mtscomp'
        raw = write_reference_file(tmp, base, streams, args.file_chunks)
        res['file_to_file'] = file_to_file(tmp, raw, args.reps)
        res['file_to_file']['dir'] = str(tmp.parent)
        res['window_10ms'] = window_p50(tmp, raw)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    print(json.dumps(res))


if __name__ == '__main__':
    main()
