# -*- coding: utf-8 -*-
"""Command-line front-ends mtscomp / mtsdecomp / mtsdesc / mtschop (reference mtscomp.py:1004-1179) and mtsrecomp."""

import argparse
import sys

import numpy as np

from .config import add_default_handler, read_config, write_config
from .core import Reader, compress, decompress, recompress


def exception_handler(exception_type, exception, traceback, debug_hook=sys.excepthook):  # pragma: no cover
    if '--debug' in sys.argv or '-v' in sys.argv:
        debug_hook(exception_type, exception, traceback)
    else:
        print("%s: %s" % (exception_type.__name__, exception))


def _shared_options(parser):
    parser.add_argument('-nc', '--no-check', action='store_false', help='no check')
    parser.add_argument('-v', '--debug', action='store_true', help='verbose')
    parser.add_argument('-p', '--cpus', type=int, help='number of CPUs to use')


def _args_to_config(parser, args, compress=True):
    pargs = parser.parse_args(args)
    # store_false: True means the flag was absent -> keep the configured default
    check_after = None if pargs.no_check is True else False
    kwargs = dict(n_threads=pargs.cpus)
    if compress:
        kwargs.update(
            sample_rate=pargs.sample_rate, n_channels=pargs.n_channels,
            dtype=pargs.dtype.strip() if pargs.dtype else pargs.dtype,
            chunk_duration=pargs.chunk, check_after_compress=check_after)
    else:
        kwargs.update(check_after_decompress=check_after)
    return pargs, read_config(**kwargs)


def mtscomp_parser():
    parser = argparse.ArgumentParser(description='Compress a raw binary file.')
    parser.add_argument('path', type=str, help='input path of a raw binary file')
    parser.add_argument('out', type=str, nargs='?', help='output path of the compressed binary file (.cbin)')
    parser.add_argument('outmeta', type=str, nargs='?', help='output path of the compression metadata JSON file (.ch)')
    parser.add_argument('-d', '--dtype', type=str, help='data type')
    parser.add_argument('-s', '--sample-rate', type=float, help='sample rate')
    parser.add_argument('-n', '--n-channels', type=int, help='number of channels')
    parser.add_argument('-c', '--chunk', type=int, help='chunk duration')
    _shared_options(parser)
    parser.add_argument('--set-default', action='store_true', help='set the specified parameters as the default')
    return parser


def mtscomp(args=None):
    """Compress a file."""
    sys.excepthook = exception_handler
    parser = mtscomp_parser()
    pargs, config = _args_to_config(parser, args or sys.argv[1:], compress=True)
    add_default_handler('DEBUG' if pargs.debug else 'INFO')
    if pargs.set_default:
        write_config(**config)
    compress(pargs.path, pargs.out, pargs.outmeta, **config)


def mtsdecomp_parser():
    parser = argparse.ArgumentParser(description='Decompress a raw binary file.')
    parser.add_argument('cdata', type=str, help='path to the input compressed binary file (.cbin)')
    parser.add_argument('cmeta', type=str, nargs='?', help='path to the input compression metadata JSON file (.ch)')
    parser.add_argument('-o', '--out', type=str, nargs='?', help='path to the output decompressed file (.bin)')
    parser.add_argument('--overwrite', '-f', action='store_true', help='overwrite existing output')
    _shared_options(parser)
    return parser


def mtsdecomp(args=None):
    """Decompress a file."""
    sys.excepthook = exception_handler
    parser = mtsdecomp_parser()
    pargs, config = _args_to_config(parser, args or sys.argv[1:], compress=False)
    add_default_handler('DEBUG' if pargs.debug else 'INFO')
    decompress(pargs.cdata, pargs.cmeta, out=pargs.out, write_output=True, overwrite=pargs.overwrite, **config)


def mtsdesc(args=None):
    """Describe a compressed file."""
    sys.excepthook = exception_handler
    parser = mtsdecomp_parser()
    parser.description = 'Describe a compressed file.'
    pargs = parser.parse_args(args or sys.argv[1:])
    r = Reader()
    r.open(pargs.cdata, pargs.cmeta)
    sr = float(r.cmeta.sample_rate)
    rows = (
        ('dtype', r.dtype), ('sample_rate', sr), ('n_channels', r.n_channels),
        ('duration', '%.1fs' % (r.n_samples / sr)), ('n_samples', r.n_samples),
        ('chunk_duration', '%.1fs' % (np.diff(r.chunk_bounds).mean() / sr)), ('n_chunks', r.n_chunks))
    for k, v in rows:
        print('{:<15}'.format(k), str(v))


def mtschop(args=None):
    """Chop a compressed file to N chunks without decompressing it."""
    sys.excepthook = exception_handler
    parser = argparse.ArgumentParser(description='Chop a compressed file to N chunks without decompressing it.')
    parser.add_argument('cdata', type=str, help='path to the input compressed binary file (.cbin)')
    parser.add_argument('-n', '--n_chunks', type=int, help='number of chunks to chop')
    parser.add_argument('-o', '--out', type=str, help='path to the output chopped compressed file (.cbin)')
    _shared_options(parser)
    pargs = parser.parse_args(args or sys.argv[1:])
    r = Reader()
    r.open(pargs.cdata)
    r.chop(pargs.n_chunks, pargs.out)
    r.close()


def mtsrecomp(args=None):
    """Re-encode a compressed file on the GPU, with or without the segment index, without decompressing it."""
    sys.excepthook = exception_handler
    parser = argparse.ArgumentParser(
        description='Re-encode a compressed file on the GPU from its chunks\' inflated bytes: adds the segment index '
                    'that speeds up decoding (or strips it with --no-index). The new file decodes to exactly what the '
                    'input decodes to.')
    parser.add_argument('cdata', type=str, help='path to the input compressed binary file (.cbin)')
    parser.add_argument('cmeta', type=str, nargs='?', help='path to the input compression metadata JSON file (.ch)')
    parser.add_argument('-o', '--out', type=str, required=True, help='path to the output compressed file (.cbin)')
    parser.add_argument('--outmeta', type=str, help='path to the output metadata file (.ch, default: next to --out)')
    parser.add_argument('--no-index', action='store_true', help='write one plain zlib stream per chunk, no index')
    parser.add_argument('--overwrite', '-f', action='store_true', help='overwrite existing output')
    _shared_options(parser)
    pargs = parser.parse_args(args or sys.argv[1:])
    add_default_handler('DEBUG' if pargs.debug else 'INFO')
    # store_false: True means the flag was absent -> keep the configured default
    check_after = None if pargs.no_check is True else False
    return recompress(pargs.cdata, pargs.cmeta, out=pargs.out, outmeta=pargs.outmeta, write_index=not pargs.no_index,
                      overwrite=pargs.overwrite, n_threads=pargs.cpus, check_after_compress=check_after)
