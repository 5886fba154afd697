# -*- coding: utf-8 -*-
"""Build recipe for the native library (nvcc, sm_100a).  `python -m mtscomp_b200.build` builds in-tree."""
import os
import subprocess
import sys
from pathlib import Path

PKG = Path(__file__).resolve().parent
CSRC = PKG / 'csrc'
BUILD = PKG / '_build'
LIB = BUILD / 'libmtscomp_b200.so'
SOURCES = ['capi.cu']
HEADERS = ['common.cuh', 'transform.cuh', 'deflate.cuh', 'inflate.cuh', 'inflate_par.cuh', 'inflate_seg.cuh', 'verify.cuh',
           '../../include/mtscomp_b200.h']


def _stale(target, deps):
    if not target.exists():
        return True
    t = target.stat().st_mtime
    return any(Path(d).stat().st_mtime > t for d in deps)


def build_native(force=False, verbose=False, out=None, extra=()):
    """nvcc -gencode arch=compute_100a,code=sm_100a -> mtscomp_b200/_build/libmtscomp_b200.so
    (`out` / `extra`: development variants, e.g. build_native(out='_build/lib_prof.so', extra=['-DMTS_LZ_PROFILE']),
    selected at run time with MTSCOMP_B200_LIB)."""
    BUILD.mkdir(exist_ok=True)
    deps = [CSRC / s for s in SOURCES] + [CSRC / h for h in HEADERS]
    if out is None and not force and not _stale(LIB, deps):
        return LIB
    nvcc = os.environ.get('NVCC', '/usr/local/cuda/bin/nvcc')
    cmd = [nvcc, '-O3', '-std=c++17', '-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo',
           '-Xcompiler', '-fPIC', '-shared', '-o', str(out or LIB)] + list(extra) + [str(CSRC / s) for s in SOURCES]
    if verbose:
        cmd.insert(1, '-Xptxas=-v')
    if os.environ.get('MTS_LZ_PROFILE'):
        cmd.insert(1, '-DMTS_LZ_PROFILE')
    cmd[1:1] = os.environ.get('MTS_EXTRA_FLAGS', '').split()
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError('nvcc failed:\n' + res.stdout + res.stderr)
    if verbose:
        print(res.stdout + res.stderr)
    return Path(out) if out else LIB


def build_emulation(force=False):
    """DEVELOPMENT ONLY: the same sources compiled for the host against csrc/emu/cuda_emu.h (kernel-logic emulation,
    never loaded by the package)."""
    out = BUILD / 'libmtscomp_b200_emu.so'
    BUILD.mkdir(exist_ok=True)
    deps = [CSRC / s for s in SOURCES] + [CSRC / h for h in HEADERS] + [CSRC / 'emu/cuda_emu.h', CSRC / 'emu/cuda_emu.cpp']
    if not force and not _stale(out, deps):
        return out
    cmd = ['g++', '-O2', '-g', '-std=c++17', '-DMTSCOMP_EMU', '-fPIC', '-shared', '-w', '-o', str(out),
           '-x', 'c++'] + [str(CSRC / s) for s in SOURCES] + [str(CSRC / 'emu/cuda_emu.cpp'), '-lpthread']
    cmd[1:1] = os.environ.get('MTS_EXTRA_FLAGS', '').split()
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError('g++ (emulation) failed:\n' + res.stdout + res.stderr)
    return out


if __name__ == '__main__':
    print(build_native(force='--force' in sys.argv, verbose='-v' in sys.argv))
