# -*- coding: utf-8 -*-
"""mtscomp_b200 — B200-native per-chunk codec behind mtscomp's Writer / Reader / compress / decompress API.

Drop-in for `import mtscomp`: same names, arguments, `.cbin` / `.ch` format.  The codec runs as hand-written sm_100a
kernels reached through a ctypes C ABI (include/mtscomp_b200.h); importing the package needs neither the native library
nor a GPU, using the codec needs both (there is no CPU fallback).
"""

from .config import (  # noqa: F401
    Bunch, CHECK_ATOL, DEFAULT_CONFIG, FORMAT_VERSION, add_default_handler, config_path, read_config, write_config)
from .rawio import load_raw_data  # noqa: F401
from .core import (  # noqa: F401
    Reader, Writer, check, compress, cumsum_along_axis, decompress, diff_along_axis, recompress)
from .cli import (  # noqa: F401
    _args_to_config, mtschop, mtscomp, mtscomp_parser, mtsdecomp, mtsdecomp_parser, mtsdesc, mtsrecomp)

__version__ = '0.1.0'
__all__ = ('load_raw_data', 'Writer', 'Reader', 'compress', 'decompress')

CONFIG_PATH = config_path()
