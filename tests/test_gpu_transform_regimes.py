"""GPU: the transform stage (K1 forward, K4 inverse) at every channel-width regime and on IEEE special values.

launch_fwd_t / launch_inv_t (csrc/capi.cu) pick a kernel by n_channels: the channel-major tile kernels with 1, 2 or 4
channels per thread up to 448, 896 and 1792 channels, the generic kernels above that and in 'C' order.  Each case goes
through four paths against oracle/codec.py (NumPy in the array's own dtype): delta_transform, inverse_transform with
its adler32, compress (zlib must return the reference's transform bytes) and decompress of reference-written streams,
on a batch of ragged chunks.  Comparisons are of bit patterns; for NaN payloads see tests/transform_cases.py."""
import numpy as np
import pytest

from transform_cases import FLAG_SETS, NAN_PAYLOAD_SKIP, check_four_paths, float_data, int_data, \
    nan_payloads_checked, ragged_rows

pytestmark = pytest.mark.gpu

WIDTHS = [447, 448, 449, 896, 897, 1792, 1793, 2100]
INT_CASES = [('int16', nc) for nc in WIDTHS] + \
    [(dt, nc) for dt in ('uint8', 'int32', 'int64') for nc in (448, 449, 896, 897, 1792, 1793)]
FLOAT_WIDTHS = [7, 93, 94, 189, 190, 385, 449, 897, 1793]


def _int_matrix(cd, dtype, nc, orders='FC'):
    rows = ragged_rows(dtype, nc)
    for kind in ('random', 'smooth'):
        x = int_data(kind, dtype, int(rows[-1]), nc, seed=nc * 7 + len(kind))
        for order in orders:
            for td, sd in FLAG_SETS:
                check_four_paths(cd, x, rows, td, sd, order)


@pytest.mark.parametrize('dtype,nc', INT_CASES)
def test_int_widths(codec, dtype, nc):
    _int_matrix(codec, dtype, nc)


@pytest.mark.parametrize('nc', WIDTHS)
def test_int_widths_multi_kernel_inverse(codec, nc):
    """The inverse as tile sums + scan + apply (or per-column sums), which otherwise only runs above 1792 channels or
    in 'C' order."""
    codec.set_param('inv_single_pass', 0)
    try:
        _int_matrix(codec, 'int16', nc, orders='F')
    finally:
        codec.set_param('inv_single_pass', 1)


def _tile_pitch_int16(nc):                          # transform.cuh tile_pitch<uint16_t>
    p = (nc + 1) & ~1
    return p + 2 if (p & 2) == 0 else p


def _tile_rows(nc, extra_rows):                     # capi.cu tile_rows for 2-byte elements
    return min(64, 98304 // (_tile_pitch_int16(nc) * 2) - extra_rows)


def test_int16_widest_generic_tile(codec):
    """'C' order: the widest n_channels whose forward tile still holds one row (plus the row above) is exact; the
    next one is refused with a clear error rather than launched."""
    from mtscomp_b200 import _native
    widest = max(nc for nc in range(20000, 30000) if _tile_rows(nc, 1) >= 1)
    assert _tile_rows(widest, 1) == 1 and _tile_rows(widest + 1, 1) < 1
    rows = np.array([0, 1, 3, 6], dtype=np.int64)
    for kind in ('random', 'smooth'):
        x = int_data(kind, 'int16', 6, widest, seed=len(kind))
        for td, sd in FLAG_SETS:
            check_four_paths(codec, x, rows, td, sd, 'C')
    y = np.zeros((3, widest + 1), np.int16)
    for td, sd in FLAG_SETS:
        with pytest.raises(_native.NativeError, match='too large for the transform tile'):
            codec.delta_transform(y, _native.flags_of(td, sd, 'C'))
        with pytest.raises(_native.NativeError, match='too large for the transform tile'):
            codec.compress(y, [0, 1, 3], _native.flags_of(td, sd, 'C'))


@pytest.mark.parametrize('dtype', ['float32', 'float64'])
@pytest.mark.parametrize('nc', FLOAT_WIDTHS)
def test_float_widths_and_special_values(codec, dtype, nc):
    """Smooth and wide-dynamic-range data with signed zeros, subnormals, overflowing differences, inf - inf, quiet
    NaNs with payloads and signalling NaNs at row 0, column 0, the last row and column and the first and last row of
    every chunk.  The generic forward kernel needs more than 48 KB of shared memory from 190 float32 / 94 float64
    channels on in 'C' order and above 1792 channels in either order."""
    rows = ragged_rows(dtype, nc)
    for kind in ('smooth', 'wild'):
        x = float_data(kind, dtype, rows, nc, seed=nc)
        for order in 'FC':
            for td, sd in FLAG_SETS:
                check_four_paths(codec, x, rows, td, sd, order)
    if not nan_payloads_checked():
        pytest.skip(NAN_PAYLOAD_SKIP)
