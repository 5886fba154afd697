"""CPU: the misled-index cases (tests/misled_cases.py) through the host emulation of the kernels."""
import pytest

import misled_cases


@pytest.fixture(scope='module')
def emu():
    from mtscomp_b200 import _native, build
    c = misled_cases.small_batches(_native.Codec(0, lib=_native.load_library(build.build_emulation())))
    yield c
    c.close()


@pytest.fixture(scope='module')
def built(emu):
    return misled_cases.build(emu)


@pytest.mark.parametrize('case', misled_cases.ALL_CASES, ids=lambda f: f.__name__)
def test_misled_emulated(case, emu, built):
    case(emu, built)
