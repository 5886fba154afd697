"""GPU: the misled-index cases (tests/misled_cases.py) on the B200."""
import pytest

import misled_cases

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def small_batches():
    """A context of its own: the cases set its sub-batch sizes and write_index."""
    from mtscomp_b200 import _native
    c = misled_cases.small_batches(_native.Codec(0))
    yield c
    c.close()


@pytest.fixture(scope='module')
def built(small_batches):
    return misled_cases.build(small_batches)


@pytest.mark.parametrize('case', misled_cases.ALL_CASES, ids=lambda f: f.__name__)
def test_misled(case, small_batches, built):
    case(small_batches, built)
