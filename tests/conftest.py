import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import golden_inputs  # noqa: E402
from sushi_b200 import _hostmem  # noqa: E402

_hostmem.keep_heap()
GOLDEN = os.path.join(ROOT, 'tests', 'golden')


def pytest_configure(config):
    config.addinivalue_line('markers', 'gpu: needs a B200 (run with -m gpu on the GPU box)')


@pytest.fixture(scope='session')
def golden_loader():
    return golden_inputs.load(os.path.join(GOLDEN, 'loader.npz'), 'loader')


@pytest.fixture(scope='session')
def golden_loader24():
    """24-bit WAV files and what the reference's own loader makes of them (oracle/gen_golden.py gen_loader24)."""
    return golden_inputs.load(os.path.join(GOLDEN, 'loader24.npz'), 'loader24')


@pytest.fixture(scope='session')
def golden_matcher():
    return golden_inputs.load(os.path.join(GOLDEN, 'matcher.npz'), 'matcher')


@pytest.fixture(scope='session')
def golden_shifts():
    return np.load(os.path.join(GOLDEN, 'shifts.npz'))


@pytest.fixture(scope='session')
def gpu_lib():
    """The initialised C-ABI library; fails (not skips) when there is no GPU: the gpu-marked
    tests are only selected on the GPU box."""
    from sushi_b200 import _native
    return _native.lib()
