import os
import sys

import pytest

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), '..'))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, 'tests', 'golden')


def pytest_configure(config):
    config.addinivalue_line('markers', 'gpu: test needs a CUDA device (run on the B200 box with -m gpu)')


@pytest.fixture(scope='session')
def golden_ops():
    import numpy as np
    return np.load(os.path.join(GOLDEN, 'ref_python_ops.npz'))


@pytest.fixture(scope='session')
def golden_fpp():
    import numpy as np
    # two files, each under 1 MB: the frame inputs + the 'spec' parameter set, and the 'stress' set
    return {**np.load(os.path.join(GOLDEN, 'ref_forward_perpix.npz')), **np.load(os.path.join(GOLDEN, 'ref_forward_perpix_stress.npz'))}
