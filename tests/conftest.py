import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line('markers', 'gpu: needs a CUDA (B200) device')


@pytest.fixture
def one_thread():
    """Torch's intra-op pool splits CPU reductions by thread count: comparisons with stored
    reference bits run on one thread, as the reference outputs were computed."""
    import torch
    n = torch.get_num_threads()
    torch.set_num_threads(1)
    yield
    torch.set_num_threads(n)


@pytest.fixture(scope='session')
def cuda_dev():
    import torch
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    from xrdslam_b200 import _cabi
    _cabi.check('xrd_check_device', _cabi.lib().xrd_check_device(0))
    return torch.device('cuda:0')
