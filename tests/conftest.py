import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, 'tests')):
    if p not in sys.path:
        sys.path.insert(0, p)


def pytest_configure(config):
    config.addinivalue_line('markers', 'gpu: needs a CUDA device')
    # torch's CPU kernels split reductions by the intra-op thread count, so the oracle reproduces the reference results
    # stored under tests/golden/ bit for bit only with the count they were written with
    import torch
    torch.set_num_threads(8)


@pytest.fixture(scope='session')
def golden():
    import torch
    import cases
    return torch.load(cases.GOLDEN_PATH, map_location='cpu', weights_only=False)
