import glob
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, 'tests', 'golden')


def pytest_configure(config):
    config.addinivalue_line('markers', 'gpu: needs a CUDA device (run on the B200 box with -m gpu)')


@pytest.fixture(scope='session')
def golden():
    import torch

    def load(name):
        """tests/golden/<name>; a set stored in parts (tests/golden/make_golden.py: save) is read from the numbered
        files under tests/golden/<stem>/ and joined back in order."""
        path = os.path.join(GOLDEN, name)
        if os.path.isfile(path):
            return torch.load(path, weights_only=False)
        files = sorted(glob.glob(os.path.join(os.path.splitext(path)[0], '*.pt')))
        assert files, f'golden set {name} not found'
        parts = [torch.load(f, weights_only=False) for f in files]
        if isinstance(parts[0], dict):
            return {k: [c for p in parts for c in p[k]] for k in parts[0]}
        return [c for p in parts for c in p]
    return load
