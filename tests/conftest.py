import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, 'tests', 'golden')


def pytest_configure(config):
    config.addinivalue_line('markers', 'gpu: needs a CUDA device (run on the B200 box: pytest -m gpu)')


def load_golden(name):
    return np.load(os.path.join(GOLDEN, name))


def cases_of(npz, key='cases'):
    return json.loads(bytes(npz[key]).decode())


def golden_input(npz, case):
    """Input `x<k>` of a golden case: stored, or -- for uniform [0, 32) inputs -- regenerated from the seed and shape the case records
    (tests/golden/make_golden.py draws them first from that seed)."""
    k = case['k']
    if f'x{k}' in npz.files:
        return npz[f'x{k}']
    return (np.random.RandomState(case['seed']).rand(*case['shape']) * 32).astype(np.float32)


def seeded_batches(seed, n, shape, relu):
    """Same generator as tests/golden/make_golden.py::batches (numpy legacy RandomState: bit-stable)."""
    r = np.random.RandomState(seed)
    out = []
    for _ in range(n):
        x = r.standard_normal(size=shape).astype(np.float32)
        if relu:
            x = np.maximum(x, 0)
        out.append(x)
    return out


@pytest.fixture(scope='session')
def oracle():
    import oracle as ora
    ora.lib()
    return ora
