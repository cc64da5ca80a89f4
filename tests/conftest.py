import json
import os
import sys

import numpy as np
import pytest

from golden_data import arrays_sha256

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, 'tests', 'golden')


def pytest_configure(config):
    config.addinivalue_line('markers', 'gpu: needs a CUDA device (run on the B200 box)')


def rel_l2(a, b):
    """Per-row relative L2 error ||a-b|| / ||b|| (the parity metric of SURVEY.md section 8d)."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    a = a.reshape(a.shape[0], -1) if a.ndim > 1 else a[None]
    b = b.reshape(b.shape[0], -1) if b.ndim > 1 else b[None]
    return np.linalg.norm(a - b, axis=1) / np.maximum(np.linalg.norm(b, axis=1), 1e-30)


@pytest.fixture(scope='session')
def manifest():
    with open(os.path.join(GOLDEN, 'manifest.json')) as f:
        return json.load(f)


def load_golden(name):
    """Arrays of tests/golden/<name>.npz and the weights they were made with.  A fixture whose weights would take it past
    1 MB stores ``sd_sha256`` instead of ``sd/*``: the weights are regenerated from the manifest's seed and must match."""
    import torch
    z = np.load(os.path.join(GOLDEN, name + '.npz'))
    sd = {k[3:]: torch.from_numpy(z[k]) for k in z.files if k.startswith('sd/')}
    if 'sd_sha256' in z.files:
        from oracle import models as om
        with open(os.path.join(GOLDEN, 'manifest.json')) as f:
            m = json.load(f)[name]
        sd = om.random_state_dict(m['model'], m['feature_dim'], seed=m['seed'], **m['model_args'])
        assert arrays_sha256(sd.items()) == str(z['sd_sha256']), f'{name}: seeded weights differ from the golden run'
    return z, sd
