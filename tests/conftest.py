import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, 'vocal-remover_b200')
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

GOLDEN = os.path.join(ROOT, 'tests', 'golden')


def pytest_configure(config):
    config.addinivalue_line('markers', 'gpu: needs a CUDA device (run on the B200 box)')


def pytest_collection_modifyitems(config, items):
    """`pytest tests` on a host without a GPU (or without the built library) skips the gpu-marked tests instead of
    failing them; on a GPU box nothing is skipped, so a missing library there is still a loud failure."""
    try:
        import torch
        have_gpu = torch.cuda.is_available()
    except Exception:
        have_gpu = False
    if have_gpu:
        return
    skip = pytest.mark.skip(reason='no CUDA device visible (gpu-marked tests run on the B200 box)')
    for item in items:
        if 'gpu' in item.keywords:
            item.add_marker(skip)


@pytest.fixture(scope='session')
def golden_default():
    import numpy as np
    return np.load(os.path.join(GOLDEN, 'ref_10s_default.npz'))


@pytest.fixture(scope='session')
def golden_small():
    import numpy as np
    return np.load(os.path.join(GOLDEN, 'ref_3s_small.npz'))


@pytest.fixture(scope='session')
def golden_functions():
    import numpy as np
    return np.load(os.path.join(GOLDEN, 'ref_functions.npz'))


def checksum(a):
    import numpy as np
    a = np.asarray(a)
    if np.iscomplexobj(a):
        return np.array([a.real.astype(np.float64).sum(), a.imag.astype(np.float64).sum(),
                         (np.abs(a).astype(np.float64) ** 2).sum(), np.abs(a).max()], dtype=np.float64)
    a64 = a.astype(np.float64)
    return np.array([a64.sum(), (a64 ** 2).sum(), a64.min(), a64.max()], dtype=np.float64)


_PARITY_PATH = os.environ.get('VR_PARITY_JSON', os.path.join(ROOT, 'gpurun_out', 'parity_gpu.json'))


def record_parity(name, value, tol=None):
    """Persist a measured parity number (max-abs error of the CUDA path vs the oracle / golden fixture) so that the
    margin under the gate is on record, not only the pass/fail bit: merged into gpurun_out/parity_gpu.json (a copy of
    the builder's last GPU run is committed as profiles/r02_parity.json)."""
    import json
    try:
        os.makedirs(os.path.dirname(_PARITY_PATH), exist_ok=True)
        data = {}
        if os.path.exists(_PARITY_PATH):
            with open(_PARITY_PATH) as f:
                data = json.load(f)
        data[name] = {'max_abs_err': float(value)} if tol is None else {'max_abs_err': float(value), 'gate': float(tol)}
        with open(_PARITY_PATH, 'w') as f:
            json.dump(data, f, indent=1, sort_keys=True)
    except OSError:
        pass
    print('PARITY %s = %.4g%s' % (name, float(value), '' if tol is None else ' (gate %.1g)' % tol))
