import glob
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN_DIR = os.path.join(ROOT, 'tests', 'golden')
GOLDEN_CASES = sorted(
    os.path.splitext(os.path.basename(p))[0]
    for p in glob.glob(os.path.join(GOLDEN_DIR, '*.npz'))
    if not os.path.basename(p).startswith(('cg_', 'big_', 'pbc_', 'ecstr_', 'dropin_'))  # iterative-solver / large-molecule / CLI fixtures have their own tests
)


def pytest_configure(config):
    config.addinivalue_line('markers', 'gpu: needs a CUDA device (run on the B200 box with -m gpu)')


def load_golden(name):
    with np.load(os.path.join(GOLDEN_DIR, name + '.npz'), allow_pickle=False) as f:
        return {k: f[k] for k in f.files}


def golden_model(g):
    """Model dict (reference layout, train.py:793-830) from a golden fixture."""
    return {
        'type': 'm',
        'z': g['z'],
        'R_desc': g['model_R_desc'],
        'R_d_desc_alpha': g['R_d_desc_alpha'],
        'alphas_F': g['alphas_F'],
        'c': float(g['c']),
        'std': float(g['std']),
        'sig': int(g['sig']),
        'lam': float(g['lam']),
        'perms': g['perms'],
        'tril_perms_lin': g['tril_perms_lin'],
        'use_E': True,
    }


def golden_task(g):
    from sgdml_b200 import synth

    N = int(g['n_atoms'])
    t = synth.make_task(N, g['R_train'].shape[0], g['perms'], int(g['sig']), lam=float(g['lam']))
    assert np.array_equal(t['R_train'], g['R_train'])  # the generator is deterministic
    return t


def rel_err(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


@pytest.fixture(params=GOLDEN_CASES)
def golden(request):
    return load_golden(request.param)
