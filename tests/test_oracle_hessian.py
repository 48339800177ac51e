"""The NumPy Hessian oracle (oracle/hessian.py) against central differences of the oracle's forces, its symmetry,
the translational sum rule and permutation equivariance; and the C-ABI table entry of the engine's Hessian call.
CPU only."""

import numpy as np
import pytest

from conftest import golden_model, load_golden  # noqa: E402

from oracle import hessian as ohess  # noqa: E402
from oracle import predict as opredict  # noqa: E402

FIXTURES = ['n5_m10_s1', 'n9_m16_s6', 'n12_m8_s12', 'n21_m6_s6', 'pbc_n6_m8', 'ecstr_n6_m8']


def _model(name):
    g = load_golden(name)
    m = golden_model(g)
    if 'lattice' in g:
        m['lattice'] = g['lattice']
    if 'alphas_E' in g:
        m['alphas_E'] = g['alphas_E']
    return g, m


def _fd_hessian(pred, r, h=1e-4):
    """H[:, j] = -(F(r + h e_j) - F(r - h e_j)) / 2h."""
    n = r.size
    Rp = r[None, :] + h * np.eye(n)
    Rm = r[None, :] - h * np.eye(n)
    _, Fp = pred.predict(Rp)
    _, Fm = pred.predict(Rm)
    return -((Fp - Fm) / (2 * h)).T


@pytest.mark.parametrize('name', FIXTURES)
@pytest.mark.parametrize('where', ['query', 'train'])
def test_oracle_hessian_matches_central_differences(name, where):
    g, model = _model(name)
    pred = opredict.Predictor(model)
    r = (g['R_query'][0] if where == 'query' else g['R_train'][0]).reshape(-1).astype(np.float64)
    H = ohess.hessian(model, r, predictor=pred)[0]
    assert np.all(np.isfinite(H))
    H_fd = _fd_hessian(pred, r)
    scale = np.max(np.abs(H))
    assert np.max(np.abs(H - H_fd)) / scale < 1e-6
    assert np.max(np.abs(H - H.T)) / scale < 1e-12
    N = r.size // 3
    rowsum = H.reshape(3 * N, N, 3).sum(axis=1)  # sum over the atoms b of H[(a, i), (b, j)]
    assert np.max(np.abs(rowsum)) / scale < 1e-11


@pytest.mark.parametrize('name', ['n9_m16_s6', 'n12_m8_s12'])
def test_oracle_hessian_permutation_equivariance(name):
    """For an atom permutation pi of the model's group: H(Pi R) = Pi H(R) Pi^T."""
    g, model = _model(name)
    N = int(g['n_atoms'])
    r = g['R_query'][1].reshape(N, 3)
    H = ohess.hessian(model, r.ravel())[0]
    for pi in g['perms'][1:3]:
        pi = np.asarray(pi)
        coord = (3 * pi[:, None] + np.arange(3)[None, :]).ravel()  # permuted coordinate order
        Hp = ohess.hessian(model, r[pi].ravel())[0]
        assert np.max(np.abs(Hp - H[np.ix_(coord, coord)])) / np.max(np.abs(H)) < 1e-11


def test_hessian_symbol_in_abi_table():
    from sgdml_b200 import _lib

    assert 'sgdml_b200_predict_hessian' in _lib.SIGNATURES
    assert _lib.KERNEL_FAMILIES[-1] == 'hessian'
