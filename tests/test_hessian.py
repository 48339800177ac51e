"""Analytic Hessian on the GPU (sgdml_b200_predict_hessian, GDMLPredict.predict_hessian) against the NumPy oracle
(oracle/hessian.py), against central differences of the engine's own forces, and its API contract."""

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from conftest import golden_model, load_golden, rel_err  # noqa: E402

from oracle import desc as odesc  # noqa: E402
from oracle import hessian as ohess  # noqa: E402


@pytest.fixture(scope='module')
def eng():
    import sgdml_b200
    from sgdml_b200 import _lib

    _lib.require_gpu()
    return sgdml_b200


def _fixture_model(name):
    g = load_golden(name)
    m = golden_model(g)
    if 'lattice' in g:
        m['lattice'] = g['lattice']
    if 'alphas_E' in g:
        m['alphas_E'] = g['alphas_E']
    return g, m


def _random_model(R_train, perms, sig, seed=0):
    """Model with random coefficients on the given training geometries (oracle descriptors, no GPU involved)."""
    M = R_train.shape[0]
    R = R_train.reshape(M, -1)
    N = R.shape[1] // 3
    x, g = odesc.from_R(R)
    alphas = np.random.default_rng(seed + 99).standard_normal(M * 3 * N)
    return {
        'type': 'm',
        'z': np.ones(N, dtype=np.int64),
        'R_desc': x.T.copy(),
        'R_d_desc_alpha': odesc.d_desc_dot_vec(g, alphas.reshape(M, -1)),
        'alphas_F': alphas,
        'c': 0.37,
        'std': 1.7,
        'sig': sig,
        'lam': 1e-10,
        'perms': np.asarray(perms, dtype=np.int64),
        'tril_perms_lin': odesc.tril_perms_lin(perms),
        'use_E': True,
    }


def _check_structure(H, tol_sym=1e-13, tol_sum=1e-11):
    B, n, _ = H.shape
    scale = np.max(np.abs(H))
    assert np.all(np.isfinite(H))
    assert np.max(np.abs(H - np.transpose(H, (0, 2, 1)))) <= tol_sym * scale  # exact mirror of the lower triangle
    rowsum = H.reshape(B, n, n // 3, 3).sum(axis=2)
    assert np.max(np.abs(rowsum)) < tol_sum * scale


@pytest.mark.parametrize('name,tol', [('n5_m10_s1', 1e-10), ('n9_m16_s6', 1e-10), ('n12_m8_s12', 1e-10),
                                      ('n21_m6_s6', 1e-10), ('pbc_n6_m8', 1e-9), ('ecstr_n6_m8', 1e-9)])
def test_hessian_fixtures_vs_oracle(eng, name, tol):
    """Query geometries and training geometries (n = 0 rows: w_uu is taken at its limit 0)."""
    g, model = _fixture_model(name)
    p = eng.GDMLPredict(model)
    for R in (g['R_query'][:5], g['R_train'].reshape(g['R_train'].shape[0], -1)[:3]):
        E, F, H = p.predict_hessian(R)
        H_ref = ohess.hessian(model, R)
        assert H.shape == H_ref.shape
        assert rel_err(H, H_ref) < tol
        _check_structure(H, tol_sum=1e-10)


@pytest.mark.parametrize(
    'N,M,rot,swap,sig',
    [
        (3, 5, 1, 0, 5),  # D = 3
        (9, 70, 1, 1, 20),  # D = 36 (DP 40)
        (10, 33, 0, 2, 20),  # D = 45 (DP 72)
        (12, 33, 1, 2, 30),  # D = 66 (DP 72)
        (13, 20, 1, 0, 30),  # D = 78 (DP 112)
        (15, 40, 2, 0, 30),  # D = 105 (DP 112)
        (16, 20, 1, 1, 30),  # D = 120 (DP 160)
        (18, 21, 1, 1, 40),  # D = 153 (DP 160)
        (19, 15, 0, 1, 40),  # D = 171 (DP 224)
        (21, 50, 1, 1, 20),  # D = 210 (DP 224), 3N = 63: one H tile
        (22, 12, 1, 0, 20),  # D = 231 (DP 256), 3N = 66: two tiles per side
        (23, 19, 0, 1, 20),  # D = 253 (DP 256)
        (24, 30, 1, 1, 30),  # D = 276: large-descriptor predictor
        (42, 9, 2, 0, 50),  # D = 861, 3N = 126
    ],
)
def test_hessian_shapes_vs_oracle(eng, N, M, rot, swap, sig):
    from sgdml_b200 import synth

    perms = synth.rotor_swap_group(N, rot, swap)
    model = _random_model(synth.geometries(N, M, N), perms, sig, seed=N)
    B = 5
    Rq = synth.geometries(N, B, 1).reshape(B, -1)
    E, F, H = eng.GDMLPredict(model).predict_hessian(Rq)
    assert rel_err(H, ohess.hessian(model, Rq)) < 1e-10
    _check_structure(H)


@pytest.mark.parametrize('name', ['big_c60_m2_s120', 'big_n100_m2_s12'])
def test_hessian_big_fixture_models(eng, name):
    """C60 (S = 120, 3N = 180: 3 x 3 tiles) and a 100-atom molecule (3N = 300: 5 x 5 tiles), random coefficients."""
    g = load_golden(name)
    model = _random_model(g['R_train'], g['perms'], int(g['sig']), seed=3)
    Rq = g['R_query'][:2]
    E, F, H = eng.GDMLPredict(model).predict_hessian(Rq)
    assert rel_err(H, ohess.hessian(model, Rq)) < 1e-10
    _check_structure(H)


def test_hessian_E_F_match_predict(eng):
    from sgdml_b200 import synth

    N, M = 21, 60
    model = _random_model(synth.geometries(N, M, 2), synth.rotor_swap_group(N, 1, 1), 20, seed=2)
    p = eng.GDMLPredict(model)
    for B in (1, 3, 40):
        Rq = synth.geometries(N, B, 5).reshape(B, -1)
        E, F, H = p.predict_hessian(Rq)
        E2, F2 = p.predict(Rq)
        assert rel_err(F, F2) < 1e-14 and rel_err(E, E2) < 1e-14


def test_hessian_vs_engine_central_differences(eng):
    from sgdml_b200 import synth

    N, M = 12, 40
    model = _random_model(synth.geometries(N, M, 4), synth.rotor_swap_group(N, 1, 2), 30, seed=4)
    p = eng.GDMLPredict(model)
    r = synth.geometries(N, 1, 9).reshape(-1)
    _, _, H = p.predict_hessian(r)
    h = 1e-4
    n = r.size
    _, Fp = p.predict(r[None, :] + h * np.eye(n))
    _, Fm = p.predict(r[None, :] - h * np.eye(n))
    H_fd = -((Fp - Fm) / (2 * h)).T
    assert rel_err(H[0], H_fd) < 1e-6


def _chunk_geos(N, M, S, D, Mpad):
    """Queries per workspace chunk (mirrors hessian_chunk_geos in csrc/hessian.cu)."""
    T = (3 * N + 63) // 64
    per_geo = 8 * (2 * S * Mpad + S + D + T * (T + 1) // 2 * 4096 + 9 * N * N)
    return max(1, min(65536, (256 << 20) // per_geo))


def test_hessian_batch_sizes_and_chunks(eng):
    from sgdml_b200 import synth

    N, M = 9, 3000
    perms = synth.rotor_swap_group(N, 1, 1)
    model = _random_model(synth.geometries(N, M, 6), perms, 20, seed=6)
    p = eng.GDMLPredict(model)
    S, D = perms.shape[0], N * (N - 1) // 2
    chunk = _chunk_geos(N, M, S, D, (M + 31) // 32 * 32)  # D <= 40: 32-point predictor tiles
    assert chunk < 2000
    R_all = synth.geometries(N, chunk + 1, 7).reshape(chunk + 1, -1)
    for B in (1, 2, 7):
        _, _, H = p.predict_hessian(R_all[:B])
        assert rel_err(H, ohess.hessian(model, R_all[:B])) < 1e-10
    _, _, H = p.predict_hessian(R_all)  # two chunks
    idx = [0, chunk - 1, chunk]
    assert rel_err(H[idx], ohess.hessian(model, R_all[idx])) < 1e-10
    _check_structure(H)


def test_hessian_training_geometry_is_finite(eng):
    """A query equal to a training geometry: n = 0 for its own rows."""
    from sgdml_b200 import synth

    N, M = 15, 20
    Rt = synth.geometries(N, M, 8)
    model = _random_model(Rt, synth.rotor_swap_group(N, 1, 1), 30, seed=8)
    R = Rt.reshape(M, -1)[[0, 7]]
    _, _, H = eng.GDMLPredict(model).predict_hessian(R)
    assert np.all(np.isfinite(H))
    assert rel_err(H, ohess.hessian(model, R)) < 1e-10


def test_hessian_torch_tensors(eng):
    import torch
    from sgdml_b200 import synth

    N, M = 9, 30
    model = _random_model(synth.geometries(N, M, 3), synth.rotor_swap_group(N, 1, 1), 20, seed=3)
    p = eng.GDMLPredict(model)
    Rq = synth.geometries(N, 4, 2).reshape(4, -1)
    E0, F0, H0 = p.predict_hessian(Rq)
    Rt = torch.from_numpy(Rq).cuda()
    E, F, H = p.predict_hessian(Rt)
    assert E.is_cuda and F.is_cuda and H.is_cuda and tuple(H.shape) == (4, 3 * N, 3 * N)
    assert rel_err(H.cpu().numpy(), H0) < 1e-14 and rel_err(F.cpu().numpy(), F0) < 1e-14
    out = (torch.empty(4, dtype=torch.float64, device='cuda'), torch.empty((4, 3 * N), dtype=torch.float64, device='cuda'),
           torch.empty((4, 3 * N, 3 * N), dtype=torch.float64, device='cuda'))
    res = p.predict_hessian(Rt, out=out)
    assert all(a is b for a, b in zip(res, out))
    assert rel_err(out[2].cpu().numpy(), H0) < 1e-14
    _, _, H1 = p.predict_hessian(Rt[0])  # 1-D input: one geometry
    assert tuple(H1.shape) == (1, 3 * N, 3 * N) and rel_err(H1[0].cpu().numpy(), H0[0]) < 1e-14
    E, F, H = p.predict_hessian(Rq[:0])
    assert H.shape == (0, 3 * N, 3 * N)


def test_hessian_rejects_bad_out_buffers(eng):
    import torch

    g, model = _fixture_model('n9_m16_s6')
    p = eng.GDMLPredict(model)
    R = g['R_query'][:3]
    B, n = R.shape
    good = (np.empty(B), np.empty((B, n)), np.empty((B, n, n)))
    with pytest.raises(ValueError):
        p.predict_hessian(R, out=(good[0], good[1], np.empty((B, n, n), dtype=np.float32)))
    with pytest.raises(ValueError):
        p.predict_hessian(R, out=(good[0], good[1], np.empty((B, n * n))))
    with pytest.raises(ValueError):
        p.predict_hessian(R, out=(good[0], good[1], np.empty((B, n, 2 * n))[:, :, :n]))
    with pytest.raises(ValueError):
        p.predict_hessian(R, out=(good[0], good[1], None))
    with pytest.raises(ValueError):
        p.predict_hessian(R, out=good[:2])
    with pytest.raises(ValueError):
        p.predict_hessian(torch.from_numpy(R).cuda(), out=good)
    with pytest.raises(ValueError):
        p.predict_hessian(R, out=(good[0], np.empty((B + 1, n)), good[2]))
    res = p.predict_hessian(R, out=(None, None, good[2]))  # E and F may be skipped
    assert res[2] is good[2] and rel_err(good[2], ohess.hessian(model, R)) < 1e-10


def test_hessian_large_descriptor_with_contraction_slices(eng):
    """set_contraction_slices does not apply to the Hessian: FP64 accuracy with 5 int8 slices set."""
    from sgdml_b200 import synth

    N, M = 30, 10
    model = _random_model(synth.geometries(N, M, 5), synth.rotor_swap_group(N, 1, 1), 40, seed=5)
    p = eng.GDMLPredict(model)
    p.set_contraction_slices(5)
    Rq = synth.geometries(N, 3, 6).reshape(3, -1)
    _, _, H = p.predict_hessian(Rq)
    assert rel_err(H, ohess.hessian(model, Rq)) < 1e-10


def test_compute_hessian_units(eng):
    from sgdml_b200.intf.ase_calc import _KCAL_PER_MOL_IN_EV, SGDMLCalculatorCore

    g, model = _fixture_model('n9_m16_s6')
    N = int(g['n_atoms'])
    calc = SGDMLCalculatorCore()
    E_to_eV, F_to_eV_Ang = _KCAL_PER_MOL_IN_EV, 2.0 * _KCAL_PER_MOL_IN_EV  # Ang_to_R = 2: a model in half-Angstrom
    calc._setup(model, E_to_eV, F_to_eV_Ang)
    pos = g['R_query'][0].reshape(N, 3) / 2.0  # Angstrom
    H = calc.compute_hessian(pos)
    H_ref = ohess.hessian(model, g['R_query'][0])[0] * E_to_eV * 4.0
    assert H.shape == (3 * N, 3 * N) and rel_err(H, H_ref) < 1e-10
