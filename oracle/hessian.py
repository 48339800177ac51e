"""Oracle (test infrastructure): analytic Hessian H = d^2 E / dR^2 of a GDML model.

The reference has no second derivatives; this is the closed form of the derivative of the forces of
``oracle.predict.Predictor._raw``.  Per permuted training row (m, p), with delta = x - X_mp, n = sqrt5 |delta|,
base = exp(-n/sig) 5/(3 sig^3), a = delta . JA_mp:

    dFd/dx = sum_mp  w_I I + w_uv (delta JA^T + JA delta^T) + w_uu delta delta^T
      w_I  = (5/sig) a base              [+ alphas_E base (n + sig)]
      w_uv = 5 base / sig
      w_uu = -25 a base / (sig^2 n)      [- alphas_E 5 base / sig]     (0 at n = 0, the limit)

and with J = dx/dR (D x 3N), u_mp = J^T delta_mp, v_mp = J^T JA_mp:

    H = -std [ (sum w_I) J^T J + sum_mp (w_uv (u v^T + v u^T) + w_uu u u^T) + sum_d Fd_d B_d ]

where B_d = d^2 x_d / dR^2: for the pair d = (a, b), r = r_a - r_b (minimum image with a lattice),
h = 3 r r^T / |r|^5 - I / |r|^3 enters the blocks (a, a) and (b, b) with +h and (a, b), (b, a) with -h.
"""

import numpy as np

from . import desc as odesc
from .predict import Predictor


def _pair_hessians(r_desc, r_d_desc):
    """h_d = 3 r r^T/|r|^5 - I/|r|^3 from x_d = 1/|r| and g_d = r/|r|^3 (so r r^T/|r|^5 = g g^T / x)."""
    gg = r_d_desc[:, :, None] * r_d_desc[:, None, :]
    return 3.0 * gg / r_desc[:, None, None] - np.eye(3)[None] * (r_desc**3)[:, None, None]


def _hessian_one(pred, x, g):
    sig = pred.sig
    sqrt5 = np.sqrt(5.0)
    base_fact = 5.0 / (3 * sig**3)
    X = pred.R_desc_perms
    JA = pred.R_d_desc_alpha_perms

    diff = x[None, :] - X
    norm = sqrt5 * np.sqrt(np.sum(diff * diff, axis=1))
    base = np.exp(-norm / sig) * base_fact
    a = np.einsum('ji,ji->j', diff, JA)
    w_I = (5.0 / sig) * a * base
    w_uv = 5.0 * base / sig
    safe = np.where(norm > 0, norm, 1.0)
    w_uu = np.where(norm > 0, -25.0 * a * base / (sig**2 * safe), 0.0)
    # descriptor-space force (as in Predictor._raw)
    Fd = w_I.dot(diff) - (base * (norm + sig)).dot(JA)
    if pred.alphas_E_lin is not None:
        ae = pred.alphas_E_lin
        Fd += ae.dot(diff * (base * (norm + sig))[:, None])
        w_I = w_I + ae * base * (norm + sig)
        w_uu = w_uu - ae * 5.0 * base / sig

    J = odesc.d_desc_from_comp(g)[0]  # (D, 3N)
    U = diff @ J  # (M*S, 3N): rows u_mp = J^T delta_mp
    V = JA @ J
    H = np.sum(w_I) * (J.T @ J)
    H += (U * w_uv[:, None]).T @ V
    H += (V * w_uv[:, None]).T @ U
    H += (U * w_uu[:, None]).T @ U

    N = pred.n_atoms
    ia, ib = odesc.tril_pairs(N)
    hd = _pair_hessians(x, g) * Fd[:, None, None]  # (D, 3, 3)
    H4 = H.reshape(N, 3, N, 3)
    np.add.at(H4, (ia, slice(None), ia, slice(None)), hd)
    np.add.at(H4, (ib, slice(None), ib, slice(None)), hd)
    np.add.at(H4, (ia, slice(None), ib, slice(None)), -hd)
    np.add.at(H4, (ib, slice(None), ia, slice(None)), -hd)
    return -pred.std * H4.reshape(3 * N, 3 * N)


def hessian(model, R, predictor=None):
    """model (reference layout), R (B, 3N) or (3N,) -> H (B, 3N, 3N) in model units (energy / length^2).
    Lattices and alphas_E are honoured as in ``oracle.predict.Predictor``."""
    pred = predictor if predictor is not None else Predictor(model)
    R = np.asarray(R, dtype=np.float64)
    if R.ndim == 1:
        R = R[None, :]
    R = R.reshape(R.shape[0], -1)
    x, g = odesc.from_R(R, pred.lat_and_inv)
    return np.array([_hessian_one(pred, xi, gi) for xi, gi in zip(x, g)])
