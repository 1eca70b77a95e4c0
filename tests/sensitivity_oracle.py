"""Exact permittivity gradients of the oracle's diagonal operator, for tests/test_sensitivity_cpu.py and test_gpu_sensitivity.py.

dlambda/deps = w^T (dA/deps) v / w^T v with the LEFT eigenvector w computed independently of the right one (dense
``scipy.linalg.eig(left=True)`` on small grids, shift-invert on A^T otherwise), A = P Q assembled by oracle/restatement.py:
  eps_xx (block (1,0) of Q holds -eps_xx):   w^T P dQ v = -(P^T w)_2 v_1
  eps_yy (block (0,1) of Q holds +eps_yy):   w^T P dQ v = +(P^T w)_1 v_2
  eps_zz (P = F iez G + mu blocks, F = [Dxf; Dyf], G = [-Dyb, Dxb]):   w^T dP Q v = -(F^T w)(G Q v) / eps_zz^2
and dn/deps = -(dlambda/deps) / (2 n), n = sqrt(-lambda) with Re n >= 0.
"""
import numpy as np
import scipy.linalg as sl
import scipy.sparse as sp
import scipy.sparse.linalg as spl

from oracle import restatement as R


def _pieces(st):
    p, q, a = R.assemble_diagonal(st)
    dxf, dxb, dyf, dyb = R.d_matrices(st)
    return p, q, a, sp.vstack([dxf, dyf]).tocsr(), sp.hstack([-dyb, dxb]).tocsr()


def grad_from_pair(st, lam, v, w, pieces=None):
    """dn/deps_{xx,yy,zz}, shape (3, nx, ny), of eigenvalue lam with right / left eigenvectors v / w (w^T A = lam w^T)."""
    p, q, _, f, g = pieces or _pieces(st)
    n = st["n"]
    y, h, wv = p.T @ w, q @ v, w @ v
    gl = np.stack([-y[n:] * v[:n], y[:n] * v[n:], -(f.T @ w) * (g @ h) / st["eps"][2, 2] ** 2]) / wv
    nc = np.sqrt(-lam + 0j)
    nc = -nc if nc.real < 0 else nc
    return (-gl / (2 * nc)).reshape(3, st["nx"], st["ny"])


def dense_modes(eps_cross, coords, freq, mode_spec, symmetry=(0, 0), k=None):
    """The k eigenpairs of A closest to the solver's shift, with exact gradients: [(lam, v, grad (3, nx, ny))], dense."""
    st = R.setup(eps_cross, coords, freq, mode_spec, symmetry)
    pieces = _pieces(st)
    lam, wl, vr = sl.eig(pieces[2].toarray(), left=True)
    sigma = -(st["target"] ** 2)
    out = []
    for i in np.argsort(np.abs(lam - sigma))[: k or mode_spec.num_modes]:
        v, w = vr[:, i], wl[:, i].conj()  # scipy's left vectors satisfy w^H A = lam w^H
        out.append((lam[i], v, grad_from_pair(st, lam[i], v, w, pieces)))
    return st, out


def sparse_grad(eps_cross, coords, freq, mode_spec, symmetry, lam0):
    """Exact gradient of the eigenvalue of A nearest lam0 (e.g. -n^2 of a device mode): right and left eigenvectors by
    shift-invert on A and A^T separately.  Returns (lam, grad (3, nx, ny))."""
    st = R.setup(eps_cross, coords, freq, mode_spec, symmetry)
    pieces = _pieces(st)
    a = pieces[2].astype(complex)
    lr, vr = spl.eigs(a, k=1, sigma=lam0, tol=1e-14)
    ll, wl = spl.eigs(a.T.tocsr(), k=1, sigma=lam0, tol=1e-14)
    assert abs(lr[0] - ll[0]) < 1e-9 * abs(lr[0])
    return lr[0], grad_from_pair(st, lr[0], vr[:, 0], wl[:, 0], pieces)


def eigenvalue_near(eps_cross, coords, freq, mode_spec, symmetry, lam0):
    """The eigenvalue of the oracle's A nearest lam0 (shift-invert, one pair)."""
    st = R.setup(eps_cross, coords, freq, mode_spec, symmetry)
    _, _, a = R.assemble_diagonal(st)
    return spl.eigs(a.astype(complex), k=1, sigma=lam0, tol=1e-14, return_eigenvectors=False)[0]
