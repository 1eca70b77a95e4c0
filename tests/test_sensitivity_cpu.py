"""CPU: the permittivity gradient dn/deps (b200ms_result.grad_eps, DESIGN.md section 10) pinned without a GPU.

* the host hook b200ms_debug_sensitivity runs the per-cell functions of the device kernel (csrc/sensitivity.cuh) on the
  oracle's right eigenvector and must reproduce w^T (dA/deps) v / w^T v built from the DENSE left eigenvector
  (tests/sensitivity_oracle.py), cell by cell, for all three components;
* that exact gradient agrees with a central finite difference of the oracle's eigenvalue;
* the ctypes Result struct mirrors the header, and every out-of-scope problem is rejected before a GPU is touched.
"""
import ctypes as C
import os
import re

import numpy as np
import pytest

from tests import sensitivity_oracle as SO
from tidy3d_b200 import workloads as W

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _case(nx=16, ny=14, pml=(0, 0), sym=(0, 0), lossy=False, nonuniform=False, aniso=False, num_modes=2):
    cx, cy = np.linspace(-1.2, 1.2, nx + 1), np.linspace(-1.0, 1.0, ny + 1)
    if nonuniform:
        g = np.linspace(-1, 1, nx + 1)
        cx = 1.2 * (0.6 * g + 0.4 * g**3)
        g = np.linspace(-1, 1, ny + 1)
        cy = 0.7 * g + 0.3 * g**3
    if nx == 1:
        cx = np.array([-0.5, 0.5])
    if ny == 1:
        cy = np.array([-0.5, 0.5])
    xm, ym = 0.5 * (cx[:-1] + cx[1:]), 0.5 * (cy[:-1] + cy[1:])
    core = (np.abs(xm)[:, None] <= 0.5) & (np.abs(ym)[None, :] <= 0.35)
    base = np.where(core, 3.48**2, 1.44**2).astype(complex) * (1 + 0.02j if lossy else 1)
    e = [base * f for f in ((1.0, 1.1, 0.9) if aniso else (1.0, 1.0, 1.0))]
    z = np.zeros((nx, ny), complex)
    ms = W.ModeSpecLike(num_modes=num_modes, num_pml=pml, target_neff=2.5)
    return [e[0], z, z, z, e[1], z, z, z, e[2]], [cx, cy], W.C_0 / 1.55, ms, sym


CASES = {
    "uniform_lossless": _case(),
    "nonuniform_aniso": _case(nonuniform=True, aniso=True),
    "pml_lossy": _case(pml=(3, 3), lossy=True),
    "pmc_min_x": _case(sym=(1, 0)),
    "pec_min_x": _case(sym=(-1, 0)),
    "pmc_pec_nonuniform_pml": _case(sym=(0, 1), pml=(3, 0), nonuniform=True, aniso=True, lossy=True),
    "slab_x1": _case(nx=1, ny=40, pml=(0, 5), num_modes=1),
    "slab_y1": _case(nx=40, ny=1, pml=(5, 0), num_modes=1),
}


def _debug_grad(cabi, eps, coords, freq, ms, sym, lam, v):
    pk = cabi.PackedProblem(eps, coords, freq, ms, sym)
    out = np.zeros((3, pk.nx, pk.ny), np.complex128)
    v = np.ascontiguousarray(v, dtype=np.complex128)
    lam = np.array([lam], np.complex128)
    rc = cabi.lib().b200ms_debug_sensitivity(C.byref(pk.struct), cabi._ptr(v.view(np.float64)), cabi._ptr(lam.view(np.float64)),
                                              cabi._ptr(out.view(np.float64)))  # fmt: skip
    return rc, out


@pytest.mark.parametrize("name", list(CASES))
def test_host_kernel_functions_match_the_exact_discrete_gradient(built_lib, name):
    eps, coords, freq, ms, sym = CASES[name]
    _, modes = SO.dense_modes(eps, coords, freq, ms, sym)
    for lam, v, g in modes:
        rc, got = _debug_grad(built_lib, eps, coords, freq, ms, sym, lam, v)
        assert rc == built_lib.OK
        scale = np.abs(g).max()
        for c in range(3):
            assert np.abs(got[c] - g[c]).max() <= 1e-9 * scale, (name, c, np.abs(got[c] - g[c]).max() / scale)


@pytest.mark.parametrize("name", ["uniform_lossless", "pml_lossy", "pmc_min_x", "slab_y1"])
def test_exact_gradient_matches_finite_differences(name):
    eps, coords, freq, ms, sym = CASES[name]
    _, modes = SO.dense_modes(eps, coords, freq, ms, sym, k=1)
    lam, _, g = modes[0]
    n0 = np.sqrt(-lam + 0j)
    nx, ny = eps[0].shape
    cells = [(nx // 2, ny // 2), (max(nx // 2 - 2, 0), ny // 2), (0, 0), (nx - 1, ny - 1)]
    for comp, idx in enumerate((0, 4, 8)):
        for cell in cells:
            d = 1e-4 * abs(eps[idx][cell])
            ns = []
            for s in (+1, -1):
                e2 = [a.copy() for a in eps]
                e2[idx][cell] += s * d
                l2 = SO.eigenvalue_near(e2, coords, freq, ms, sym, lam)
                ns.append(np.sqrt(-l2 + 0j))
            fd = (ns[0] - ns[1]) / (2 * d)
            ref = g[comp][cell]
            if abs(ref) < 1e-3 * np.abs(g).max():  # the difference of two eigenvalues is roundoff there
                continue
            assert abs(fd - ref) <= 1e-5 * abs(ref), (name, comp, cell, fd, ref)
    assert n0.real > 0


def test_result_struct_matches_the_header(built_lib):
    text = open(os.path.join(ROOT, "include", "b200ms.h")).read()
    body = text[text.index("typedef struct {\n  double *fields;") : text.index("} b200ms_result;")]
    names = re.findall(r"^\s+(?:double|int)\s+\*?(\w+);", body, flags=re.M)
    assert names == [n for n, _ in built_lib.Result._fields_]
    assert names[-1] == "grad_eps"


def _problem(**kw):
    wl = W.si_strip(24, 2)
    p = dict(eps_cross=wl.eps_cross, coords=wl.coords, freq=float(wl.freqs[0]), mode_spec=wl.mode_spec)
    p.update(kw)
    return p


def _bent():
    p = _problem()
    p["mode_spec"] = W.ModeSpecLike(num_modes=2, bend_radius=5.0, bend_axis=1)
    return p


def _angled():
    p = _problem()
    p["mode_spec"] = W.ModeSpecLike(num_modes=2, angle_theta=0.2)
    return p


def _with_pec():
    p = _problem()
    e = [a.copy() for a in p["eps_cross"]]
    e[0][0, 0] = -1e8
    p["eps_cross"] = e
    return p


def _offdiag():
    p = _problem()
    e = [a.copy() for a in p["eps_cross"]]
    e[1] = 0.05 * e[0]
    p["eps_cross"] = e
    return p


OUT_OF_SCOPE = {
    "bend": _bent,
    "angled": _angled,
    "pec_cell": _with_pec,
    "tensorial": _offdiag,
    "mu_cross": lambda: _problem(mu_cross=[np.ones((24, 24), complex) if i in (0, 4, 8) else np.zeros((24, 24), complex) for i in range(9)]),
    "split_curl": lambda: _problem(split_curl_scaling=np.ones((3, 24, 24))),
    "basis_fields": lambda: _problem(solver_basis_fields=np.zeros((6, 24, 24, 1, 2), complex)),
}


@pytest.mark.parametrize("name", list(OUT_OF_SCOPE))
def test_out_of_scope_problems_raise_before_the_gpu(monkeypatch, name):
    from tidy3d_b200 import solver

    def no_gpu(*a, **k):
        raise AssertionError("a GPU handle was requested")

    monkeypatch.setattr(solver, "get_handle", no_gpu)
    ok = _problem()
    with pytest.raises(NotImplementedError):
        solver.compute_modes_batch([ok, OUT_OF_SCOPE[name]()], want_fields=False, return_info=True, grad_eps=True)
    with pytest.raises(NotImplementedError):  # only the problem that asks for the gradient is checked
        solver.compute_modes_batch([ok, OUT_OF_SCOPE[name]()], want_fields=False, return_info=True, grad_eps=[False, True])


def test_host_hook_rejects_out_of_scope_problems(built_lib):
    for make in (_bent, _with_pec, _offdiag):
        p = make()
        pk = built_lib.PackedProblem(p["eps_cross"], p["coords"], p["freq"], p["mode_spec"])
        v = np.zeros(2 * pk.nx * pk.ny, np.complex128)
        out = np.zeros(3 * pk.nx * pk.ny, np.complex128)
        lam = np.array([-4.0 + 0j])
        rc = built_lib.lib().b200ms_debug_sensitivity(C.byref(pk.struct), built_lib._ptr(v.view(np.float64)), built_lib._ptr(lam.view(np.float64)),
                                                      built_lib._ptr(out.view(np.float64)))  # fmt: skip
        assert rc == built_lib.ERR_UNSUPPORTED
