"""CPU: the oracle restatement is pinned to the reference -- golden fixtures (generated from the unmodified
reference), the reference's own exact known-answer test, and, in the build container, the reference itself."""
import os

import numpy as np
import pytest

from oracle import ref_shim
from oracle import restatement as R
from tests.golden.cases import CASES, resolve_kwargs
from tests.helpers import load_golden, mode_overlaps, signature

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

FAST = ["c1_64", "c1_64_minus", "c1_64_sym_pmc_pec", "lossy_48", "nonuniform_56", "slab1d_x1", "slab1d_y1",
        "angled_48_minus", "angled_phi_48", "offdiag_48", "c3_96", "c4_96", "c4_96_axis0", "strip_128_m4", "pec_block_40", "lossy_angled_40", "lossy_angled_40_minus", "angle_bend_44",
        "mu_cross_40", "split_curl_40", "pec_split_40"]  # fmt: skip


@pytest.mark.parametrize("name", FAST)
def test_restatement_matches_golden(name):
    fac, kw, _ = CASES[name]
    wl = fac()
    kw = resolve_kwargs(wl, kw)
    g = load_golden(name)
    fields, n, spec = R.compute_modes(wl.eps_cross, wl.coords, wl.freqs[0], wl.mode_spec, **kw)
    assert spec == str(g["spec"])
    # same algorithm, same ARPACK tolerance (1.19e-7) and start vector: agreement well below that tolerance (the
    # reference's incidence-matrix products change the rounding of the split-curl / mu_cross cases: 3e-9 there)
    assert np.abs(n - g["n_ref"]).max() < 2e-8
    assert np.abs(signature(fields) - g["sig_ref"]).max() < 1e-4
    if "fields_tight" in g.files:
        ft, nt, _ = R.compute_modes(wl.eps_cross, wl.coords, wl.freqs[0], wl.mode_spec, tol=1e-12, **kw)
        assert np.abs(nt - g["n_tight"]).max() < 1e-10
        gaps = np.abs(nt[:, None] - nt[None, :]) + np.eye(nt.size)
        ok = gaps.min(axis=1) > 1e-4  # per-mode overlap is only meaningful for isolated modes
        assert (mode_overlaps(ft, g["fields_tight"])[ok] > 1 - 1e-6).all()


def test_relative_solver_restatement_matches_golden():
    from tests.golden.cases import relative_case

    wl = relative_case()
    g = load_golden("relative_48")
    f, n, spec = R.compute_modes(wl.eps_cross, wl.coords, wl.freqs[0], wl.mode_spec, solver_basis_fields=g["basis"])
    assert spec == str(g["spec"]) and np.abs(n - g["n_ref"]).max() < 1e-12
    assert (mode_overlaps(f, g["fields_tight"]) > 1 - 1e-10).all()


def test_pml_profile_known_answer():
    """Restates the reference's own exact test ``test_pml_params`` (tests/test_plugins/test_mode_solver.py:783-806)."""
    omega, n, npml = 1.0, 10, 4
    dls = np.ones(n)
    sf = R.sfactor("f", omega, dls, n, npml, True, (1.0, 1.0))
    sb = R.sfactor("b", omega, dls, n, npml, True, (1.0, 1.0))
    k = lambda step: 1 + 2 * step**3  # noqa: E731
    s = lambda step: 2 * step**3 / (R.ETA_0 * R.EPSILON_0)  # noqa: E731
    # forward profile: half-integer steps, backward: integer steps
    for i, step in zip(range(npml), [(npml - i - 0.5) / npml for i in range(npml)]):
        assert np.isclose(sf[i], k(step) + 1j * s(step))
    for i, step in zip(range(npml), [(npml - i) / npml for i in range(npml)]):
        assert np.isclose(sb[i], k(step) + 1j * s(step))
    for i in range(n - npml, n):
        assert np.isclose(sf[i], k((i - (n - npml) + 0.5) / npml) + 1j * s((i - (n - npml) + 0.5) / npml))
    assert np.allclose(sf[npml : n - npml], 1) and np.allclose(sb[npml : n - npml + 1], 1)


def test_matrix_free_model_equals_assembled_operator():
    """The radius-1 matrix-free form that the CUDA stencil implements equals P.Q (solver.py:479-490)."""
    for name in ["c1_64", "c3_96", "c4_96", "nonuniform_56", "lossy_48"]:
        fac, kw, _ = CASES[name]
        wl = fac()
        st = R.setup(wl.eps_cross, wl.coords, wl.freqs[0], wl.mode_spec, kw.get("symmetry", (0, 0)))
        _, _, A = R.assemble_diagonal(st)
        rng = np.random.default_rng(0)
        v = rng.standard_normal(2 * st["n"]) + 1j * rng.standard_normal(2 * st["n"])
        y0 = A @ v
        y1 = R.apply_diagonal_matrix_free(st, v)
        assert np.abs(y0 - y1).max() / np.abs(y0).max() < 1e-12


@pytest.mark.parametrize("name", ["c1_64", "c1_64_sym_pmc_pec", "lossy_48", "nonuniform_56", "angled_48_minus", "offdiag_48", "c4_96"])
def test_restatement_matches_live_reference(name):
    """The reference's result is computed live where its source tree (or oracle/_ref) is present, else read from the golden
    fixture it produced (tests/golden/make_golden.py: same inputs, same call)."""
    fac, kw, _ = CASES[name]
    wl = fac()
    if ref_shim.available():
        f0, n0, s0 = ref_shim.compute_modes(wl.eps_cross, wl.coords, wl.freqs[0], wl.mode_spec, **kw)
        sig0 = signature(f0)
    else:
        g = load_golden(name)
        n0, sig0, s0 = g["n_ref"], g["sig_ref"], str(g["spec"])
    f1, n1, s1 = R.compute_modes(wl.eps_cross, wl.coords, wl.freqs[0], wl.mode_spec, **kw)
    assert s0 == s1
    assert np.abs(n0 - n1).max() < 1e-10
    assert np.abs(sig0 - signature(f1)).max() < 1e-5


@pytest.mark.reference
@pytest.mark.skipif(not ref_shim.available(), reason="reference tree not present (GPU box)")
def test_reference_pml_factors_match():
    """create_sfactor_f/b of the unmodified reference vs the restatement on a graded PML case."""
    import importlib

    ref_shim.load()
    der = importlib.import_module("tidy3d.plugins.mode.derivatives")
    dls = np.linspace(0.01, 0.02, 30)
    for n_pml in (0, 5, 12):
        for dmin in (True, False):
            if n_pml == 0:
                continue
            a = der.create_sfactor_f(2e15, dls, 30, n_pml, dmin, (0.6, 0.7))
            b = R.sfactor("f", 2e15, dls, 30, n_pml, dmin, (0.6, 0.7))
            assert np.allclose(a, b, rtol=1e-14)
            a = der.create_sfactor_b(2e15, dls, 30, n_pml, dmin, (0.6, 0.7))
            b = R.sfactor("b", 2e15, dls, 30, n_pml, dmin, (0.6, 0.7))
            assert np.allclose(a, b, rtol=1e-14)


def test_built_reference_loads_without_the_source_tree(tmp_path):
    """oracle/_ref (byte-compiled by oracle/build_ref.py) is the reference itself: loaded with /root/reference hidden, in a
    clean interpreter, it reproduces the golden made from the source tree to the last bit of the ARPACK run."""
    import json
    import subprocess
    import sys

    from oracle import build_ref

    if not build_ref.build():
        pytest.skip("no reference tree here and no oracle/_ref shipped")
    man = json.load(open(build_ref.manifest_path()))
    assert set(man["sha256"]) == set(build_ref.FILES)
    if ref_shim.source_available():  # build container: the byte code was made from exactly the files under /root/reference
        import hashlib

        for f, sha in man["sha256"].items():
            assert hashlib.sha256(open(os.path.join(ref_shim.REF_ROOT, "tidy3d", f), "rb").read()).hexdigest() == sha
    code = (
        "import numpy as np, sys\n"
        "from oracle import ref_shim\n"
        "from tests.golden.cases import CASES\n"
        "assert ref_shim.origin() == 'built', ref_shim.origin()\n"
        "fac, kw, _ = CASES['c1_64']\n"
        "wl = fac()\n"
        "f, n, s = ref_shim.compute_modes(wl.eps_cross, wl.coords, wl.freqs[0], wl.mode_spec, **kw)\n"
        "assert sys.modules['tidy3d.plugins.mode.solver'].__file__.endswith('.pyc')\n"
        "np.save(sys.argv[1], n)\n"
    )
    out = str(tmp_path / "n.npy")
    env = dict(os.environ, B200MS_REFERENCE=str(tmp_path / "no_reference_here"), PYTHONPATH=ROOT)
    subprocess.run([sys.executable, "-c", code, out], check=True, cwd=ROOT, env=env, timeout=300)
    g = np.load(os.path.join(ROOT, "tests", "golden", "c1_64.npz"))
    assert np.abs(np.load(out) - g["n_ref"]).max() < 1e-12
