"""CPU: oracle/postprocess.py (the f-1 restatement every GPU post-processing test compares with) PINNED to the unmodified
reference's own post-processing code.

``tests/golden/post_<case>.npz`` hold seeded inputs and what the reference's ``ModeSolver.data_raw`` / ``ModeSolverData``
methods make of them (executed by oracle/ref_post.py in the build container, generator: tests/golden/make_post_golden.py).
Here the restatement must reproduce every stored quantity: grid-correction factors, flux, TE fraction, normalised Yee fields,
colocated fields, dot / outer_dot between neighbouring frequencies, the sorting and phases of ``overlap_sort`` and the final
(filtered, tracked) data.  Tolerance 1e-12 relative to the largest entry (measured <= 5e-14: the only differences are the
order of floating-point sums).  The ``reference``-marked tests repeat the comparison against the live reference tree.
"""
import os
import warnings

import numpy as np
import pytest

from tests import post_cases as PC

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
TOL = 1e-12


@pytest.mark.parametrize("name", list(PC.CASES))
def test_restatement_reproduces_the_reference_fixture(name):
    z = np.load(os.path.join(GOLDEN, f"post_{name}.npz"))
    c = PC.from_arrays(name, {k: z[f"in_{k}"] for k in PC.ARRAYS})
    ref = {k: z[f"ref_{k}"] for k in PC.KEYS}
    err = PC.compare(ref, PC.oracle_results(c), skip=PC.skipped_keys(c))
    assert max(err.values()) < TOL, err
    assert np.array_equal(ref["sorting"], PC.oracle_results(c)["sorting"])
    if c["track"] and c["swaps"]:  # the case really exercises a re-ordering
        assert not np.array_equal(ref["sorting"], np.tile(np.arange(c["m"]), (c["nf"], 1)))


def test_fixture_inputs_are_the_seeded_ones():
    """The stored inputs are what tests/post_cases.inputs generates (the generator and the fixtures belong together)."""
    for name in ("plain", "track_central_swap"):
        z = np.load(os.path.join(GOLDEN, f"post_{name}.npz"))
        c = PC.inputs(name)
        assert np.allclose(z["in_fields"], np.array(c["fields"]), rtol=0, atol=0) or np.allclose(z["in_fields"], np.array(c["fields"]))
        assert np.allclose(z["in_x"], c["coords"][0])


def _live():
    from oracle import ref_post

    return ref_post.available()


@pytest.mark.parametrize("name", list(PC.CASES))
def test_restatement_against_the_live_reference(name):
    """On the seeded inputs: the reference's results are computed live where its source tree is present, else read from the
    fixture it produced for these inputs (tests/golden/make_post_golden.py)."""
    c = PC.inputs(name)
    if _live():
        with warnings.catch_warnings():
            warnings.simplefilter("ignore", RuntimeWarning)
            ref = PC.reference_results(c)
    else:
        z = np.load(os.path.join(GOLDEN, f"post_{name}.npz"))
        ref = {k: z[f"ref_{k}"] for k in PC.KEYS}
    err = PC.compare(ref, PC.oracle_results(c), skip=PC.skipped_keys(c))
    assert max(err.values()) < TOL, err


@pytest.mark.reference
def test_restatement_fuzzed_against_the_live_reference():
    """40 random cases over the whole option space (tests/post_cases.random_case; 240 were run when the fixtures were made:
    tools/fuzz_reference.py): restatement == the reference's own code."""
    if not _live():
        pytest.skip("no reference tree here")
    rng = np.random.default_rng(20260924)
    for _ in range(40):
        case = PC.random_case(rng)
        PC.CASES["_fuzz"] = case
        try:
            c = PC.inputs("_fuzz")
            with warnings.catch_warnings():
                warnings.simplefilter("ignore", RuntimeWarning)
                ref = PC.reference_results(c)
            err = PC.compare(ref, PC.oracle_results(c), skip=PC.skipped_keys(c))
        finally:
            PC.CASES.pop("_fuzz")
        assert max(err.values()) < 1e-10, (case, err)


@pytest.mark.reference
def test_fixtures_are_current():
    """The committed fixtures are what the reference tree in this container produces."""
    if not _live():
        pytest.skip("no reference tree here")
    for name in ("sym_both", "grid_corr_minus", "filter_tm_track"):
        z = np.load(os.path.join(GOLDEN, f"post_{name}.npz"))
        with warnings.catch_warnings():
            warnings.simplefilter("ignore", RuntimeWarning)
            ref = PC.reference_results(PC.inputs(name))
        for k in PC.KEYS:
            assert np.allclose(z[f"ref_{k}"], ref[k], rtol=1e-13, atol=1e-15, equal_nan=True), (name, k)


@pytest.mark.reference
def test_harness_reads_the_reference_not_a_copy():
    """oracle/ref_post.py holds no method body of its own for the pinned path: every name in ``_PARTS`` is cut out of the
    reference's files at run time (a changed reference would change the result), and the repository contains none of them."""
    if not _live():
        pytest.skip("no reference tree here")
    from oracle import ref_post as RP

    src = open(RP.__file__).read()
    for rel, cls, names in (p for parts in RP._PARTS.values() for p in parts):
        for text in RP._cut(rel, cls, names):
            body = [ln.strip() for ln in text.splitlines() if len(ln.strip()) > 40 and not ln.strip().startswith(("#", '"""'))]
            assert not any(ln in src for ln in body[:5]), (rel, cls)


def test_mini_xarray_semantics():
    """The labelled-array stand-in does what xarray documents for the operations the reference's bodies use."""
    from scipy.interpolate import interp1d

    from oracle.mini_xarray import DataArray

    rng = np.random.default_rng(0)
    a = DataArray(rng.standard_normal((3, 4, 2)), coords=dict(x=[0.0, 1.0, 3.0], y=[0.0, 0.5, 1.0, 2.0], m=[0, 1]))
    w = DataArray(rng.standard_normal((4, 3)), dims=("y", "x"))
    p = a * w  # broadcasting by NAME, not by position
    assert p.dims == ("x", "y", "m") and np.allclose(p.values, a.values * w.values.T[:, :, None])
    b = DataArray(np.arange(2.0), coords=dict(m=[1, 2]))
    assert (a + b).sizes["m"] == 1 and np.allclose((a + b).values[..., 0], a.values[..., 1] + 0.0)  # inner join on labels
    s = (a * np.nan).sum(dim=("x", "y"))
    assert s.dims == ("m",) and np.all(s.values == 0.0)  # skipna
    i = a.interp(x=[0.5, 2.0, 4.0], y=[0.25], assume_sorted=True)
    ref = interp1d([0.0, 1.0, 3.0], a.values, axis=0, bounds_error=False)([0.5, 2.0, 4.0])
    ref = interp1d([0.0, 0.5, 1.0, 2.0], ref, axis=1, bounds_error=False)([0.25])
    assert np.allclose(i.values, ref, equal_nan=True) and np.isnan(i.values[2]).all()
    assert a.interp(x=0.5).dims == ("y", "m")  # a scalar drops the dimension
    n = a.sel(x=[2.9, 0.4, 0.5], method="nearest")
    assert list(n.coords["x"].values) == [3.0, 0.0, 1.0]  # ties go to the larger index (pandas)
    c = a.copy()
    c[{"x": [0, 2]}] *= -2.0
    assert np.allclose(c.values[[0, 2]], -2.0 * a.values[[0, 2]]) and np.allclose(c.values[1], a.values[1])
    d = a.copy()
    view = d.values
    d /= DataArray([1.0, 2.0], dims=("m",))
    assert d.values is view and np.allclose(view[..., 1], a.values[..., 1] / 2)  # in place: the owner sees it
    assert a.isel(m=0).dims == ("x", "y") and a.isel(m=[0]).dims == ("x", "y", "m")
    assert np.allclose(np.abs(a).values, np.abs(a.values)) and np.allclose((2 - a).values, 2 - a.values)
    assert a.squeeze(drop=True).dims == a.dims and a.isel(m=[1]).squeeze(drop=True).dims == ("x", "y")


@pytest.mark.parametrize("name", ["track_lowest", "track_central_swap", "track_highest_sym"])
def test_product_mode_tracking_on_the_reference_overlaps(name):
    """The product's host half (tidy3d_b200/postprocess.py: ``overlap_sort`` over the M x M matrices the device returns)
    fed with the reference's own ``outer_dot`` matrices reproduces the reference's sorting and phases."""
    from tidy3d_b200 import postprocess as PP

    z = np.load(os.path.join(GOLDEN, f"post_{name}.npz"))
    c = PC.from_arrays(name, {k: z[f"in_{k}"] for k in PC.ARRAYS})
    mats = [None] + list(z["ref_outer_next"])
    sorting, phase, _ = PP.overlap_sort(mats, track_freq=c["track"], direction=c["direction"])
    assert np.array_equal(sorting, z["ref_sorting"]) and np.allclose(phase, z["ref_phase"], atol=1e-12)
    n_sorted, f_sorted = PP.apply_sorting(list(z["in_n_complex"]), [f for f in np.moveaxis(z["ref_normalized_yee"], -2, 0)], sorting, phase)
    assert np.allclose(np.array(n_sorted), z["ref_final_n_complex"])
    assert np.allclose(np.stack(f_sorted, axis=-2), z["ref_final_yee"], rtol=1e-12, atol=1e-14)


@pytest.mark.parametrize("name", ["filter_te", "filter_tm_track"])
def test_product_polarisation_filter_on_the_reference_fractions(name):
    from tidy3d_b200 import postprocess as PP

    z = np.load(os.path.join(GOLDEN, f"post_{name}.npz"))
    c = PC.from_arrays(name, {k: z[f"in_{k}"] for k in PC.ARRAYS})
    if c["track"]:
        return  # the tracked order is covered by test_restatement_reproduces_the_reference_fixture
    for i in range(c["nf"]):
        order = PP.filter_polarization(z["ref_te_fraction"][i], c["filter_pol"])
        assert np.allclose(z["in_n_complex"][i][order], z["ref_final_n_complex"][i])


def test_library_tables_with_a_finite_plane_reproduce_the_reference_flux(built_lib):
    """b200ms_problem.plane_bounds (ABI v203): the integration weights the library uploads for a finite mode plane whose
    edges cut through cells (host code of csrc/api.cu, b200ms_debug_post_tables_bounded), applied in numpy to the gauge-fixed
    fields of the ``finite_plane`` fixture, give the flux the reference's ``_diff_area`` truncation gives
    (monitor_data.py:437-455) -- and differ from the untruncated weights."""
    from oracle import postprocess as OP

    z = np.load(os.path.join(GOLDEN, "post_finite_plane.npz"))
    c = PC.from_arrays("finite_plane", {k: z[f"in_{k}"] for k in PC.ARRAYS})
    pb = c["plane_bounds"]
    areas = []
    for ax, (co, n) in enumerate(zip(c["coords"], (c["nx"], c["ny"]))):
        idx, wgt, area = np.zeros(4 * (n + 1), np.int32), np.zeros(4 * (n + 1)), np.zeros(n + 1)
        P = built_lib.lib().b200ms_debug_post_tables_bounded(built_lib._ptr(np.ascontiguousarray(co)), n, 0, pb[2 * ax], pb[2 * ax + 1], n + 1,
                                                             idx.ctypes.data_as(built_lib._ip), built_lib._ptr(wgt), built_lib._ptr(area))
        assert P == n - 1
        areas.append(area[:P].copy())
    da = np.outer(*areas)
    assert np.abs(da - OP.diff_area(c["coords"], (0, 0), pb)).max() < 1e-15
    assert np.abs(da - OP.diff_area(c["coords"], (0, 0))).max() > 1e-3  # the truncation matters in this case
    for i in range(c["nf"]):
        col = OP.colocate(OP.gauge(c["fields"][i])[0], c["coords"])
        fl = np.einsum("xym,xy->m", 0.5 * np.real(col["Ex"] * np.conj(col["Hy"]) - col["Ey"] * np.conj(col["Hx"])), da)
        assert np.allclose(fl, z["ref_flux_yee"][i], rtol=1e-12)
    # the ctypes mirror carries the bounds to the struct
    from tidy3d_b200 import workloads as W

    wl = W.c1()
    pk = built_lib.PackedProblem(wl.eps_cross, wl.coords, wl.freqs[0], wl.mode_spec, plane_bounds=(-1.0, 1.2, -0.5, 0.7))
    assert [pk.struct.plane_bounds[k] for k in range(4)] == [-1.0, 1.2, -0.5, 0.7]
    assert not built_lib.PackedProblem(wl.eps_cross, wl.coords, wl.freqs[0], wl.mode_spec).struct.plane_bounds
    with pytest.raises(ValueError):
        built_lib.PackedProblem(wl.eps_cross, wl.coords, wl.freqs[0], wl.mode_spec, plane_bounds=(1.0, -1.0, 0.0, 1.0))


def test_plane_bounds_of_reads_the_plane_of_the_mode_solver():
    import types

    import tidy3d_b200.plugin as plugin

    for normal, want in ((0, [-2.0, 4.0, -0.5, 2.5]), (1, [0.5, 1.5, -0.5, 2.5]), (2, [0.5, 1.5, -2.0, 4.0])):
        size = [1.0, 6.0, 3.0]
        size[normal] = 0.0
        center = np.array([1.0, 1.0, 1.0])
        bounds = (tuple(center - np.array(size) / 2), tuple(center + np.array(size) / 2))
        ms = types.SimpleNamespace(normal_axis=normal, plane=types.SimpleNamespace(bounds=bounds))
        assert np.allclose(plugin.plane_bounds_of(ms), want)


@pytest.mark.parametrize("name", ["plain", "sym_pmc_x", "sym_pec_y", "sym_both", "one_cell_y"])
def test_product_colocate_reproduces_the_reference_colocated_data(built_lib, name):
    """``tidy3d_b200.postprocess.colocate`` (library tables) on the reference's normalised Yee-grid data == the data the
    reference's ``ModeSolver(colocate=True)`` delivers (``_colocate_data`` before ``_normalize_modes``: the two commute up to
    the flux the normalisation divides by, which is the same number), symmetry planes and a one-cell axis included."""
    from tidy3d_b200 import postprocess as PP

    z = np.load(os.path.join(GOLDEN, f"post_{name}.npz"))
    c = PC.from_arrays(name, {k: z[f"in_{k}"] for k in PC.ARRAYS})
    for i in range(c["nf"]):
        yee = z["ref_normalized_yee"][:, :, :, :, i, :][:, :, :, :, None, :]
        got, (px, py) = PP.colocate(yee, c["coords"], c["symmetry"])
        want = z["ref_colocated"][:, :, :, :, i, :]
        assert got.shape[2:4] == want.shape[2:4] == (px.size, py.size)
        assert np.abs(got[:, :, :, :, 0, :] - want).max() < 1e-12 * np.abs(want).max()


@pytest.mark.parametrize("name", ["angled", "angled_sym", "angled_sym_x", "sym_both", "plain"])
def test_device_te_fraction_arithmetic_on_the_reference_fixtures(built_lib, name):
    """The TE fraction exactly as csrc/post.cuh post_scan_kernel forms it -- colocation by the library's tables, |E1|^2 / |E2|^2
    per point by ``te_tm_terms`` (the host+device function the kernel calls, reached here through b200ms_debug_te_terms with the
    same symmetry -> cross-term rule), half-domain trapezoid weights -- on the gauge-fixed fields of the reference fixtures
    equals the reference's ``pol_fraction``, also for an angled plane WITH symmetry walls, where the reference integrates the
    symmetry-expanded plane and the products of opposite-parity components cancel."""
    from oracle import postprocess as OP
    from tidy3d_b200 import postprocess as PP

    z = np.load(os.path.join(GOLDEN, f"post_{name}.npz"))
    c = PC.from_arrays(name, {k: z[f"in_{k}"] for k in PC.ARRAYS})
    areas = []
    for co, n, s in zip(c["coords"], (c["nx"], c["ny"]), c["symmetry"]):
        idx, wgt, area = np.zeros(4 * (n + 1), np.int32), np.zeros(4 * (n + 1)), np.zeros(n + 1)
        P = built_lib.lib().b200ms_debug_post_tables(built_lib._ptr(np.ascontiguousarray(co)), n, int(s), n + 1, idx.ctypes.data_as(built_lib._ip),
                                                     built_lib._ptr(wgt), built_lib._ptr(area))
        areas.append(area[:P].copy())
    da = np.outer(*areas)
    for i in range(c["nf"]):
        g, _ = OP.gauge(c["fields"][i])
        col, _ = PP.colocate(g, c["coords"], c["symmetry"])
        te, tm = np.zeros(c["m"]), np.zeros(c["m"])
        for m in range(c["m"]):
            e = np.ascontiguousarray(np.moveaxis(col[0, :, :, :, 0, m], 0, -1))  # (Px, Py, 3)
            out = np.zeros(e.shape[:2] + (2,))
            rc = built_lib.lib().b200ms_debug_te_terms(built_lib._ptr(e.view(np.float64)), e.shape[0], e.shape[1], c["theta"], c["phi"],
                                                       int(c["symmetry"][0]), int(c["symmetry"][1]), built_lib._ptr(out))
            assert rc == 0
            te[m], tm[m] = (out[..., 0] * da).sum(), (out[..., 1] * da).sum()
        assert np.abs(te / (te + tm) - z["ref_te_fraction"][i]).max() < 1e-12, name
