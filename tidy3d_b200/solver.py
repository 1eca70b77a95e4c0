"""Host-side mirror of the reference mode-solver interface, backed by the CUDA library.

``compute_modes`` has the signature, return value and error behaviour of
``tidy3d.plugins.mode.solver.compute_modes`` (tidy3d/plugins/mode/solver.py:33-44, 941-943):

    fields, n_complex, eps_spec = compute_modes(eps_cross, coords, freq, mode_spec, symmetry=..., direction=...)

``fields`` has shape ``(2, 3, Nx, Ny, 1, num_modes)`` (E/H, component, x, y, 1, mode), ``n_complex`` is
``n_eff + 1j*k_eff`` sorted by descending ``n_eff`` and ``eps_spec`` is ``"diagonal"``, ``"tensorial_real"`` or
``"tensorial_complex"``.  ``compute_modes_batch`` is the batched entry point that corresponds to the
frequency loop of ``ModeSolver._solve_all_freqs`` (tidy3d/plugins/mode/mode_solver.py:655-672): all problems are
solved concurrently on the GPU.
"""
from __future__ import annotations

import threading
from typing import List, Optional, Sequence, Tuple

import numpy as np

from . import _cabi

_handles = {}
_hlock = threading.Lock()

# Tolerance presets.  "reference" (the default of the library) asks for what the reference asks ARPACK for
# (tol = TOL_EIGS = fp_eps, solver.py:20, 745); "tight" is the setting the parity tests use to pin n_eff to 1e-8.
TOLERANCES = {"reference": dict(eig_tol=1.1920928955078125e-07, inner_tol=1e-8), "tight": dict(eig_tol=1e-9, inner_tol=1e-10)}


def get_handle(device: int = -1, tolerance: str = "reference") -> _cabi.Handle:
    """One cached solver handle per (GPU, tolerance preset).  Calls on one handle are serialised by a per-handle lock
    (ctypes releases the GIL during the solve and the C ABI forbids overlapping calls on a handle)."""
    key = (device, tolerance)
    with _hlock:
        if key not in _handles:
            _handles[key] = _cabi.Handle(device, **TOLERANCES[tolerance])
        return _handles[key]


def _raise_for(rc: int, handle, where="", msg=None):
    msg = handle.last_error() if msg is None else msg
    if rc == _cabi.ERR_SHAPE:
        raise ValueError("Mismatch between 'coords' and 'esp_cross' shapes.")  # solver.py:107
    if rc == _cabi.ERR_NO_MODES:
        raise RuntimeError("Could not find any eigenmodes for this waveguide.")  # solver.py:876
    if rc == _cabi.ERR_UNSUPPORTED:
        raise NotImplementedError(f"tidy3d_b200: {msg}")
    if rc == _cabi.ERR_NOCONV:
        raise RuntimeError(f"tidy3d_b200: eigen-iteration did not converge {where}: {msg}")  # ArpackNoConvergence
    if rc == _cabi.ERR_CUDA:
        raise RuntimeError(f"tidy3d_b200: CUDA failure (no CPU fallback): {msg}")
    if rc != _cabi.OK:
        raise RuntimeError(f"tidy3d_b200: error {rc}: {msg}")


PEC_VAL = -1e8  # tidy3d/constants.py


def _apply_split_curl(eps_cross, split):
    """solver.py:122-124: eps_rr -> eps_rr / scaling_r outside PEC (scaling == 0 marks PEC)."""
    eps = [np.array(eps_cross[i], dtype=np.complex128, copy=True) for i in range(9)]
    for comp, idx in enumerate((0, 4, 8)):
        sc = np.asarray(split[comp])
        outside = ~np.isclose(sc, 0)
        eps[idx][outside] /= sc[outside]
    return eps


def _undo_split_curl(fields, split):
    """solver.py:904-919 applied to the packed (2,3,Nx,Ny,1,M) array: E -> E / scaling, zero inside PEC."""
    split = np.asarray(split)
    outside = ~np.isclose(split, 0)
    scale = np.where(outside, split, 1.0)
    fields[0] = (fields[0] / scale[:, :, :, None, None] * outside[:, :, :, None, None]).astype(fields.dtype)
    return fields


def _check_grad_scope(p: dict):
    """Raise NotImplementedError when the permittivity gradient of problem ``p`` is outside the diagonal path (DESIGN.md
    section 10).  What needs the rasterised medium of a ``section`` (off-diagonal or PEC-valued sites) is checked by the library."""
    ms = p["mode_spec"]
    if getattr(ms, "bend_radius", None) is not None:
        raise NotImplementedError("grad_eps: bent waveguides are not supported")
    if float(getattr(ms, "angle_theta", 0.0)) != 0.0:
        raise NotImplementedError("grad_eps: angled problems are not supported")
    for key in ("mu_cross", "split_curl_scaling", "solver_basis_fields"):
        if p.get(key) is not None:
            raise NotImplementedError(f"grad_eps: problems with {key} are not supported")
    if p.get("eps_cross") is not None:
        ec = p["eps_cross"]
        ec = ec if isinstance(ec, np.ndarray) else np.array([np.asarray(c) for c in ec])
        if np.any(np.abs(ec) >= 0.9 * abs(PEC_VAL)):
            raise NotImplementedError("grad_eps: problems with PEC-valued cells are not supported")
        if np.any(np.abs(ec[[1, 2, 3, 5, 6, 7]]) > 1e-6):  # the tensorial test of solver.py:336-339
            raise NotImplementedError("grad_eps: tensorial (off-diagonal eps) problems are not supported")


def compute_modes_batch(
    problems: Sequence[dict], device: int = -1, want_fields: bool = True, return_info: bool = False, handle=None,
    fields_ptrs=None, post: Optional[Sequence[str]] = None, grad_eps=False, grad_eps_ptrs=None,
):
    """Solve many independent mode problems in one device call.

    Each problem is a dict with the keyword arguments of ``compute_modes`` (``eps_cross, coords, freq, mode_spec``
    and optionally ``symmetry, direction``).  Problems that share the same ``eps_cross`` object are packed once.
    Returns a list of ``(fields, n_complex, eps_spec)`` tuples (``fields`` is None when ``want_fields=False``),
    plus a list of per-problem info dicts when ``return_info``.  ``fields_ptrs`` (list of raw addresses, host or device
    memory) makes the library write each problem's fields there instead (``fields`` is then None): used to keep the
    fields in HBM for the NCCL gather of ``tidy3d_b200.sharding`` / on-device post-processing.

    ``post``: on-device post-processing applied to the fields before they are delivered (``tidy3d_b200.postprocess``):
    any of ``"gauge"`` (mode_solver.py:802-810), ``"normalize"`` (flux normalisation, mode_solver.py:517-521), ``"flux"``
    (report each mode's flux and TE polarisation fraction in the info dict) and ``"overlaps"`` (M x M modal overlap matrix with the previous problem of
    the call, monitor_data.py:640-697, in the info dict as ``overlap_prev``; the input of ``postprocess.overlap_sort``).
    With ``want_fields=False`` only ``n_complex`` and these small results leave the GPU.  A problem may carry
    ``grid_correction=postprocess.grid_correction_table(...)``: flux, normalisation and overlaps then include the
    finite-grid correction factors of ``ModeSolver._grid_correction`` (mode_solver.py:847-904), like the reference's; and
    ``plane_bounds=(xmin, xmax, ymin, ymax)`` (``plugin.plane_bounds_of``): the extent of a finite mode plane, to which the
    integration weights are truncated like the reference's ``_diff_area`` (monitor_data.py:437-455).

    ``grad_eps``: True (every problem) or one bool per problem.  The info dict of such a problem then carries ``grad_eps``, an
    ndarray ``(M, 3, Nx, Ny)`` complex128 = d n_complex[m] / d eps_cross[c, c][ix, iy] for c in xx, yy, zz, from the left
    eigenvector of the diagonal operator (no extra solve; works with ``want_fields=False``).  ``grad_eps_ptrs``: one raw
    address per problem (host or device memory, 0 / None = no gradient) the library writes that array to instead.  Only the
    diagonal path is differentiable: bends, angles, off-diagonal eps, ``mu_cross``, ``split_curl_scaling``,
    ``solver_basis_fields`` and PEC-valued cells raise NotImplementedError.
    """
    post = tuple(post or ())
    if grad_eps_ptrs is not None:
        want_grad = [bool(a) for a in grad_eps_ptrs]
    elif isinstance(grad_eps, (bool, np.bool_)):
        want_grad = [bool(grad_eps)] * len(problems)
    else:
        want_grad = [bool(g) for g in grad_eps]
    if len(want_grad) != len(problems):
        raise ValueError("grad_eps / grad_eps_ptrs need one entry per problem")
    for p, g in zip(problems, want_grad):
        if g:
            _check_grad_scope(p)
    unknown = set(post) - {"gauge", "normalize", "flux", "overlaps"}
    if unknown:
        raise ValueError(f"unknown post-processing step(s): {sorted(unknown)}")
    post_flags = (1 if "gauge" in post else 0) | (2 if "normalize" in post else 0)
    packed, cache = [], {}
    for p in problems:
        split = p.get("split_curl_scaling")
        target_override = None
        if split is not None and getattr(p["mode_spec"], "target_neff", None) is None and not isinstance(p.get("eps_cross"), np.ndarray):
            # solver.py:204-207: the default target comes from `eps_cross` as passed; for a list/tuple input that is the
            # permittivity BEFORE the split-curl division (format_medium_data copies, solver.py:900)
            ec = np.array([np.asarray(c) for c in p["eps_cross"]])
            target_override = float(np.sqrt(np.max(np.abs(ec[np.abs(ec) < abs(PEC_VAL)]))))
        if split is not None and p.get("solver_basis_fields") is not None:
            raise RuntimeError("Split curl not yet implemented for relative mode solver.")  # solver.py:938
        section = p.get("section")
        if section is not None and (split is not None or p.get("eps_cross") is not None):
            raise ValueError("give either 'eps_cross' or 'section' (a section cannot be combined with split_curl_scaling)")
        key = id(p.get("eps_cross"))
        eps_in = None if section is not None else (_apply_split_curl(p["eps_cross"], split) if split is not None else p["eps_cross"])
        pk = _cabi.PackedProblem(
            eps_in, p["coords"], p["freq"], p["mode_spec"], p.get("symmetry", (0, 0)), p.get("direction", "+"),
            eps_packed=None if (split is not None or section is not None) else cache.get(key), basis_fields=p.get("solver_basis_fields"),
            section=section,
            mu_cross=p.get("mu_cross"), target_override=target_override,
            incidence=(split is not None or p.get("mu_cross") is not None),  # solver.py:93
            post=post_flags, grid_correction=p.get("grid_correction"), plane_bounds=p.get("plane_bounds"),
        )  # fmt: skip
        if split is None and section is None:
            cache[key] = pk.eps
        if section is None and key in cache and len(packed) and packed[-1].eps is pk.eps:
            # share the coordinate arrays too so the library can detect identical cross-sections
            prev = packed[-1]
            if np.array_equal(prev.cx, pk.cx) and np.array_equal(prev.cy, pk.cy):
                pk.cx, pk.cy = prev.cx, prev.cy
                pk.struct.coords_x, pk.struct.coords_y = prev.struct.coords_x, prev.struct.coords_y
        packed.append(pk)
    h = handle or get_handle(device)  # after input validation: argument errors do not need a GPU
    with h.lock:
        grad_kw = dict(grad_eps=want_grad, grad_eps_ptrs=grad_eps_ptrs) if any(want_grad) else {}
        rc, fields, ncs, results = h.solve_batch(packed, want_fields, fields_ptrs, want_flux=("flux" in post or "normalize" in post),
                                                 want_overlaps="overlaps" in post, **grad_kw)
        flux_out, te_out, ov_out = h.last_flux, h.last_te, h.last_overlaps
        grad_out = h.last_grad if grad_kw else [None] * len(packed)
        err = h.last_error() if rc != _cabi.OK else ""
    if rc != _cabi.OK:
        bad = [i for i in range(len(packed)) if results[i].status != _cabi.OK]
        _raise_for(rc, h, f"(problems {bad[:8]})", err)
    out, infos = [], []
    for i, pk in enumerate(packed):
        f = fields[i] if fields is not None else None
        if f is not None and problems[i].get("split_curl_scaling") is not None:
            f = _undo_split_curl(f, problems[i]["split_curl_scaling"])
        out.append((f, ncs[i], _cabi.SPEC_NAMES[results[i].eps_spec]))
        r = results[i]
        infos.append(
            dict(converged=r.converged, restarts=r.outer_iters, op_applies=r.op_applies, inner_iters=r.inner_iters,
                 stencil_applies=r.stencil_applies, is_complex=bool(r.is_complex), solve_ms=r.solve_ms, total_ms=r.total_ms,
                 max_residual=r.max_residual)
        )  # fmt: skip
        if flux_out:
            infos[-1]["flux"] = flux_out[i]
            infos[-1]["te_fraction"] = te_out[i]
        if ov_out:
            infos[-1]["overlap_prev"] = ov_out[i]
        if grad_out[i] is not None:
            infos[-1]["grad_eps"] = grad_out[i]
    return (out, infos) if return_info else out


def compute_modes(
    eps_cross,
    coords,
    freq,
    mode_spec,
    mu_cross=None,
    split_curl_scaling=None,
    symmetry=(0, 0),
    direction="+",
    solver_basis_fields=None,
    handle=None,
) -> Tuple[np.ndarray, np.ndarray, str]:
    """Drop-in for ``tidy3d.plugins.mode.solver.compute_modes`` (solver.py:941).  ``handle`` (not in the reference
    signature) selects a solver handle, e.g. ``get_handle(tolerance="tight")``."""
    return compute_modes_batch(
        [dict(eps_cross=eps_cross, coords=coords, freq=freq, mode_spec=mode_spec, symmetry=symmetry, direction=direction,
              solver_basis_fields=solver_basis_fields, mu_cross=mu_cross, split_curl_scaling=split_curl_scaling)],
        handle=handle,
    )[0]
