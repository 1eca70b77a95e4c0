"""ctypes binding of ``libb200ms.so`` (C ABI declared in ``include/b200ms.h``).

This is the only way the Python layer reaches the solver; there is no Python/NumPy compute path.  If the
shared library is missing the import of this module raises (build it with ``python -c "import
__graft_entry__ as g; g.build()"``), and if no CUDA device is usable ``Handle()`` raises -- the product
never falls back to the CPU.
"""
from __future__ import annotations

import ctypes as C
import math
import os
import threading

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("B200MS_LIB") or os.path.join(_HERE, "libb200ms.so")  # B200MS_LIB: developer override (A/B of builds)

ABI_VERSION = 205  # B200MS_VERSION of include/b200ms.h
OK, ERR_SHAPE, ERR_NO_MODES, ERR_UNSUPPORTED, ERR_CUDA, ERR_NOCONV, ERR_ARG = range(7)
SPEC_NAMES = {0: "diagonal", 1: "tensorial_real", 2: "tensorial_complex"}

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)


class SectionStruct(C.Structure):
    _fields_ = [("nrect", C.c_int), ("rects", _dp), ("medium", _ip), ("nmedia", C.c_int), ("eps_table", _dp),
                ("shape", _ip), ("poly_start", _ip), ("poly_xy", _dp), ("site_medium", C.POINTER(C.c_ushort))]


class Problem(C.Structure):
    _fields_ = [
        ("nx", C.c_int), ("ny", C.c_int), ("num_modes", C.c_int), ("num_pml", C.c_int * 2),
        ("symmetry", C.c_int * 2), ("bend_axis", C.c_int), ("direction", C.c_int), ("precision", C.c_int), ("incidence", C.c_int), ("post", C.c_int),
        ("freq", C.c_double), ("target_neff", C.c_double), ("bend_radius", C.c_double),
        ("angle_theta", C.c_double), ("angle_phi", C.c_double),
        ("eps", _dp), ("coords_x", _dp), ("coords_y", _dp), ("mu", _dp), ("section", C.POINTER(SectionStruct)), ("basis_e", _dp),
        ("grid_correction", _dp), ("plane_bounds", _dp),
    ]  # fmt: skip


class Result(C.Structure):
    _fields_ = [
        ("fields", _dp), ("n_complex", _dp), ("flux", _dp), ("te_fraction", _dp), ("overlap_prev", _dp), ("eps_spec", C.c_int), ("status", C.c_int), ("converged", C.c_int),
        ("outer_iters", C.c_int), ("op_applies", C.c_int), ("inner_iters", C.c_int), ("stencil_applies", C.c_int),
        ("is_complex", C.c_int), ("solve_ms", C.c_double), ("total_ms", C.c_double), ("max_residual", C.c_double),
        ("grad_eps", _dp),
    ]  # fmt: skip


class Options(C.Structure):
    _fields_ = [
        ("eig_tol", C.c_double), ("inner_tol", C.c_double), ("ncv", C.c_int), ("max_restarts", C.c_int),
        ("gmres_restart", C.c_int), ("gmres_maxit", C.c_int), ("mg_nu", C.c_int), ("mg_min_size", C.c_int),
        ("mg_coarse_iters", C.c_int), ("max_batch", C.c_int), ("mg_omega", C.c_double), ("mg_ppw", C.c_double),
        ("verbose", C.c_int), ("mg_pml_phase", C.c_double), ("inner_relax", C.c_double), ("inner_relax_cap", C.c_double), ("gmres_cgs2", C.c_int), ("mg_nu_growth", C.c_int), ("use_graph", C.c_int), ("mg_cycles", C.c_int),
        ("inner_ir", C.c_int), ("ir_floor", C.c_double), ("ir_trust", C.c_double), ("inner_relax_complex", C.c_double), ("mg_fuse_first", C.c_int), ("ks_keep", C.c_int), ("cluster_gap", C.c_double), ("mg_fused_tail", C.c_int), ("kappa_cap", C.c_double), ("outer_dgks", C.c_int), ("stencil_pair", C.c_int), ("stencil_pair_rows", C.c_int), ("transfer_vec", C.c_int), ("tensor_mg_cycles", C.c_int),
    ]  # fmt: skip


class Stats(C.Structure):
    _fields_ = [
        ("device_ms", C.c_double), ("setup_ms", C.c_double), ("download_ms", C.c_double), ("total_ms", C.c_double),
        ("launches", C.c_longlong), ("inner_iters", C.c_longlong), ("op_applies", C.c_longlong), ("host_syncs", C.c_longlong),
        ("device_batches", C.c_int), ("nprob", C.c_int),
    ]  # fmt: skip


EXPORTS = [
    "b200ms_version", "b200ms_get_stats", "b200ms_default_options", "b200ms_create", "b200ms_destroy", "b200ms_set_options",
    "b200ms_last_error", "b200ms_host_alloc", "b200ms_host_free", "b200ms_solve_batch", "b200ms_bench_stencil", "b200ms_debug_schur", "b200ms_debug_setup",
    "b200ms_debug_hierarchy", "b200ms_debug_apply", "b200ms_debug_vcycle", "b200ms_debug_solve", "b200ms_debug_march2_geometry", "b200ms_debug_post_tables", "b200ms_debug_post_tables_bounded", "b200ms_debug_te_terms", "b200ms_debug_grid_factors",
    "b200ms_debug_sensitivity",
]  # fmt: skip

_lib = None
_lock = threading.Lock()


def lib():
    """Load the shared library (raises OSError with a build hint if it is missing)."""
    global _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise OSError(
                    f"{LIB_PATH} not found: the CUDA library is not built. Run `python -c \"import __graft_entry__ "
                    'as g; g.build()"` at the repo root. tidy3d_b200 has no CPU fallback.'
                )
            L = C.CDLL(LIB_PATH)
            L.b200ms_version.restype = C.c_int
            if L.b200ms_version() != ABI_VERSION:  # the ctypes structs below mirror include/b200ms.h of exactly this version
                raise OSError(
                    f"{LIB_PATH} implements ABI version {L.b200ms_version()}, this package expects {ABI_VERSION}: rebuild it "
                    '(`python -c "import __graft_entry__ as g; g.build()"` at the repo root)'
                )
            L.b200ms_default_options.argtypes = [C.POINTER(Options)]
            L.b200ms_default_options.restype = None
            L.b200ms_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
            L.b200ms_destroy.argtypes = [C.c_void_p]
            L.b200ms_set_options.argtypes = [C.c_void_p, C.POINTER(Options)]
            L.b200ms_last_error.argtypes = [C.c_void_p]
            L.b200ms_last_error.restype = C.c_char_p
            L.b200ms_get_stats.argtypes = [C.c_void_p, C.POINTER(Stats)]
            L.b200ms_host_alloc.argtypes = [C.c_size_t]
            L.b200ms_host_alloc.restype = C.c_void_p
            L.b200ms_host_free.argtypes = [C.c_void_p]
            L.b200ms_host_free.restype = None
            L.b200ms_solve_batch.argtypes = [C.c_void_p, C.c_int, C.POINTER(Problem), C.POINTER(Result)]
            L.b200ms_bench_stencil.argtypes = [C.c_void_p, C.POINTER(Problem), C.c_int, C.c_int, C.c_int, C.c_int, _dp, _dp, _dp, _dp]
            L.b200ms_debug_schur.argtypes = [C.c_int, _dp, _dp, _dp]
            L.b200ms_debug_setup.argtypes = [C.POINTER(Problem), _dp, _ip, _dp, _dp, _dp, _dp, _dp]
            L.b200ms_debug_hierarchy.argtypes = [C.POINTER(Problem), C.POINTER(Options), C.c_int, _ip]
            L.b200ms_debug_apply.argtypes = [C.c_void_p, C.POINTER(Problem), C.c_int, C.c_int, _dp, _dp, _dp]
            L.b200ms_debug_vcycle.argtypes = [C.c_void_p, C.POINTER(Problem), _dp, _dp]
            L.b200ms_debug_solve.argtypes = [C.c_void_p, C.POINTER(Problem), _dp, _dp, _ip, _dp]
            L.b200ms_debug_march2_geometry.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, _ip, _ip, _ip]
            L.b200ms_debug_post_tables.argtypes = [_dp, C.c_int, C.c_int, C.c_int, _ip, _dp, _dp]
            L.b200ms_debug_post_tables_bounded.argtypes = [_dp, C.c_int, C.c_int, C.c_double, C.c_double, C.c_int, _ip, _dp, _dp]
            L.b200ms_debug_te_terms.argtypes = [_dp, C.c_int, C.c_int, C.c_double, C.c_double, C.c_int, C.c_int, _dp]
            L.b200ms_debug_grid_factors.argtypes = [C.POINTER(Problem), _dp, _dp, _dp]
            L.b200ms_debug_sensitivity.argtypes = [C.POINTER(Problem), _dp, _dp, _dp]
            _lib = L
    return _lib


def _ptr(a):
    return a.ctypes.data_as(_dp)


class PackedProblem:
    """Owns the contiguous arrays a ``Problem`` struct points to."""

    def __init__(self, eps_cross, coords, freq, mode_spec, symmetry=(0, 0), direction="+", eps_packed=None, basis_fields=None,
                 mu_cross=None, target_override=None, incidence=False, post=0, section=None, grid_correction=None, plane_bounds=None):
        self.section = None
        if section is not None:  # geometric cross-section rasterised on the device (tidy3d_b200/sections.py); no eps array
            self.section, self._section_arrays = section.pack(float(freq), (len(coords[0]) - 1, len(coords[1]) - 1))
            eps = None
        elif eps_packed is not None:
            eps = eps_packed
        elif isinstance(eps_cross, np.ndarray) and eps_cross.dtype == np.complex128 and eps_cross.flags.c_contiguous and eps_cross.ndim == 3:
            # what ModeSolver._solver_eps returns (mode_solver.py:647-653): used in place, no host copy
            if eps_cross.shape[0] != 9:
                raise ValueError("Wrong input to mode solver pemittivity/permeability!")
            eps = eps_cross
        else:
            if isinstance(eps_cross, np.ndarray):
                if eps_cross.shape[0] != 9:
                    raise ValueError("Wrong input to mode solver pemittivity/permeability!")
                comps = [eps_cross[i] for i in range(9)]
            else:
                if len(eps_cross) != 9:
                    raise ValueError("Wrong input to mode solver pemittivity/permeability!")
                comps = list(eps_cross)
            eps = np.ascontiguousarray(np.stack([np.asarray(c, dtype=np.complex128) for c in comps]))
        self.cx = np.ascontiguousarray(coords[0], dtype=np.float64)
        self.cy = np.ascontiguousarray(coords[1], dtype=np.float64)
        if eps is None:
            self.nx, self.ny = self.cx.size - 1, self.cy.size - 1
        else:
            if eps.ndim != 3:
                raise ValueError("Wrong input to mode solver pemittivity/permeability!")
            self.nx, self.ny = eps.shape[1], eps.shape[2]
        self.eps = eps
        if self.cx.size != self.nx + 1 or self.cy.size != self.ny + 1:
            raise ValueError("Mismatch between 'coords' and 'esp_cross' shapes.")
        p = Problem()
        p.nx, p.ny = self.nx, self.ny
        p.num_modes = int(mode_spec.num_modes)
        npml = getattr(mode_spec, "num_pml", (0, 0))
        p.num_pml[0], p.num_pml[1] = int(npml[0]), int(npml[1])
        p.symmetry[0], p.symmetry[1] = int(symmetry[0]), int(symmetry[1])
        br = getattr(mode_spec, "bend_radius", None)
        p.bend_radius = math.nan if br is None else float(br)
        ba = getattr(mode_spec, "bend_axis", None)
        p.bend_axis = -1 if ba is None else int(ba)
        p.direction = -1 if direction == "-" else 1
        p.precision = 1 if getattr(mode_spec, "precision", "single") == "single" else 0
        p.incidence = 1 if incidence else 0
        p.post = int(post)
        p.freq = float(freq)
        tn = getattr(mode_spec, "target_neff", None) if target_override is None else target_override
        p.target_neff = math.nan if tn is None else float(tn)
        p.angle_theta = float(getattr(mode_spec, "angle_theta", 0.0))
        p.angle_phi = float(getattr(mode_spec, "angle_phi", 0.0))
        p.coords_x, p.coords_y = _ptr(self.cx), _ptr(self.cy)
        if self.eps is not None:
            p.eps = _ptr(self.eps.view(np.float64))
        else:
            p.section = C.pointer(self.section)
        self.mu = None
        if mu_cross is not None:
            if isinstance(mu_cross, np.ndarray):
                mcomps = [mu_cross[i] for i in range(9)]
            else:
                if len(mu_cross) != 9:
                    raise ValueError("Wrong input to mode solver pemittivity/permeability!")
                mcomps = list(mu_cross)
            self.mu = np.ascontiguousarray(np.stack([np.asarray(c, dtype=np.complex128) for c in mcomps]))
            if self.mu.shape != (9, self.nx, self.ny):
                raise ValueError("Wrong input to mode solver pemittivity/permeability!")
            p.mu = _ptr(self.mu.view(np.float64))
        self.basis = None
        if basis_fields is not None:
            try:  # solver.py:222-230
                b = np.asarray(basis_fields)[:3, ...].reshape((3, self.nx * self.ny, p.num_modes))
            except ValueError:
                raise ValueError(
                    "Shape mismatch between 'basis_fields' and requested mode data. "
                    "Make sure the mode solvers are set up the same, and that the "
                    "basis mode solver data has 'colocate=False'."
                )
            self.basis = np.ascontiguousarray(b[:2], dtype=np.complex128)
            p.basis_e = _ptr(self.basis.view(np.float64))
        self.grid_correction = None
        if grid_correction is not None:  # 8 numbers, see tidy3d_b200.postprocess.grid_correction_table / b200ms_problem.grid_correction
            self.grid_correction = np.ascontiguousarray(grid_correction, dtype=np.float64).ravel()
            if self.grid_correction.size != 8:
                raise ValueError("grid_correction must hold 8 numbers (postprocess.grid_correction_table)")
            p.grid_correction = _ptr(self.grid_correction)
        self.plane_bounds = None
        if plane_bounds is not None:  # (xmin, xmax, ymin, ymax) of a finite mode plane, see b200ms_problem.plane_bounds
            self.plane_bounds = np.ascontiguousarray(plane_bounds, dtype=np.float64).ravel()
            if self.plane_bounds.size != 4 or not (self.plane_bounds[0] <= self.plane_bounds[1] and self.plane_bounds[2] <= self.plane_bounds[3]):
                raise ValueError("plane_bounds must be (xmin, xmax, ymin, ymax)")
            p.plane_bounds = _ptr(self.plane_bounds)
        self.struct = p
        self.num_modes = p.num_modes


class PinnedPool:
    """Recycling pool of page-locked host buffers for the field results (D2H at full link speed, no first-touch page
    faults).  A buffer returns to the pool when the numpy array built on it (and every view of it) is garbage
    collected; at most ``max_cached`` bytes are kept, the rest is freed."""

    def __init__(self, max_cached=int(os.environ.get("B200MS_PINNED_CACHE_GB", "48")) << 30):
        self.free = {}
        self.cached = 0
        self.max_cached = max_cached
        self._lock = threading.Lock()

    def empty(self, shape, dtype=np.complex128):
        import weakref

        nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
        with self._lock:
            lst = self.free.get(nbytes)
            ptr = lst.pop() if lst else None
            if ptr is not None:
                self.cached -= nbytes
        if ptr is None:
            ptr = lib().b200ms_host_alloc(nbytes)
            if not ptr:
                return np.empty(shape, dtype=dtype)  # pinned allocation failed: ordinary pageable memory still works
        raw = (C.c_char * nbytes).from_address(ptr)
        weakref.finalize(raw, self._release, ptr, nbytes)
        return np.frombuffer(raw, dtype=dtype).reshape(shape)

    def _release(self, ptr, nbytes):
        with self._lock:
            if self.cached + nbytes <= self.max_cached:
                self.free.setdefault(nbytes, []).append(ptr)
                self.cached += nbytes
                return
        try:
            lib().b200ms_host_free(ptr)
        except Exception:  # noqa: BLE001  (interpreter shutdown)
            pass


_pool = PinnedPool()


class Handle:
    """One solver handle == one GPU (``b200ms_create`` / ``b200ms_destroy``)."""

    def __init__(self, device: int = -1, **options):
        self._h = C.c_void_p()
        self.lock = threading.Lock()
        rc = lib().b200ms_create(device, C.byref(self._h))
        if rc != OK:
            raise RuntimeError(
                "b200ms_create failed: no usable CUDA device (tidy3d_b200 is GPU-only, there is no CPU fallback)"
            )
        self.options = Options()
        lib().b200ms_default_options(C.byref(self.options))
        if options:
            self.set_options(**options)

    def set_options(self, **kw):
        for k, v in kw.items():
            if not hasattr(self.options, k):
                raise AttributeError(f"unknown solver option {k!r}")
            setattr(self.options, k, v)
        lib().b200ms_set_options(self._h, C.byref(self.options))

    def last_error(self) -> str:
        return lib().b200ms_last_error(self._h).decode()

    def last_stats(self) -> dict:
        """Counters of the most recent solve_batch call on this handle (b200ms_get_stats)."""
        st = Stats()
        lib().b200ms_get_stats(self._h, C.byref(st))
        return {k: getattr(st, k) for k, _ in Stats._fields_}

    def close(self):
        if self._h:
            lib().b200ms_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def solve_batch(self, packed, want_fields=True, fields_ptrs=None, want_flux=False, want_overlaps=False, grad_eps=None,
                    grad_eps_ptrs=None):
        """packed: list of PackedProblem.  Returns (rc, fields list | None, n_complex list, Result structs).

        ``fields_ptrs``: optional list of raw addresses (host or DEVICE memory, e.g. ``tensor.data_ptr()``) the library
        writes the fields of each problem to, instead of freshly allocated pinned host arrays; then ``fields`` is None.
        Fields are complex128, or complex64 for ``precision == "single"`` problems (solver.py:265-267).

        ``grad_eps``: optional list of bools, one per problem: allocate a (M, 3, Nx, Ny) complex128 array for dn/deps of that
        problem (``self.last_grad``, None where not asked).  ``grad_eps_ptrs``: list of raw addresses (host or device, 0 = none)
        the library writes the gradient to instead."""
        n = len(packed)
        probs = (Problem * n)(*[p.struct for p in packed])
        results = (Result * n)()
        fields, ncs = [], []
        self.last_flux, self.last_te, self.last_overlaps, self.last_grad = [], [], [], []
        for i, p in enumerate(packed):
            if grad_eps_ptrs is not None:
                results[i].grad_eps = C.cast(C.c_void_p(int(grad_eps_ptrs[i])), _dp) if grad_eps_ptrs[i] else None
                self.last_grad.append(None)
            elif grad_eps is not None and grad_eps[i]:
                g = np.zeros((p.num_modes, 3, p.nx, p.ny), dtype=np.complex128)
                self.last_grad.append(g)
                results[i].grad_eps = _ptr(g.view(np.float64))
            else:
                self.last_grad.append(None)
            nc = np.zeros(p.num_modes, dtype=np.complex128)
            ncs.append(nc)
            results[i].n_complex = _ptr(nc.view(np.float64))
            if want_flux:
                fl, te = np.zeros(p.num_modes), np.zeros(p.num_modes)
                self.last_flux.append(fl)
                self.last_te.append(te)
                results[i].flux = _ptr(fl)
                results[i].te_fraction = _ptr(te)
            if want_overlaps:
                ov = np.zeros((p.num_modes, p.num_modes), dtype=np.complex128)
                self.last_overlaps.append(ov)
                results[i].overlap_prev = _ptr(ov.view(np.float64))
            if fields_ptrs is not None:
                results[i].fields = C.cast(C.c_void_p(int(fields_ptrs[i])), _dp)
            elif want_fields:
                dt = np.complex64 if p.struct.precision == 1 else np.complex128
                f = _pool.empty((2, 3, p.nx, p.ny, 1, p.num_modes), dtype=dt)
                fields.append(f)
                results[i].fields = C.cast(C.c_void_p(f.ctypes.data), _dp)
            else:
                results[i].fields = None
        rc = lib().b200ms_solve_batch(self._h, n, probs, results)
        return rc, (fields if (want_fields and fields_ptrs is None) else None), ncs, results
