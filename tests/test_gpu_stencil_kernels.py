"""GPU: the three stencil kernel families of the real fp32 multigrid path compute the same operator -- the one-column marching
kernel (round 1, itself pinned to the numpy model and, through the solves, to the reference), the pair-marching kernel
(csrc/march2.cuh) and its TMA row-staging variant (csrc/march2_tma.cuh).  All modes (apply, residual, stored-diagonal sweep, the
fused first two sweeps), several levels, widths that need one strip / several strips / are not a multiple of four columns
(register fallback of the TMA variant) / odd (one-column fallback).  The arithmetic is the same expression for expression, so the
difference is fp32 rounding of the fused-multiply-add contraction at most."""
import ctypes as C

import numpy as np
import pytest

from tidy3d_b200 import _cabi
from tidy3d_b200 import workloads as W

pytestmark = pytest.mark.gpu


def _rect(nx, ny, symmetry=(0, 0)):
    eps, coords = W.strip_eps(nx, ny)
    return W.Workload(name=f"strip_{nx}x{ny}", eps_cross=W._iso(eps), coords=coords, freqs=np.array([W.C_0 / 1.55]),
                      mode_spec=W.ModeSpecLike(num_modes=2, precision="double"), symmetry=symmetry)


def _apply(h, pk, level, mode, x, rhs):
    L = _cabi.lib()
    y = np.zeros(x.size, complex)
    xa = np.ascontiguousarray(x.ravel().astype(complex))
    ra = np.ascontiguousarray(rhs.ravel().astype(complex))
    rc = L.b200ms_debug_apply(h._h, C.byref(pk.struct), level, mode, _cabi._ptr(xa.view(float)), _cabi._ptr(ra.view(float)), _cabi._ptr(y.view(float)))
    assert rc == 0, (rc, h.last_error())
    return y


@pytest.mark.parametrize("shape,symmetry", [((96, 128), (0, 0)), ((150, 202), (0, 0)), ((70, 1100), (0, 0)), ((64, 64), (1, -1)), ((75, 131), (0, 0))])
def test_pair_and_tma_kernels_match_the_one_column_kernel(shape, symmetry):
    wl = _rect(*shape, symmetry=symmetry)
    pk = _cabi.PackedProblem(wl.eps_cross, wl.coords, wl.freqs[0], wl.mode_spec, wl.symmetry, "+")
    sh = (C.c_int * 40)()
    n = _cabi.lib().b200ms_debug_hierarchy(C.byref(pk.struct), None, 20, sh)
    shapes = [(sh[2 * i], sh[2 * i + 1]) for i in range(n)]
    hs = {sp: _cabi.Handle(stencil_pair=sp) for sp in (0, 1)}
    hs[9] = _cabi.Handle(stencil_pair=1, stencil_pair_rows=9)  # many short marches: every CTA boundary case
    rng = np.random.default_rng(7)
    try:
        for lvl, (nx, ny) in enumerate(shapes[:3]):
            if nx < 32:
                continue
            x, rhs = rng.standard_normal((2, nx, ny)), rng.standard_normal((2, nx, ny))
            for mode in (16, 17, 18, 20):  # + 16: the multigrid-precision operator also on level 0 (csrc/api.cu debug_run)
                ys = {sp: _apply(h, pk, lvl, mode, x, rhs) for sp, h in hs.items()}
                scale = np.abs(ys[0]).max()
                assert np.isfinite(scale) and scale > 0
                for sp, y in ys.items():
                    assert np.abs(y - ys[0]).max() <= 2e-6 * scale, (shape, lvl, mode, sp)
    finally:
        for h in hs.values():
            h.close()


@pytest.mark.parametrize("shape,symmetry", [((256, 256), (0, 0)), ((150, 300), (0, 0)), ((96, 128), (1, -1))])
def test_vcycle_is_the_same_with_every_kernel_family(shape, symmetry):
    """One multigrid V-cycle (b200ms_debug_vcycle) with the round-2 kernels everywhere (one-column stencil, per-range restriction,
    scalar prolongation) against the defaults (TMA pair stencil, packed-list restriction, 128-bit prolongation): same operator,
    same summation order in the transfers."""
    wl = _rect(*shape, symmetry=symmetry)
    pk = _cabi.PackedProblem(wl.eps_cross, wl.coords, wl.freqs[0], wl.mode_spec, wl.symmetry, "+")
    nx, ny = shape
    rng = np.random.default_rng(3)
    r = rng.standard_normal((2, nx, ny)) + 0j
    if symmetry[1] != 1 and ny > 1:
        r[0][:, 0] = 0  # PEC wall rows are held at zero (the V-cycle's input never has them)
    if symmetry[0] != 1 and nx > 1:
        r[1][0, :] = 0
    ra = np.ascontiguousarray(r.ravel())
    zs = {}
    for name, opts in (("round2", dict(stencil_pair=0, transfer_vec=0)), ("default", {}), ("transfers_only", dict(stencil_pair=0, transfer_vec=3))):
        h = _cabi.Handle(**opts)
        z = np.zeros(ra.size, complex)
        rc = _cabi.lib().b200ms_debug_vcycle(h._h, C.byref(pk.struct), _cabi._ptr(ra.view(float)), _cabi._ptr(z.view(float)))
        assert rc == 0, (rc, h.last_error())
        h.close()
        zs[name] = z
    scale = np.abs(zs["round2"]).max()
    assert np.isfinite(scale) and scale > 0
    assert np.abs(zs["transfers_only"] - zs["round2"]).max() <= 2e-6 * scale  # same expressions, same order
    assert np.abs(zs["default"] - zs["round2"]).max() <= 2e-5 * scale
