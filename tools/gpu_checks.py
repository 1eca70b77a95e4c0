"""DEV TOOL: component-by-component comparison of the CUDA path with the numpy model (run under gpurun)."""
import ctypes as C
import sys
import time

import numpy as np

sys.path.insert(0, "/root/repo")
sys.path.insert(0, "/root/repo/tools")
import proto as P  # noqa: E402
from oracle import restatement as R  # noqa: E402
from tests.golden.cases import CASES  # noqa: E402
from tidy3d_b200 import _cabi, compute_modes_batch  # noqa: E402
from tidy3d_b200 import workloads as W  # noqa: E402

L = _cabi.lib()
H = _cabi.Handle()
rng = np.random.default_rng(3)


def cvec(shape):
    return rng.standard_normal(shape) + 1j * rng.standard_normal(shape)


def dev_apply(pk, level, mode, x, rhs, n2):
    y = np.zeros(n2, complex)
    xa = np.ascontiguousarray(x.ravel().astype(complex))
    ra = np.ascontiguousarray(rhs.ravel().astype(complex)) if rhs is not None else None
    rc = L.b200ms_debug_apply(H._h, C.byref(pk.struct), level, mode, _cabi._ptr(xa.view(float)), _cabi._ptr(ra.view(float)) if ra is not None else None, _cabi._ptr(y.view(float)))
    assert rc == 0, (rc, H.last_error())
    return y


def rel(a, b):
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


def components(name, wl, kw):
    sym = kw.get("symmetry", (0, 0))
    pk = _cabi.PackedProblem(wl.eps_cross, wl.coords, wl.freqs[0], wl.mode_spec, sym, kw.get("direction", "+"))
    st = R.setup(wl.eps_cross, wl.coords, wl.freqs[0], wl.mode_spec, sym)
    real = not np.issubdtype(R.solver_dtype(st, "double"), np.complexfloating)
    sigma = -st["target"] ** 2
    lv0 = P.fine_level(st, sigma)
    ph = 0.7853981633974483
    lim = lambda l: np.abs(l) * np.exp(1j * np.clip(np.angle(l), -ph, ph))  # noqa: E731
    st_p = dict(st); st_p["slen"] = [(lim(lf), lim(lb)) for lf, lb in st["slen"]]
    lvp = P.fine_level(st_p, sigma)
    kmax = np.sqrt(max(0.0, max(lv0.exx.real.max(), lv0.eyy.real.max()) - st["target"] ** 2))
    indef = kmax**2 > 1e-6
    mg = P.Multigrid(lvp, min_size=12, nu=2, omega=0.8, coarse_sweeps=16, coarse_gmres=16 if indef else 0,
                     kh_limit=2 * np.pi / 4 if indef else 0.0, kmax=kmax)
    print(f"== {name}: real={real} levels={[(l.nx, l.ny) for l in mg.levels]} indef={indef}")
    mk = (lambda s: cvec(s).real + 0j) if real else cvec
    for li, lv in enumerate([lv0] + mg.levels[1:3]):
        x = mk((2, lv.nx, lv.ny)); rhs = mk((2, lv.nx, lv.ny))
        n2 = 2 * lv.nx * lv.ny
        y = dev_apply(pk, li, 0, x, None, n2)
        y0 = lv.apply(x).ravel()
        e0 = rel(y, y0)
        y = dev_apply(pk, li, 1, x, rhs, n2)
        e1 = rel(y, (rhs - lv.apply(x)).ravel())
        y = dev_apply(pk, li, 2, x, rhs, n2)
        e2 = rel(y, (x + 0.8 * (rhs - lv.apply(x)) / lv.diag).ravel())
        y = dev_apply(pk, li, 3, x, rhs, n2)
        e3 = rel(y, (0.8 * rhs / lv.diag).ravel())
        print(f"   level {li} ({lv.nx}x{lv.ny}): apply {e0:.1e} resid {e1:.1e} jacobi {e2:.1e} jacobi0 {e3:.1e}")
    # V-cycle
    r = mk((2, st["nx"], st["ny"]))
    if not st["pmc"][1] and st["ny"] > 1:
        r[0][:, 0] = 0
    if not st["pmc"][0] and st["nx"] > 1:
        r[1][0, :] = 0
    z = np.zeros(r.size, complex)
    ra = np.ascontiguousarray(r.ravel())
    rc = L.b200ms_debug_vcycle(H._h, C.byref(pk.struct), _cabi._ptr(ra.view(float)), _cabi._ptr(z.view(float)))
    assert rc == 0, (rc, H.last_error())
    z0 = mg(r).ravel()
    print(f"   vcycle rel diff {rel(z, z0):.2e}   (|z| {np.abs(z).max():.2e})")
    # inner solve
    x = np.zeros(r.size, complex); it = C.c_int(); rr = C.c_double()
    t0 = time.time()
    rc = L.b200ms_debug_solve(H._h, C.byref(pk.struct), _cabi._ptr(ra.view(float)), _cabi._ptr(x.view(float)), C.byref(it), C.byref(rr))
    dt = time.time() - t0
    assert rc == 0, (rc, H.last_error())
    true_res = np.linalg.norm(r.ravel() - lv0.apply(x.reshape(r.shape)).ravel()) / np.linalg.norm(r)
    print(f"   fgmres: iters {it.value} est {rr.value:.1e} true {true_res:.1e}  wall {dt:.2f}s")


def full(names):
    for name in names:
        fac, kw, _ = CASES[name]
        wl = fac()
        g = np.load(f"/root/repo/tests/golden/{name}.npz")
        t0 = time.time()
        try:
            out, info = compute_modes_batch([dict(eps_cross=wl.eps_cross, coords=wl.coords, freq=wl.freqs[0], mode_spec=wl.mode_spec, **kw)], return_info=True)
        except Exception as e:  # noqa: BLE001
            print(f"## {name}: FAILED {type(e).__name__}: {e}")
            continue
        dt = time.time() - t0
        f, n, spec = out[0]
        dn = np.abs(n - g["n_tight"]).max()
        msg = f"## {name}: max|dn| {dn:.2e} {info[0]} wall {dt:.2f}s"
        if "fields_tight" in g.files:
            ft = g["fields_tight"]
            ovs = []
            for m in range(n.size):
                a, b = f[:, :, ..., m].ravel(), ft[:, :, ..., m].ravel()
                ovs.append(abs(np.vdot(a, b)) / (np.linalg.norm(a) * np.linalg.norm(b)))
            msg += f" overlaps(E,H all comps) {np.round(ovs, 6)}"
        print(msg)
        print("     n =", n)


if __name__ == "__main__":
    which = sys.argv[1:] or ["comp", "full"]
    if "comp" in which:
        for name in ["c1_64", "c1_64_sym_pmc_pec", "c3_96", "lossy_48", "c4_96", "nonuniform_56", "slab1d_x1", "slab1d_y1", "strip_128_m4", "c4_128"]:
            fac, kw, _ = CASES[name]
            try:
                components(name, fac(), kw)
            except Exception as e:  # noqa: BLE001
                print(f"== {name}: FAILED {type(e).__name__}: {e}")
    if "rand" in which:
        # the reference's own smoke test test_compute_modes (tests/test_plugins/test_mode_solver.py:170-181)
        rs = np.random.default_rng(0)
        eps_cross = rs.random((10, 10, 9))
        coords = np.arange(11)
        ms = W.ModeSpecLike(num_modes=3, target_neff=2.0, precision="single")
        ec = [eps_cross[..., i].astype(complex) for i in range(9)]
        try:
            f0, n0, s0 = R.compute_modes(ec, [coords, coords], 1.0, ms, direction="-")
            print("oracle", n0, s0)
            out = compute_modes_batch([dict(eps_cross=ec, coords=[coords, coords], freq=1.0, mode_spec=ms, direction="-")], return_info=True)
            print("gpu   ", out[0][0][1], out[0][0][2], out[1][0])
        except Exception as e:  # noqa: BLE001
            print("rand case FAILED", type(e).__name__, e)
        full(["pec_block_40"])
    if "tensor" in which:
        full(["angled_48_minus", "offdiag_48", "angled_phi_48", "angled_64"])
    if "full" in which:
        full(["c1_64", "c1_64_minus", "c1_64_sym_pmc_pec", "strip_128_m4", "lossy_48", "c3_96", "c4_96", "nonuniform_56", "slab1d_x1", "slab1d_y1", "c4_96_axis0"])
