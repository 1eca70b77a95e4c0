"""GPU: the permittivity gradient dn/deps of the device (compute_modes_batch(grad_eps=...), autograd.n_complex).

Against the oracle's exact discrete gradient (left eigenvectors of A^T by shift-invert, tests/sensitivity_oracle.py), against
central differences of the device's own n_complex, inside large batches, with host and device delivery, and through
torch autograd.  "tight" tolerance preset throughout.
"""
import numpy as np
import pytest

from tests import sensitivity_oracle as SO
from tests.golden import cases as GC
from tests.helpers import well_separated
from tidy3d_b200 import _cabi
from tidy3d_b200 import workloads as W
from tidy3d_b200.solver import compute_modes_batch, get_handle

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def tight():
    return get_handle(tolerance="tight")


def _problem(wl, **kw):
    p = dict(eps_cross=wl.eps_cross, coords=wl.coords, freq=float(wl.freqs[0]), mode_spec=wl.mode_spec)
    p.update(kw)
    return p


def _golden_problem(name):
    factory, kw, _ = GC.CASES[name]
    wl = factory()
    return _problem(wl, **GC.resolve_kwargs(wl, kw))


@pytest.mark.parametrize("name", ["c1_64", "lossy_48", "nonuniform_56", "c1_64_sym_pmc_pec"])
def test_device_gradient_matches_the_exact_gradient(tight, name):
    p = _golden_problem(name)
    (res,), (info,) = compute_modes_batch([p], want_fields=False, return_info=True, handle=tight, grad_eps=True)
    n, g = res[1], info["grad_eps"]
    assert g.shape == (p["mode_spec"].num_modes, 3) + p["eps_cross"][0].shape
    ok = well_separated(n)
    for m in np.flatnonzero(ok):
        _, ref = SO.sparse_grad(p["eps_cross"], p["coords"], p["freq"], p["mode_spec"], p.get("symmetry", (0, 0)), -(n[m] ** 2))
        err = np.abs(g[m] - ref).max() / np.abs(ref).max()
        assert err <= 1e-6, (name, m, err)


def _core_mask(wl):
    e = np.abs(np.asarray(wl.eps_cross[0]))
    return e >= 0.99 * e.max()


@pytest.mark.parametrize("make", [lambda: W.c3(96), lambda: W.si_strip(64, 2)], ids=["c3_96", "strip_64"])
def test_gradient_sums_to_the_central_difference_of_the_solver(tight, make):
    wl = make()
    mask = _core_mask(wl)
    delta = 1e-2
    probs = []
    for s in (0.0, +1.0, -1.0):
        e = [np.array(a, copy=True) for a in wl.eps_cross]
        for k in (0, 4, 8):
            e[k][mask] += s * delta
        probs.append(_problem(wl, eps_cross=e))
    out, infos = compute_modes_batch(probs, want_fields=False, return_info=True, handle=tight, grad_eps=[True, False, False])
    fd = (out[1][1][0] - out[2][1][0]) / (2 * delta)
    ad = infos[0]["grad_eps"][0][:, mask].sum()
    assert abs(fd - ad) <= 1e-3 * abs(ad), (fd, ad)


def _distinct_batch(n=48, count=64):
    probs = []
    for i in range(count):
        wl = W.si_strip(n, 2, w=0.40 + 0.005 * i)
        probs.append(_problem(wl))
    return probs


def test_batched_gradient_matches_a_lone_solve_and_delivery_paths_agree(tight):
    import torch

    probs = _distinct_batch()
    _, infos = compute_modes_batch(probs, want_fields=False, return_info=True, handle=tight, grad_eps=True)
    j = 37
    _, (lone,) = compute_modes_batch([probs[j]], want_fields=False, return_info=True, handle=tight, grad_eps=True)
    g, g1 = infos[j]["grad_eps"], lone["grad_eps"]
    assert np.abs(g - g1).max() <= 1e-6 * np.abs(g1).max()
    dev = [torch.empty(g.shape, dtype=torch.complex128, device="cuda") for _ in probs]
    compute_modes_batch(probs, want_fields=False, return_info=True, handle=tight, grad_eps_ptrs=[t.data_ptr() for t in dev])
    torch.cuda.synchronize()
    for i in (0, j, len(probs) - 1):
        assert np.array_equal(dev[i].cpu().numpy(), infos[i]["grad_eps"])


def test_no_change_without_a_gradient(tight):
    probs = _distinct_batch(count=6)
    plain = compute_modes_batch(probs, want_fields=False, handle=tight)
    mixed, infos = compute_modes_batch(probs, want_fields=False, return_info=True, handle=tight, grad_eps=[True, False] * 3)
    for i in range(len(probs)):
        assert ("grad_eps" in infos[i]) == (i % 2 == 0)
        assert np.array_equal(mixed[i][1], plain[i][1])
    # an out-of-scope problem in the same library call fails alone
    bent = _problem(W.c4(48))
    angled = _problem(W.angled(48))
    packed = [_cabi.PackedProblem(p["eps_cross"], p["coords"], p["freq"], p["mode_spec"]) for p in (probs[0], bent, probs[1], angled)]
    with tight.lock:
        rc, _, ncs, results = tight.solve_batch(packed, want_fields=False, grad_eps=[True, True, False, True])
    assert rc == _cabi.ERR_UNSUPPORTED
    assert [results[i].status for i in range(4)] == [_cabi.OK, _cabi.ERR_UNSUPPORTED, _cabi.OK, _cabi.ERR_UNSUPPORTED]
    pair = compute_modes_batch(probs[:2], want_fields=False, handle=tight)  # the same device batch, without a gradient
    assert np.array_equal(ncs[0], pair[0][1]) and np.array_equal(ncs[2], pair[1][1])
    with pytest.raises(NotImplementedError):
        compute_modes_batch([probs[0], bent], want_fields=False, handle=tight, grad_eps=[False, True])


@pytest.mark.parametrize("device", ["cpu", "cuda"])
def test_autograd_matches_a_finite_difference_of_the_loss(tight, device, monkeypatch):
    import torch

    from tidy3d_b200 import autograd, solver

    monkeypatch.setattr(solver, "get_handle", lambda device=-1, tolerance="reference": get_handle(device, "tight"))
    wl = W.si_strip(48, 2)
    freqs = W.C_0 / np.array([1.50, 1.55, 1.60])
    e = np.asarray(wl.eps_cross[0]) * (1 + 0.01j)
    eps0 = torch.tensor(np.stack([e, e * 1.02, e * 0.98])[None], dtype=torch.complex128, device=device)
    xm = 0.5 * (wl.coords[0][:-1] + wl.coords[0][1:])
    bump = np.exp(-(xm[:, None] ** 2 + xm[None, :] ** 2) / 0.1)
    rng = np.random.default_rng(3)
    direction = torch.tensor(np.stack([c * bump for c in rng.normal(size=3) + 1j * rng.normal(size=3)])[None], dtype=torch.complex128, device=device)
    w_re = torch.tensor(rng.normal(size=(3, 2)), dtype=torch.float64, device=device)
    w_im = torch.tensor(rng.normal(size=(3, 2)), dtype=torch.float64, device=device)

    def loss(eps):
        n = autograd.n_complex(eps, wl.coords, freqs, wl.mode_spec)
        return (w_re * n.real).sum() + 100.0 * (w_im * n.imag).sum()

    eps = eps0.clone().requires_grad_(True)
    loss(eps).backward()
    assert eps.grad.device == eps0.device and eps.grad.dtype == eps0.dtype and eps.grad.shape == eps0.shape
    ad = float(torch.real((eps.grad.conj() * direction).sum()))
    t = 1e-3
    with torch.no_grad():
        fd = float((loss(eps0 + t * direction) - loss(eps0 - t * direction)) / (2 * t))
    assert abs(fd - ad) <= 1e-3 * abs(ad), (fd, ad)
