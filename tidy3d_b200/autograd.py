"""PyTorch autograd for the effective index: ``n_complex(eps_diag, ...)`` is differentiable with respect to the permittivity.

The forward pass solves the modes of every frequency in one library call with ``want_fields=False`` and asks the library for
dn/deps of every cell (``compute_modes_batch(grad_eps=...)``, DESIGN.md section 10): the Jacobian comes from the left
eigenvector of the diagonal operator, so the backward pass is a contraction and needs no further solve.  Only diagonal
permittivity is differentiable (no bends, angles or PEC-valued cells; the off-diagonal components are zero by construction).

    eps = torch.tensor(..., dtype=torch.complex128, requires_grad=True)   # (F or 1, 3, Nx, Ny): xx, yy, zz
    n = autograd.n_complex(eps, coords, freqs, mode_spec)                 # (F, M) complex128
    loss = n.real[:, 0].sum(); loss.backward()                            # eps.grad: (F or 1, 3, Nx, Ny)
"""
from __future__ import annotations

import numpy as np
import torch

from . import solver


class _NComplex(torch.autograd.Function):
    @staticmethod
    def forward(ctx, eps_diag, coords, freqs, mode_spec, symmetry, direction):
        if eps_diag.dim() != 4 or eps_diag.shape[1] != 3:
            raise ValueError("eps_diag must have shape (F or 1, 3, Nx, Ny)")
        freqs = np.atleast_1d(np.asarray(freqs, dtype=np.float64))
        nf, nfe = freqs.size, eps_diag.shape[0]
        if nfe not in (1, nf):
            raise ValueError("eps_diag must hold one permittivity per frequency, or one for all")
        eps = eps_diag.detach().to("cpu", torch.complex128).numpy()
        nx, ny = eps.shape[2], eps.shape[3]
        m = int(mode_spec.num_modes)
        problems = []
        for f in range(nf):
            e = eps[f if nfe > 1 else 0]
            z = np.zeros((nx, ny), dtype=np.complex128)
            eps_cross = np.ascontiguousarray(np.stack([e[0], z, z, z, e[1], z, z, z, e[2]]))
            problems.append(dict(eps_cross=eps_cross, coords=coords, freq=float(freqs[f]), mode_spec=mode_spec, symmetry=symmetry,
                                 direction=direction))
        # the Jacobian stays where the input lives: a CUDA input gets it written straight into device memory
        jac = torch.empty((nf, m, 3, nx, ny), dtype=torch.complex128, device=eps_diag.device)
        device = eps_diag.device.index if eps_diag.is_cuda else -1
        if eps_diag.is_cuda and device is None:
            device = torch.cuda.current_device()
        ptrs = [jac[f].data_ptr() for f in range(nf)] if jac.is_cuda else None
        out, infos = solver.compute_modes_batch(problems, device=device, want_fields=False, return_info=True, grad_eps=True,
                                                grad_eps_ptrs=ptrs)
        if not jac.is_cuda:
            for f, info in enumerate(infos):
                jac[f] = torch.from_numpy(info["grad_eps"])
        ctx.save_for_backward(jac)
        ctx.nfe, ctx.in_dtype = nfe, eps_diag.dtype
        return torch.from_numpy(np.stack([o[1] for o in out])).to(eps_diag.device)

    @staticmethod
    def backward(ctx, grad_out):
        (jac,) = ctx.saved_tensors
        # holomorphic n(eps): torch's convention is grad_in = grad_out * conj(dn/deps)
        g = torch.einsum("fm,fmcxy->fcxy", grad_out.to(jac.dtype), jac.conj())
        if ctx.nfe == 1:
            g = g.sum(dim=0, keepdim=True)
        return g.to(ctx.in_dtype), None, None, None, None, None


def n_complex(eps_diag: torch.Tensor, coords, freqs, mode_spec, symmetry=(0, 0), direction="+") -> torch.Tensor:
    """n_eff + i k_eff, shape (F, num_modes), of the diagonal permittivity ``eps_diag`` (complex, (F or 1, 3, Nx, Ny): the xx,
    yy, zz components; one array for all frequencies when the first dimension is 1), differentiable with respect to it."""
    return _NComplex.apply(eps_diag, coords, freqs, mode_spec, tuple(symmetry), direction)
