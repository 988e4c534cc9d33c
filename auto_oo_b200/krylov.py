"""Matrix-free Newton step: the lowest eigenpair of a symmetric operator by Davidson-Liu and the shifted Newton solve
by deflated preconditioned CG, from products ``matvec(v)`` and the diagonal alone -- the matrix is never formed.

Written against any ``matvec`` that maps a device vector ``(n,)`` to ``H v`` on the same device (and ``(n, m)`` to
``H V``) and its diagonal ``diag (n,)``; :class:`auto_oo_b200.OrbitalHessian` supplies both from the class buffer.
Everything between two products is a kernel of ``csrc/krylov.cu`` on the device; the host reads the residual norm
once per iteration (with Davidson's breakdown flag, in the same copy) for the convergence test.

Semantics of :func:`newton_step` are those of ``NewtonStep.newton_step`` on the formed matrix:
``lambda_0`` = lowest eigenvalue, ``sigma = mu + rho |lambda_0|`` when ``lambda_0 < lambda_min`` and ``aug``, else 0,
``dp = -(H + sigma)^-1 g``; both differ from the dense route by the solver tolerances only.
"""
from __future__ import annotations

import torch

from .engine import F64, HotPathEngine

__all__ = ["lowest_eigenpair", "shifted_solve", "newton_step", "KMAX", "DIAG_FLOOR"]

KMAX = 32                     # Davidson basis size before a thick restart to [x, x_prev]
DIAG_FLOOR = 1e-8             # |D - theta| below this is replaced by +-DIAG_FLOOR in the correction


def _engine(engine, device):
    return engine if engine is not None else HotPathEngine.for_tensors(2, device=device)


def _davidson(matvec, D, guess, tol, max_iter, kmax, eng, info):
    """(lambda_0, x_0, H x_0) with ||H x_0 - lambda_0 x_0|| <= tol; see :func:`lowest_eigenpair`."""
    n, dev = D.numel(), D.device
    kmax = max(3, min(int(kmax), n))
    Vt = torch.zeros(kmax, n, dtype=F64, device=dev)
    HVt = torch.zeros(kmax, n, dtype=F64, device=dev)
    S = torch.zeros(kmax, kmax, dtype=F64, device=dev)
    w = torch.zeros(kmax, dtype=F64, device=dev)
    Y = torch.zeros(kmax, kmax, dtype=F64, device=dev)
    yprev = torch.zeros(kmax, dtype=F64, device=dev)
    x = torch.empty(n, dtype=F64, device=dev)
    hx = torch.empty(n, dtype=F64, device=dev)
    rnorm = torch.empty(2, dtype=F64, device=dev)           # ||r||, breakdown flag
    # start: the unit vector at argmin diag(H), and the guess (the gradient) made orthonormal to it
    i0 = torch.argmin(D).reshape(1)
    Vt[0].index_fill_(0, i0, 1.0)
    k = 1
    if guess is not None and n > 1:
        u = guess.detach().to(device=dev, dtype=F64).reshape(n).clone().index_fill_(0, i0, 0.0)
        nrm = torch.linalg.vector_norm(u)
        other = torch.zeros(n, dtype=F64, device=dev).index_fill_(0, torch.remainder(i0 + 1, n), 1.0)
        Vt[1] = torch.where(nrm > 0, u / torch.where(nrm > 0, nrm, 1.0), other)
        k = 2
    HVt[:k] = matvec(Vt[:k].T.contiguous()).T
    products = k
    for m in range(k):
        eng.davidson_project(Vt, m + 1, HVt[m], S[m], 1, S[:, m], kmax)
    it = restarts = 0
    while True:
        eng.subspace_eigh(S, k, w, Y)
        restart = k == kmax
        eng.davidson_expand(Vt, HVt, k, Y, w[:1], D, S, x, hx, yprev, rnorm, DIAG_FLOOR)
        res, broke = rnorm.tolist()
        if res <= tol:
            break
        if broke:
            raise RuntimeError(f"Davidson: breakdown after {it + 1} iterations -- the preconditioned correction lies in "
                               f"the search space while the residual norm is {res:.3e} > {tol:.1e}")
        it += 1
        if it >= max_iter:
            raise RuntimeError(f"Davidson: no convergence in {max_iter} iterations, residual norm {res:.3e} > {tol:.1e}")
        restarts += restart
        k = 3 if restart else k + 1
        HVt[k - 1] = matvec(Vt[k - 1])
        products += 1
        eng.davidson_project(Vt, k, HVt[k - 1], S[k - 1], 1, S[:, k - 1], kmax)
    if info is not None:
        info.update(davidson_products=products, davidson_iterations=it + 1, davidson_restarts=restarts,
                    davidson_residual=res)
    return w[0].item(), x, hx


def lowest_eigenpair(matvec, diag, guess=None, tol=1e-7, max_iter=200, kmax=KMAX, engine=None, info=None):
    """Lowest eigenpair ``(lambda_0, x_0)`` of the symmetric operator ``matvec`` by Davidson-Liu, preconditioned by
    ``diag``.  Start vectors: the unit vector at ``argmin diag`` and ``guess`` (optional) made orthonormal to it.
    Converged when ``||H x - lambda x|| <= tol``; the Ritz value is an upper bound on ``lambda_0`` with an error of
    order ``tol^2 / gap``.  ``x_0`` is a unit device vector.  Raises ``RuntimeError`` after ``max_iter`` iterations
    without convergence.  ``info`` (a dict) receives the product and iteration counts."""
    eng = _engine(engine, diag.device if torch.is_tensor(diag) and diag.is_cuda else None)
    D = eng.dev(diag).reshape(-1)
    if D.numel() == 0:
        raise ValueError("lowest_eigenpair of an empty operator")
    lam, x, _ = _davidson(matvec, D, guess, tol, max_iter, kmax, eng, info)
    return lam, x


def _cg(matvec, D, rhs, shift, tol, max_iter, deflate, eng, info):
    n, dev = D.numel(), D.device
    if not bool(((D + shift) > 0).all()):
        raise ValueError("shifted_solve: the preconditioner diag + shift is not positive; the shifted system is "
                         "not positive definite")
    x = torch.zeros(n, dtype=F64, device=dev)
    r = rhs.detach().to(device=dev, dtype=F64).reshape(n).clone()
    p = torch.empty(n, dtype=F64, device=dev)
    state = torch.zeros(2, dtype=F64, device=dev)
    rnorm = torch.empty(1, dtype=F64, device=dev)
    bnorm = torch.linalg.vector_norm(r).item()
    if bnorm == 0.0:
        return x
    w = aw = None
    if deflate is not None:
        w, hw = deflate
        aw = torch.add(hw, w, alpha=float(shift))
    eng.pcg_step(None, shift, D, x, r, p, state, rnorm, w=w, aw=aw, init=True)
    res, it = rnorm.item(), 0
    while res > tol * bnorm:
        if it >= max_iter:
            raise RuntimeError(f"CG: no convergence in {max_iter} iterations, relative residual {res / bnorm:.3e} > "
                               f"{tol:.1e}")
        Ap = matvec(p)
        eng.pcg_step(Ap, shift, D, x, r, p, state, rnorm, w=w, aw=aw)
        res = rnorm.item()
        it += 1
    if info is not None:
        info.update(cg_products=it, cg_residual=res / bnorm)
    return x


def shifted_solve(matvec, diag, rhs, shift=0.0, tol=1e-12, max_iter=1000, deflate=None, engine=None, info=None):
    """``x = (H + shift)^-1 rhs`` by preconditioned CG (preconditioner ``diag + shift``, which must be positive; the
    shifted operator must be positive definite).  ``deflate = (w, H w)``: start from the Galerkin solution in span{w}
    and keep every search direction ``(H + shift)``-orthogonal to ``w`` -- with ``w`` the lowest eigenvector this
    removes the mode that makes the shifted system ill-conditioned.  Converged when ``||(H + shift) x - rhs|| <=
    tol ||rhs||``; ``RuntimeError`` after ``max_iter`` products without convergence.  Returns a device vector."""
    eng = _engine(engine, diag.device if torch.is_tensor(diag) and diag.is_cuda else None)
    D = eng.dev(diag).reshape(-1)
    if rhs.shape != (D.numel(),):
        raise ValueError(f"shifted_solve expects a right-hand side of shape ({D.numel()},), got {tuple(rhs.shape)}")
    return _cg(matvec, D, eng.dev(rhs), shift, tol, max_iter, deflate, eng, info)


def newton_step(matvec, diag, gradient, mu=1e-6, rho=1.1, lambda_min=1e-6, aug=True, eig_tol=1e-7, lin_tol=1e-12,
                eig_max_iter=200, lin_max_iter=1000, engine=None, info=None):
    """``(dp, lambda_0)`` of ``NewtonStep.newton_step`` without forming H: Davidson for ``lambda_0`` (started from the
    gradient), then deflated PCG on ``(H + sigma) dp = -g``.  ``aug=False`` with ``lambda_0 < lambda_min`` is an
    indefinite system that CG cannot solve: ``ValueError`` (the dense route handles it).  ``dp`` is a device
    vector."""
    eng = _engine(engine, diag.device if torch.is_tensor(diag) and diag.is_cuda else None)
    D = eng.dev(diag).reshape(-1)
    n = D.numel()
    if tuple(gradient.shape) != (n,):
        raise ValueError(f"newton_step expects a gradient of shape ({n},), got {tuple(gradient.shape)}")
    g = eng.dev(gradient)
    lam, x0, hx0 = _davidson(matvec, D, g, eig_tol, eig_max_iter, KMAX, eng, info)
    sigma = 0.0
    if lam < lambda_min:
        if not aug:
            raise ValueError(f"matrix-free Newton step with aug=False and lowest eigenvalue {lam:.3e} < lambda_min = "
                             f"{lambda_min:.1e}: the Newton system is indefinite and CG cannot solve it; use the dense "
                             f"route (NewtonStep.newton_step on the formed matrix)")
        sigma = mu + rho * abs(lam)
    if not lam + sigma > 0:
        raise ValueError(f"matrix-free Newton step: H + sigma is not positive definite (lowest eigenvalue {lam:.3e}, "
                         f"sigma {sigma:.3e})")
    dp = _cg(matvec, D, -g, sigma, lin_tol, lin_max_iter, (x0, hx0), eng, info)
    if info is not None:
        info.update(shift=sigma, lowest_eigenvalue=lam)
    return dp, lam
