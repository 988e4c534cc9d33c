"""Damped / augmented-Hessian Newton step with Armijo backtracking -- the optimiser that calls
the hot path as ``objective_fn`` (reference ``utils/newton_raphson.py:16-224``; same
hyper-parameters, return values and failure behaviour).  Works on tensors of any torch device
(the reference's version adds a CPU identity to the Hessian, ``newton_raphson.py:117-119``)."""
from __future__ import annotations

import math as _math

import torch


def wolfe(t, grad, dp, alpha=1e-4):
    """Armijo decrease ``alpha t <grad, dp>`` (reference ``newton_raphson.py:12-13``)."""
    return alpha * t * torch.dot(grad, dp)


def split_list_shapes(parameters, paramshapes):
    """Split a flat vector into tensors of the given shapes (reference ``:214-224``)."""
    chunks, start = [], 0
    for shape in paramshapes:
        size = int(_math.prod(shape))
        chunks.append(parameters[start:start + size].reshape(shape))
        start += size
    return chunks


class NewtonStep:
    """``x <- x - H^{-1} G`` with ``H <- H + (mu + rho |lambda_0|) I`` when ``lambda_0 < lambda_min``
    and step halving until ``f(x + t dx) <= f(x) + alpha t G.dx`` (at most ``lmax`` halvings,
    then ``t = 0``)."""

    def __init__(self, alpha=0.0001, beta=.5, mu=1e-6, rho=1.1, lmax=20, lambda_min=1e-6, aug=True,
                 verbose=1, speculate=0):
        """``speculate`` > 1: when the objective offers ``objective_fn.batched(list_of_parameter_tuples)
        -> energies`` (``OO_energy.energy_from_kappa`` does), the line search evaluates that many step
        lengths ``t, beta t, beta^2 t, ...`` per batched call and accepts the first that satisfies the
        Armijo condition -- the same result as the sequential search, fewer round trips."""
        self.alpha, self.beta, self.mu, self.rho = alpha, beta, mu, rho
        self.lmax, self.lambda_min, self.aug, self.verbose = lmax, lambda_min, aug, verbose
        self.speculate = int(speculate)

    def newton_step(self, gradient, hessian):
        """Returns ``(dp, lowest eigenvalue of the un-augmented Hessian)`` (reference ``:78-129``).  ``hessian`` is a
        matrix, or an operator with ``matvec`` and ``diagonal`` (``OrbitalHessian``): then H is never formed -- Davidson
        finds the lowest eigenpair and deflated CG solves the shifted system (``auto_oo_b200/krylov.py``)."""
        if hasattr(hessian, "matvec") and hasattr(hessian, "diagonal"):
            return self._matrix_free_step(gradient, hessian)
        evals, evecs = torch.linalg.eigh(hessian)
        lowest_eigenvalue = evals[0].item()
        if self.verbose:
            print("lowest eigval hessian =", lowest_eigenvalue)
        if lowest_eigenvalue < self.lambda_min and self.aug:
            if self.verbose:
                print("augmenting hessian...")
            # H + shift I has the eigenvectors of H and its eigenvalues moved by shift: the reference's second
            # eigh (newton_raphson.py:117-121) is not needed
            evals = evals + (self.mu + self.rho * abs(lowest_eigenvalue))
            if self.verbose:
                print("Lowest eigenvalue of augmented hessian:", evals[0].item())
        # -(V diag(1/w) V^T) g without forming the inverse
        return -(evecs @ ((evecs.T @ gradient) / evals)), lowest_eigenvalue

    def _matrix_free_step(self, gradient, hessian):
        kw = dict(mu=self.mu, rho=self.rho, lambda_min=self.lambda_min, aug=self.aug)
        if hasattr(hessian, "newton_step"):
            dp, lowest_eigenvalue = hessian.newton_step(gradient, **kw)
        else:
            from .. import krylov
            dp, lowest_eigenvalue = krylov.newton_step(hessian.matvec, hessian.diagonal(), gradient, **kw)
            dp = dp.to(gradient.device)
        if self.verbose:
            print("lowest eigval hessian =", lowest_eigenvalue)
            if lowest_eigenvalue < self.lambda_min and self.aug:
                print("augmenting hessian...")
        return dp, lowest_eigenvalue

    def backtracking(self, objective_fn, parameters, dp, gradient):
        """Reference ``:131-192``."""
        nargs = len(parameters)
        t = 1.
        energy = objective_fn(*parameters).item()
        flat = torch.cat([p.reshape(-1) for p in parameters])
        shapes = [tuple(p.shape) for p in parameters]
        test_energy = objective_fn(*split_list_shapes(flat + t * dp, shapes))
        batched = getattr(objective_fn, "batched", None)
        if (self.speculate > 1 and batched is not None
                and test_energy > energy + wolfe(t, gradient, dp, alpha=self.alpha)):
            return self._speculative_backtracking(objective_fn, batched, parameters, flat, shapes, dp, gradient,
                                                  energy, nargs)
        if test_energy > energy + wolfe(t, gradient, dp, alpha=self.alpha):
            assert wolfe(t, gradient, dp, alpha=self.alpha) < 0
            num = 0
            if self.verbose:
                print("test_energy:", test_energy.item(), "... old energy:", energy)
                print("do backtracking line search...")
            while test_energy > energy + wolfe(t, gradient, dp, alpha=self.alpha):
                t = self.beta * t
                if self.verbose:
                    print("t =", t)
                test_energy = objective_fn(*split_list_shapes(flat + t * dp, shapes))
                num += 1
                if num > self.lmax:
                    t = 0.
                    test_energy = objective_fn(*parameters)
                    if self.verbose:
                        print("Warning: line search failed. Output previous parameters.")
                    break
        new_energy = test_energy.item()
        newp = flat + t * dp
        if self.verbose:
            print("new energy:", new_energy)
            print("old energy:", energy)
        new_parameters = tuple(split_list_shapes(newp, shapes)) if nargs > 1 else newp
        return new_parameters, new_energy

    def _speculative_backtracking(self, objective_fn, batched, parameters, flat, shapes, dp, gradient, energy,
                                  nargs):
        """Backtracking with ``speculate`` candidate step lengths per batched evaluation; accepts exactly
        the step the sequential search (reference ``:156-176``) would accept."""
        assert wolfe(1., gradient, dp, alpha=self.alpha) < 0
        slope = torch.dot(gradient, dp).item()
        t, num, accepted, new_energy = 1., 0, None, None
        while accepted is None and num < self.lmax:
            ts = []
            # the sequential search (reference :165-176) gives up when the (lmax+1)-th halving fails, i.e. it can
            # accept at most beta^lmax: no more than lmax candidates in total
            while len(ts) < self.speculate and num + len(ts) < self.lmax:
                t = self.beta * t
                ts.append(t)
            if not ts:
                break
            energies = batched([tuple(split_list_shapes(flat + tt * dp, shapes)) for tt in ts])
            for tt, e in zip(ts, energies):
                num += 1
                if not (e.item() > energy + self.alpha * tt * slope):
                    accepted, new_energy = tt, e.item()
                    break
        if accepted is None:                                # line search failed: keep the old parameters
            accepted, new_energy = 0., objective_fn(*parameters).item()
            if self.verbose:
                print("Warning: line search failed. Output previous parameters.")
        if self.verbose:
            print("new energy:", new_energy)
            print("old energy:", energy)
        newp = flat + accepted * dp
        new_parameters = tuple(split_list_shapes(newp, shapes)) if nargs > 1 else newp
        return new_parameters, new_energy

    def damped_newton_step(self, objective_fn, parameters, gradient, hessian):
        """One optimiser step; returns ``(new parameters, lowest Hessian eigenvalue before the
        step)`` (reference ``:194-211``)."""
        dp, lowest_eigenvalue = self.newton_step(gradient, hessian)
        new_parameters, _ = self.backtracking(objective_fn, parameters, dp, gradient)
        return new_parameters, lowest_eigenvalue
