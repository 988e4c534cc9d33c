"""``OO_energy`` and the free functions of the reference's ``auto_oo.oo_energy`` module
(``/root/reference/src/auto_oo/oo_energy.py:21-474``), re-implemented on top of the sm_100a
C-ABI library (``include/oo_b200.h``) through :class:`auto_oo_b200.engine.HotPathEngine`.

Interface contract (SURVEY section 8b): same names, argument meaning and error behaviour as the
reference; inputs are float64 torch tensors (CPU, possibly carrying an autograd graph back to the
circuit parameters) or numpy arrays; results come back on the device / in the array type of the
inputs, so the reference's drivers (``NewtonStep``, ``OO_pqc.full_optimization``, the Berry-phase
loop) run unchanged.  Every number is produced by a CUDA kernel; there is no CPU path.

Differences a caller can observe, all deliberate:

* one four-index transform per set of MO coefficients serves energy, gradient and Hessian
  (the reference redoes it in each call: ``oo_energy.py:207-208, :410-411, :421-422``);
* ``analytic_hessian`` returns an :class:`OrbitalHessian` (device resident, I-space form) instead
  of a dense ``(N,N,N,N)`` tensor; ``full_hessian_to_matrix`` accepts it (and still accepts a dense
  tensor), ``OrbitalHessian.dense()`` materialises the reference's rank-4 tensor on request;
* differentiability: energy is differentiable (to any order) in the RDMs, the gradient once in the
  RDMs -- what ``OO_pqc`` needs (``oo_pqc.py:86-123``).  ``energy_from_kappa``, ``kappa_to_mo_coeff`` and
  ``get_transformed_mo`` are differentiable once in ``kappa`` (and the last in ``mo_coeff``) through the
  device adjoint of ``expm(-K)`` (``oo_kappa_rotation_vjp_f64``); a second derivative in ``kappa`` raises.
  ``energy_from_mo_coeff`` is not differentiable in ``mo_coeff``, and the batched entry points
  (``energies_from_kappas``, ``energy_gradient_hessian``, ``OO_energy_geometries``) detach their inputs.
"""
from __future__ import annotations

from functools import partial

import numpy as np
import torch

from .engine import HotPathEngine, F64
from .utils.newton_raphson import NewtonStep

__all__ = [
    "OO_energy", "OO_energy_geometries", "OrbitalHessian", "PendingEvaluation", "unpack_hessian",
    "general_4index_transform", "uniform_4index_transform",
    "int1e_transform", "int2e_transform", "mo_ao_to_mo_oao", "vector_to_skew_symmetric",
    "skew_symmetric_to_vector", "non_redundant_indices",
]


# --------------------------------------------------------------------------------------
# array plumbing
# --------------------------------------------------------------------------------------
def _like(result, template):
    """Return the device tensor ``result`` in the container type / device of ``template``."""
    if torch.is_tensor(template):
        return result.to(device=template.device, dtype=template.dtype if template.is_floating_point() else F64)
    return result.cpu().numpy()


def _as_tensor(x):
    return x if torch.is_tensor(x) else torch.as_tensor(np.asarray(x, dtype=np.float64))


# --------------------------------------------------------------------------------------
# free functions                                               (reference oo_energy.py:21-118)
# --------------------------------------------------------------------------------------
def general_4index_transform(M, C0, C1, C2, C3):
    """``M'_ijkl = sum_pqrs C0_pi C1_qj C2_rk C3_sl M_pqrs`` (reference ``oo_energy.py:21-30``).

    Four quarter transforms on FP64 tensor cores (``oo_int2e_transform_f64``)."""
    Mt = _as_tensor(M)
    n = Mt.shape[0]
    eng = HotPathEngine.for_tensors(n)
    g = eng.to_padded(Mt, 4)
    Cs = [eng.to_padded(_as_tensor(c), 2) for c in (C0, C1, C2, C3)]
    out = eng.from_padded(eng.int2e_transform(*Cs, g_ao=g), 4)[0]
    return _like(out, M)


def uniform_4index_transform(M, C):
    """Reference ``oo_energy.py:33-41``."""
    return general_4index_transform(M, C, C, C, C)


def int1e_transform(int1e_ao, mo_coeff):
    """``C^T h C`` (reference ``oo_energy.py:44-46``)."""
    h = _as_tensor(int1e_ao)
    eng = HotPathEngine.for_tensors(h.shape[0])
    out = eng.from_padded(eng.int1e_transform(eng.to_padded(_as_tensor(mo_coeff), 2),
                                              h_ao=eng.to_padded(h, 2)), 2)[0]
    return _like(out, int1e_ao)


def int2e_transform(int2e_ao, mo_coeff):
    """Reference ``oo_energy.py:49-51``."""
    return uniform_4index_transform(int2e_ao, mo_coeff)


def mo_ao_to_mo_oao(mo_coeff, overlap):
    """``S^{1/2} C`` for numpy arrays (reference ``oo_energy.py:54-60``).  Initialisation-time
    helper on N x N host arrays; kept on the host like the reference's numpy implementation."""
    w, v = np.linalg.eigh(np.asarray(overlap))
    return (v * np.sqrt(w)) @ v.T @ np.asarray(mo_coeff)


def vector_to_skew_symmetric(vector):
    """Pack a vector into the strict lower triangle (``np.tril_indices`` order) of a skew matrix:
    ``[1..6] -> [[0,-1,-2,-4],[1,0,-3,-5],[2,3,0,-6],[4,5,6,0]]`` (reference ``oo_energy.py:63-87``).
    Pure index bookkeeping on the caller's array type (differentiable for torch)."""
    n = int(np.sqrt(8 * vector.shape[0] + 1) + 1) // 2
    rows, cols = np.tril_indices(n, k=-1)
    if torch.is_tensor(vector):
        r = torch.as_tensor(rows, device=vector.device)
        c = torch.as_tensor(cols, device=vector.device)
        out = torch.zeros((n, n), dtype=vector.dtype, device=vector.device)
        out = out.index_put((r, c), vector)
        return out.index_put((c, r), -vector)
    vector = np.asarray(vector)
    out = np.zeros((n, n), dtype=vector.dtype)
    out[rows, cols] = vector
    out[cols, rows] = -vector
    return out


def skew_symmetric_to_vector(kappa_matrix):
    """Reference ``oo_energy.py:90-94``."""
    rows, cols = np.tril_indices(kappa_matrix.shape[0], k=-1)
    return kappa_matrix[rows, cols]


def non_redundant_indices(occ_idx, act_idx, virt_idx, freeze_active):
    """Positions in the tril vector of the rotations that are not occ-occ, virt-virt or (when
    ``freeze_active``) act-act (reference ``oo_energy.py:97-118``)."""
    no, na, nv = len(occ_idx), len(act_idx), len(virt_idx)
    nao = no + na + nv
    cls = np.full(nao, -1)
    cls[np.asarray(occ_idx, dtype=int)] = 0
    cls[np.asarray(act_idx, dtype=int)] = 1
    cls[np.asarray(virt_idx, dtype=int)] = 2
    rows, cols = np.tril_indices(nao, -1)
    same = cls[rows] == cls[cols]
    redundant = same & ((cls[rows] == 0) | (cls[rows] == 2) | ((cls[rows] == 1) & bool(freeze_active)))
    params_idx = np.nonzero(~redundant)[0].astype(int)
    n_kappa = no * na + na * nv + no * nv + (0 if freeze_active else na * (na - 1) // 2)
    assert n_kappa == len(params_idx)
    return params_idx


# --------------------------------------------------------------------------------------
# autograd bridges: E and G are affine in the RDMs
# --------------------------------------------------------------------------------------
class _EnergyFn(torch.autograd.Function):
    """E = c0 + <c1, gamma> + <c2, Gamma> with the dot products done by ``oo_energy_f64``;
    dE/dgamma = c1, dE/dGamma = c2 (SURVEY Appendix A.4)."""

    @staticmethod
    def forward(ctx, one_rdm, two_rdm, eng, c0, c1, c2):
        E = eng.energy(c0, c1, c2, eng.dev(one_rdm), eng.dev(two_rdm))[0]
        ctx.c1 = c1[0].to(one_rdm.device)
        ctx.c2 = c2[0].to(two_rdm.device)
        return E.to(one_rdm.device)

    @staticmethod
    def backward(ctx, grad_out):
        return grad_out * ctx.c1, grad_out * ctx.c2, None, None, None, None


class _GradientFn(torch.autograd.Function):
    """G = 2 (F - F^T) by ``oo_fock_gradient_f64``; the adjoint w.r.t. (gamma, Gamma) by
    ``oo_fock_gradient_vjp_f64`` (SURVEY Appendix A.5)."""

    @staticmethod
    def forward(ctx, one_rdm, two_rdm, eng, ints):
        FI, FA, F, G, _ = ints.fock_gradient(eng.dev(one_rdm), eng.dev(two_rdm), want_vector=False)
        ctx.eng, ctx.ints, ctx.FI = eng, ints, FI
        ctx.hold = ints.hold()                       # backward reads the integrals: keep their buffer from reuse
        ctx.dev1, ctx.dev2 = one_rdm.device, two_rdm.device
        return eng.from_padded(G, 2)[0].to(one_rdm.device)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gbar):
        eng = ctx.eng
        g1, g2 = ctx.ints.fock_gradient_vjp(ctx.FI, eng.to_padded(gbar, 2))
        return g1.to(ctx.dev1), g2.to(ctx.dev2), None, None


_SECOND_ORDER_KAPPA = ("energy_from_kappa is differentiable once in kappa; for second derivatives in kappa use "
                       "analytic_hessian (or OrbitalHessian.matvec)")


def _wants_grad(*xs):
    return torch.is_grad_enabled() and any(torch.is_tensor(x) and x.requires_grad for x in xs)


class _KappaEnergyFn(torch.autograd.Function):
    """``energy_from_kappa`` for a kappa that requires grad: the forward is the plain evaluation (same kernels), and
    it keeps a hold on the transformed integrals for the backward.  dE/dgamma = c1, dE/dGamma = c2 as in
    :class:`_EnergyFn`; dE/dkappa by :class:`_KappaBarFn`."""

    @staticmethod
    def forward(ctx, kappa, one_rdm, two_rdm, oo):
        eng = oo.engine
        ints = oo._mo_integrals(kappa=kappa.detach())
        c0, c1, c2 = ints.active_hamiltonian()
        E = eng.energy(c0, c1, c2, eng.dev(one_rdm), eng.dev(two_rdm))[0]
        ctx.oo, ctx.ints = oo, ints
        ctx.hold = ints.hold()                       # backward reads the integrals: keep their buffer from reuse
        ctx.c1 = c1[0].to(one_rdm.device)
        ctx.c2 = c2[0].to(two_rdm.device)
        ctx.save_for_backward(kappa, one_rdm, two_rdm)
        return E.to(one_rdm.device)

    @staticmethod
    def backward(ctx, grad_out):
        kappa, one, two = ctx.saved_tensors
        kbar = _KappaBarFn.apply(kappa, one, two, grad_out, ctx.oo, ctx.ints) if ctx.needs_input_grad[0] else None
        return kbar, grad_out * ctx.c1, grad_out * ctx.c2, None


class _KappaBarFn(torch.autograd.Function):
    """``grad_out * dE/dkappa`` at ``C' = C expm(-K)``: with the full gradient matrix G = 2 (F - F^T) at C' (its
    act-act block included, also when those rotations are frozen), the cotangent of U is ``-U G / 2`` and the rotation's
    adjoint (``oo_kappa_rotation_vjp_f64``) maps it to kappa.  Its own backward raises: a second derivative in kappa
    needs the second Frechet derivative of exp, which is not implemented."""

    @staticmethod
    def forward(ctx, kappa, one_rdm, two_rdm, grad_out, oo, ints):
        eng = oo.engine
        kd = eng.dev(kappa).reshape(1, -1)
        U = eng.rotation(kd)
        G = ints.fock_gradient(eng.dev(one_rdm), eng.dev(two_rdm), want_matrix=True, want_vector=False)[3]
        kbar = eng.rotation_vjp(kd, eng.matmul(U[0], G[0], alpha=-0.5))[0]
        return kbar.to(device=kappa.device, dtype=kappa.dtype).reshape(kappa.shape) * grad_out.to(kappa.device)

    @staticmethod
    def backward(ctx, *grads):
        raise RuntimeError(_SECOND_ORDER_KAPPA)


class _RotationFn(torch.autograd.Function):
    """``U = expm(-K(kappa))`` (N x N); the backward is ``oo_kappa_rotation_vjp_f64``."""

    @staticmethod
    def forward(ctx, kappa, eng):
        ctx.eng = eng
        ctx.save_for_backward(kappa)
        U = eng.rotation(kappa.detach().reshape(1, -1))
        return _like(eng.from_padded(U, 2)[0], kappa)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, Ubar):
        kappa, = ctx.saved_tensors
        eng = ctx.eng
        kbar = eng.rotation_vjp(kappa.detach().reshape(1, -1), eng.to_padded(Ubar, 2)[None])[0]
        return kbar.to(device=kappa.device, dtype=kappa.dtype).reshape(kappa.shape), None


class _TransformedMOFn(torch.autograd.Function):
    """``M expm(-K(kappa))``; backward: ``Mbar = Outbar U^T``, ``Ubar = M^T Outbar`` -> ``oo_kappa_rotation_vjp_f64``."""

    @staticmethod
    def forward(ctx, mo_coeff, kappa, eng):
        U = eng.rotation(kappa.detach().reshape(1, -1))[0]
        M = eng.to_padded(mo_coeff, 2)
        ctx.eng, ctx.U, ctx.M = eng, U, M
        ctx.save_for_backward(mo_coeff, kappa)
        return _like(eng.from_padded(eng.matmul(M, U)[None], 2)[0], mo_coeff)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, out_bar):
        mo_coeff, kappa = ctx.saved_tensors
        eng = ctx.eng
        ob = eng.to_padded(out_bar, 2)
        mbar = kbar = None
        if ctx.needs_input_grad[0]:
            mbar = _like(eng.from_padded(eng.matmul(ob, ctx.U, transB=True)[None], 2)[0], mo_coeff)
        if ctx.needs_input_grad[1]:
            kbar = eng.rotation_vjp(kappa.detach().reshape(1, -1), eng.matmul(ctx.M, ob, transA=True)[None])[0]
            kbar = kbar.to(device=kappa.device, dtype=kappa.dtype).reshape(kappa.shape)
        return mbar, kbar, None


class PendingEvaluation:
    """Results of :meth:`OO_energy.energy_gradient_hessian` that may still be on their way to the host."""

    def __init__(self, results, event, copy):
        self._results, self._event, self._copy = results, event, copy

    def wait(self):
        """``(E, gradient, Hessian)`` once every device->host copy of the call has completed."""
        if self._event is not None:
            self._event.synchronize()
            self._event = None
        if self._copy:
            self._results = tuple(None if t is None else t.clone() for t in self._results)
            self._copy = False
        return self._results


def unpack_hessian(packed):
    """``(..., n (n+1)/2)`` lower triangle in ``np.tril_indices`` order (``hessian_format="packed"``) ->
    symmetric ``(..., n, n)``, in the array type of the input."""
    m = packed.shape[-1]
    n = (int(np.sqrt(8 * m + 1)) - 1) // 2
    assert n * (n + 1) // 2 == m
    rows, cols = np.tril_indices(n)
    if torch.is_tensor(packed):
        r = torch.as_tensor(rows, device=packed.device)
        c = torch.as_tensor(cols, device=packed.device)
        out = packed.new_empty(packed.shape[:-1] + (n, n))
    else:
        r, c = rows, cols
        out = np.empty(packed.shape[:-1] + (n, n), dtype=packed.dtype)
    out[..., r, c] = packed
    out[..., c, r] = packed
    return out


class OrbitalHessian:
    """Device-resident orbital Hessian in the I-space form (``T`` and ``F``, SURVEY Appendix A.6):
    what ``analytic_hessian`` returns instead of the reference's dense ``(N,N,N,N)`` tensor."""

    def __init__(self, eng, ints, F, one_rdm, two_rdm, like):
        self._eng, self._ints, self._F = eng, ints, F
        self._hold = ints.hold()                     # matrix() / dense() / matvec() / diagonal() read the integrals later
        self._d1, self._d2 = eng.dev(one_rdm), eng.dev(two_rdm)
        self._like = like
        self.shape = (eng.N,) * 4

    def matrix(self, pair_l=None, pair_r=None):
        """``H[l_j, r_j, l_k, r_k]`` for the engine's non-redundant pairs (or the given ones)."""
        return self._ints.hessian(self._F, self._d1, self._d2, pair_l=pair_l, pair_r=pair_r)

    def matvec(self, v):
        """``H @ v`` for ``v (n_kappa,)`` or ``(n_kappa, nv)`` (numpy or torch, any device), without forming H:
        one streamed pass over the transformed integrals per block of vectors.  Same shape, array type and device
        as ``v``."""
        eng = self._eng
        shape = tuple(v.shape)
        if len(shape) not in (1, 2) or shape[0] != eng.nk:
            raise ValueError(f"matvec expects ({eng.nk},) or ({eng.nk}, nv), got {shape}")
        V = eng.dev(v).reshape(eng.nk, 1 if len(shape) == 1 else shape[1])
        if V.numel() == 0:
            return _like(torch.zeros(shape, dtype=F64, device=eng.device), v)
        HV = self._ints.hessian_vector(self._F, self._d1, self._d2, V)
        return _like(HV.reshape(shape), v)

    def diagonal(self):
        """``matrix().diagonal()`` without forming H, ``(n_kappa,)`` in the array type of ``full_hessian_to_matrix``."""
        return _like(self._ints.hessian_diagonal(self._F, self._d1, self._d2), self._like)

    # ---- matrix-free second-order steps (auto_oo_b200/krylov.py): products and the diagonal only, H never formed
    def _device_matvec(self, v):
        shape = tuple(v.shape)
        V = v.reshape(self._eng.nk, -1).contiguous()
        return self._ints.hessian_vector(self._F, self._d1, self._d2, V).reshape(shape)

    def _device_diagonal(self):
        return self._ints.hessian_diagonal(self._F, self._d1, self._d2)

    def lowest_eigenpair(self, tol=1e-7, max_iter=200, info=None):
        """``(lambda_0, x_0)``: the lowest eigenvalue of H and its unit eigenvector (in the array type of
        :meth:`diagonal`) by Davidson on :meth:`matvec`, to ``||H x_0 - lambda_0 x_0|| <= tol``.  A negative
        ``lambda_0`` at a converged orbital optimisation means a saddle point, not a minimum."""
        from . import krylov
        if self._eng.nk == 0:
            raise ValueError("the Hessian has no parameters")
        lam, x = krylov.lowest_eigenpair(self._device_matvec, self._device_diagonal(), tol=tol, max_iter=max_iter,
                                         engine=self._eng, info=info)
        return lam, _like(x, self._like)

    def solve(self, rhs, shift=0.0, tol=1e-12, max_iter=1000, info=None):
        """``(H + shift)^-1 rhs`` by preconditioned CG on :meth:`matvec` (``H + shift`` must be positive definite),
        to ``||(H + shift) x - rhs|| <= tol ||rhs||``; same array type, device and shape as ``rhs (n_kappa,)``."""
        from . import krylov
        nk = self._eng.nk
        if tuple(rhs.shape) != (nk,):
            raise ValueError(f"solve expects ({nk},), got {tuple(rhs.shape)}")
        x = krylov.shifted_solve(self._device_matvec, self._device_diagonal(), self._eng.dev(rhs), shift=shift,
                                 tol=tol, max_iter=max_iter, engine=self._eng, info=info)
        return _like(x, rhs)

    def newton_step(self, gradient, mu=1e-6, rho=1.1, lambda_min=1e-6, aug=True, eig_tol=1e-7, lin_tol=1e-12,
                    eig_max_iter=200, lin_max_iter=1000, info=None):
        """``(dp, lambda_0)`` of ``NewtonStep.newton_step(gradient, matrix())`` without forming H: Davidson for the
        lowest eigenpair, deflated PCG for ``dp = -(H + sigma)^-1 g``.  ``dp`` has the array type, device and shape of
        ``gradient (n_kappa,)``.  ``aug=False`` with ``lambda_0 < lambda_min`` raises ``ValueError`` (indefinite
        system: use the formed matrix); no convergence raises ``RuntimeError``."""
        from . import krylov
        nk = self._eng.nk
        if tuple(gradient.shape) != (nk,):
            raise ValueError(f"newton_step expects a gradient of shape ({nk},), got {tuple(gradient.shape)}")
        dp, lam = krylov.newton_step(self._device_matvec, self._device_diagonal(), self._eng.dev(gradient), mu=mu,
                                     rho=rho, lambda_min=lambda_min, aug=aug, eig_tol=eig_tol, lin_tol=lin_tol,
                                     eig_max_iter=eig_max_iter, lin_max_iter=lin_max_iter, engine=self._eng, info=info)
        return _like(dp, gradient), lam

    def dense(self):
        """The reference's rank-4 tensor ``H[p,q,r,s]`` (``oo_energy.py:311-340``); O(N^4) memory."""
        N = self._eng.N
        idx = torch.arange(N, device=self._eng.device, dtype=torch.int32)
        pl = idx.repeat_interleave(N).contiguous()
        pr = idx.repeat(N).contiguous()
        return _like(self.matrix(pl, pr).reshape(N, N, N, N), self._like)


# --------------------------------------------------------------------------------------
# OO_energy                                                  (reference oo_energy.py:121-474)
# --------------------------------------------------------------------------------------
class OO_energy:
    """Orbital-optimised energy for any given RDMs, with analytic orbital gradient and Hessian
    (reference ``oo_energy.py:121-171``).  ``mol`` is duck-typed: ``int1e_ao, int2e_ao, overlap,
    oao_coeff, nuc, nao, get_active_space_idx`` (+ ``run_rhf``/``hf.mo_coeff`` when
    ``oao_mo_coeff`` is None)."""

    # bases up to this size are launch-bound: whole evaluations are replayed from CUDA graphs
    GRAPH_MAX_NAO = 128

    def __init__(self, mol, ncas, nelecas, oao_mo_coeff=None, freeze_active=False, interface='torch',
                 device=None, integral_path="class", eri_symmetry="auto", cuda_graphs="auto", eri_packing="8fold",
                 shard=None, group=None):
        """``integral_path``: ``"class"`` (default) transforms only the J/K integral classes that
        energy, gradient and Hessian read; ``"full"`` runs the complete four-index transform for
        every set of MO coefficients, as the reference does.  ``eri_symmetry``: ``"auto"`` lets the
        class path use the 8-fold symmetry of ``int2e_ao`` when the device check finds it (real-orbital
        integrals always have it), ``"off"`` never assumes it.  ``eri_packing``: ``"8fold"`` keeps the symmetric
        integrals with both pairs packed (an eighth of N^4, unpacked by the quarter-1 producer), ``"pair"`` with one.  ``cuda_graphs``: ``"auto"`` replays the batched
        evaluations (``energy_gradient_hessian``, ``energies_from_kappas``) from a CUDA graph when the basis has
        at most ``GRAPH_MAX_NAO`` orbitals, ``True`` / ``False`` force it."""
        assert integral_path in ("class", "full")
        assert cuda_graphs in ("auto", True, False)
        assert shard in (None, "pairs")
        pair_shard = None
        if shard == "pairs":
            # ONE evaluation over the ranks of `group` (torch.distributed must be initialised): every rank builds the
            # same OO_energy; `mol.int2e_ao` is the full tensor, or -- when `mol.int2e_packed_slab(lo, hi)` exists --
            # only this rank's slab of the 8-fold packed integrals is ever materialised (distributed.PairShard)
            from .distributed import PairShard
            pair_shard = PairShard(group, slab_given=hasattr(mol, "int2e_packed_slab"))
            assert integral_path == "class", "the sharded evaluation is the class path"
            cuda_graphs = False                               # a collective sits in the middle of every evaluation
        self.integral_path = integral_path
        self.cuda_graphs = (mol.nao <= self.GRAPH_MAX_NAO) if cuda_graphs == "auto" else bool(cuda_graphs)
        if interface != 'torch':
            raise ValueError("auto_oo_b200 implements the torch interface only (no JAX/XLA dispatch)")
        if oao_mo_coeff is None:
            mol.run_rhf()
            oao_mo_coeff = mo_ao_to_mo_oao(mol.hf.mo_coeff, mol.overlap)
        self.oao_mo_coeff = _as_tensor(oao_mo_coeff).detach().clone().to(F64)
        self.interface = interface

        self.overlap = mol.overlap
        self.nuc = mol.nuc
        self.nao = mol.nao
        self.ncas = ncas
        self.nelecas = nelecas
        self.occ_idx, self.act_idx, self.virt_idx = mol.get_active_space_idx(ncas, nelecas)
        no, na = len(self.occ_idx), len(self.act_idx)
        if not (np.array_equal(self.occ_idx, np.arange(no))
                and np.array_equal(self.act_idx, no + np.arange(na))
                and np.array_equal(self.virt_idx, np.arange(no + na, self.nao))):
            raise ValueError("orbital classes must be the contiguous ranges occ|act|virt "
                             "(what Moldata_pyscf.get_active_space_idx returns)")
        self.params_idx = non_redundant_indices(self.occ_idx, self.act_idx, self.virt_idx, freeze_active)
        self.n_kappa = len(self.params_idx)

        # integrals go to HBM once (padded layout); host copies are kept as the public attributes
        self.int1e_ao = _as_tensor(mol.int1e_ao)
        self.oao_coeff = _as_tensor(mol.oao_coeff)
        if pair_shard is not None and pair_shard.slab_given:
            from .distributed import pair_slab_range
            from .engine import pad_even
            ldp = pad_even(pad_even(self.nao) * (pad_even(self.nao) + 1) // 2)
            self.int2e_ao = _as_tensor(mol.int2e_packed_slab(*pair_slab_range(ldp, pair_shard.world, pair_shard.rank)))
            packed8 = None
        else:
            # `mol.int2e_packed8`: 8-fold packed integrals (io.load_problem(..., eri="packed")) instead of the dense tensor
            packed8 = getattr(mol, "int2e_packed8", None) if getattr(mol, "int2e_ao", None) is None else None
            self.int2e_ao = None if packed8 is not None else _as_tensor(mol.int2e_ao)
            if packed8 is not None and integral_path != "class":
                raise ValueError("8-fold packed integrals serve the class path only (integral_path='class')")
        self.engine = HotPathEngine(self.int1e_ao, self.int2e_ao if packed8 is None else None, self.oao_coeff, self.nuc,
                                    self.nao, no, na, self.params_idx, device=device, eri_symmetry=eri_symmetry,
                                    eri_packing=eri_packing, pair_shard=pair_shard,
                                    eri_packed8=None if packed8 is None else _as_tensor(packed8))

    # ------------------------------------------------------------------ orbitals
    @property
    def mo_coeff(self):
        """AO->MO coefficients ``X C_oao``; follows writes to ``oao_mo_coeff`` (``oo_energy.py:173-176``)."""
        eng = self.engine
        C = eng.mo_coeff(eng.to_padded(self.oao_mo_coeff, 2))
        return _like(eng.from_padded(C, 2)[0], self.oao_mo_coeff)

    def kappa_vector_to_matrix(self, kappa):
        """Reference ``oo_energy.py:213-219``."""
        kappa = _as_tensor(kappa)
        full = torch.zeros(self.nao * (self.nao - 1) // 2, dtype=kappa.dtype, device=kappa.device)
        full = full.index_put((torch.as_tensor(self.params_idx, device=kappa.device),), kappa)
        return vector_to_skew_symmetric(full)

    def kappa_matrix_to_vector(self, kappa_matrix):
        """Reference ``oo_energy.py:221-224``."""
        return skew_symmetric_to_vector(kappa_matrix)[self.params_idx]

    def kappa_to_mo_coeff(self, kappa):
        """``expm(-K(kappa))`` (reference ``oo_energy.py:226-230``) by ``oo_kappa_rotation_f64``; differentiable in a
        ``kappa`` tensor (backward: ``oo_kappa_rotation_vjp_f64``)."""
        eng = self.engine
        if _wants_grad(kappa):
            return _RotationFn.apply(kappa, eng)
        U = eng.rotation(_as_tensor(kappa).detach().reshape(1, -1))
        return _like(eng.from_padded(U, 2)[0], kappa)

    def get_transformed_mo(self, mo_coeff, kappa):
        """``mo_coeff @ expm(-K)`` (reference ``oo_energy.py:232-236``); differentiable in a ``kappa`` tensor and in
        a ``mo_coeff`` tensor (a numpy ``mo_coeff`` gives a numpy result, without a gradient)."""
        eng = self.engine
        if torch.is_tensor(mo_coeff) and torch.is_tensor(kappa) and _wants_grad(mo_coeff, kappa):
            return _TransformedMOFn.apply(mo_coeff, kappa, eng)
        U = eng.rotation(_as_tensor(kappa).detach().reshape(1, -1))
        out = eng.matmul(eng.to_padded(_as_tensor(mo_coeff), 2), U[0])
        return _like(eng.from_padded(out[None], 2)[0], mo_coeff)

    # ------------------------------------------------------------------ energy
    def _mo_integrals(self, mo_coeff=None, kappa=None):
        """Transformed integrals at ``mo_coeff`` (default: the current ``self.mo_coeff``, optionally rotated by
        ``kappa``), cached under what they were computed from: the same tensor object with an unchanged version
        counter, or equal values (compared on the host for host tensors), is a hit without a device round trip."""
        eng = self.engine
        if mo_coeff is None:
            src = _as_tensor(self.oao_mo_coeff)               # (callers may have assigned a numpy array)
            if kappa is None:
                make = lambda: eng.mo_coeff(eng.to_padded(src, 2))[0]
            else:
                make = lambda: eng.mo_coeff(eng.to_padded(src, 2), eng.rotation(kappa.reshape(1, -1)))[0]
            return eng.integrals_for(self.integral_path, "oao", src, make, kappa=kappa)
        src = _as_tensor(mo_coeff)
        return eng.integrals_for(self.integral_path, "mo", src, lambda: eng.to_padded(src.detach(), 2))

    def get_active_integrals(self, mo_coeff):
        """``(c0, c1, c2)`` of the active-space Hamiltonian in chemist notation
        (reference ``oo_energy.py:204-211``, ``utils/active_space.py:177-212``)."""
        c0, c1, c2 = self._mo_integrals(mo_coeff).active_hamiltonian()
        return _like(c0[0], mo_coeff), _like(c1[0], mo_coeff), _like(c2[0], mo_coeff)

    def energy_from_mo_coeff(self, mo_coeff, one_rdm, two_rdm):
        """Reference ``oo_energy.py:178-197``.  0-d tensor, differentiable in the RDMs."""
        c0, c1, c2 = self._mo_integrals(mo_coeff).active_hamiltonian()
        one, two = _as_tensor(one_rdm), _as_tensor(two_rdm)
        return _EnergyFn.apply(one, two, self.engine, c0, c1, c2)

    def energy_from_kappa(self, kappa, one_rdm, two_rdm):
        """Energy at ``C' = C expm(-K(kappa))`` (reference ``oo_energy.py:199-202``).  Differentiable in the RDMs
        (to any order) and, for a ``kappa`` tensor that requires grad, once in ``kappa``: the gradient comes back on
        ``kappa``'s device and dtype; a second derivative in ``kappa`` raises ``RuntimeError``."""
        if _wants_grad(kappa):
            return _KappaEnergyFn.apply(kappa, _as_tensor(one_rdm), _as_tensor(two_rdm), self)
        c0, c1, c2 = self._mo_integrals(kappa=_as_tensor(kappa).detach()).active_hamiltonian()
        return _EnergyFn.apply(_as_tensor(one_rdm), _as_tensor(two_rdm), self.engine, c0, c1, c2)

    def energies_from_kappas(self, kappas, one_rdm, two_rdm):
        """``energy_from_kappa`` for a batch ``kappas (B, n_kappa)`` in one pass (batched launches);
        returns ``(B,)`` on the device of ``kappas``.  Used by the speculative line search.  Not differentiable:
        ``kappas`` and the RDMs are detached."""
        eng = self.engine
        kappas = _as_tensor(kappas).detach().reshape(-1, self.n_kappa)
        run = eng.evaluate_graphed if self.cuda_graphs else eng.evaluate
        E, _, _ = run(eng.to_padded(self.oao_mo_coeff, 2), eng.dev(one_rdm), eng.dev(two_rdm),
                      kappa=eng.dev(kappas), want_hessian=False, path=self.integral_path)
        return E.to(kappas.device)

    # ------------------------------------------------------------------ Fock matrices / gradient
    def _padded_integrals(self, int1e_mo, int2e_mo):
        eng = self.engine
        return eng.to_padded(_as_tensor(int1e_mo), 2)[None], eng.to_padded(_as_tensor(int2e_mo), 4)[None]

    def _given_integrals(self, int1e_mo, int2e_mo):
        """Caller-supplied dense MO integrals (the ``*_from_integrals`` methods)."""
        from .engine import MOIntegrals
        h, g = self._padded_integrals(int1e_mo, int2e_mo)
        return MOIntegrals(self.engine, "full", h=h, g=g)

    def fock_core(self, int1e_mo, int2e_mo):
        """``F^I`` (reference ``oo_energy.py:272-284``)."""
        h, g = self._padded_integrals(int1e_mo, int2e_mo)
        d1 = torch.zeros(self.ncas, self.ncas, dtype=F64, device=self.engine.device)
        d2 = torch.zeros((self.ncas,) * 4, dtype=F64, device=self.engine.device)
        FI = self.engine.fock_gradient(h, g, d1, d2, want_matrix=False, want_vector=False)[0]
        return _like(self.engine.from_padded(FI, 2)[0], int1e_mo)

    def fock_active(self, int2e_mo, one_rdm):
        """``F^A`` (reference ``oo_energy.py:286-298``)."""
        eng = self.engine
        g = eng.to_padded(_as_tensor(int2e_mo), 4)[None]
        h = torch.zeros(1, eng.ld, eng.ld, dtype=F64, device=eng.device)
        d2 = torch.zeros((self.ncas,) * 4, dtype=F64, device=eng.device)
        FA = eng.fock_gradient(h, g, eng.dev(one_rdm), d2, want_matrix=False, want_vector=False)[1]
        return _like(eng.from_padded(FA, 2)[0], int2e_mo)

    def fock_generalized(self, int1e_mo, int2e_mo, one_rdm, two_rdm):
        """Generalized Fock matrix (reference ``oo_energy.py:238-270``)."""
        h, g = self._padded_integrals(int1e_mo, int2e_mo)
        eng = self.engine
        F = eng.fock_gradient(h, g, eng.dev(one_rdm), eng.dev(two_rdm), want_matrix=False, want_vector=False)[2]
        return _like(eng.from_padded(F, 2)[0], int1e_mo)

    def analytic_gradient_from_integrals(self, int1e_mo, int2e_mo, one_rdm, two_rdm):
        """``G = 2 (F - F^T)`` (reference ``oo_energy.py:300-309``)."""
        ints = self._given_integrals(int1e_mo, int2e_mo)
        return _GradientFn.apply(_as_tensor(one_rdm), _as_tensor(two_rdm), self.engine, ints)

    def analytic_gradient(self, one_rdm, two_rdm, mo_coeff=None):
        """Reference ``oo_energy.py:404-413``; differentiable in the RDMs."""
        ints = self._mo_integrals(mo_coeff)
        return _GradientFn.apply(_as_tensor(one_rdm), _as_tensor(two_rdm), self.engine, ints)

    # ------------------------------------------------------------------ Hessian
    def full_rdms(self, one_rdm, two_rdm):
        """RDMs embedded in the full orbital space (reference ``oo_energy.py:342-379``).  Dense
        N^2 / N^4 buffers exactly as the reference defines them; the Hessian kernels never build
        these (they are zero outside occ+act), the method exists for API parity."""
        eng = self.engine
        d1, d2 = eng.full_rdms(eng.dev(one_rdm), eng.dev(two_rdm))
        return d1.cpu().numpy(), d2.cpu().numpy()

    def y_matrix(self, int2e_mo, two_full):
        """Reference ``oo_energy.py:381-393`` for arbitrary dense ``two_full``: three
        ``N^2 x N^2 x N^2`` contractions on the TN-DGEMM kernel."""
        eng = self.engine
        out = eng.y_matrix_dense(_as_tensor(int2e_mo), _as_tensor(two_full))
        return _like(out, int2e_mo)

    def analytic_hessian_from_integrals(self, int1e_mo, int2e_mo, one_rdm, two_rdm):
        """Reference ``oo_energy.py:311-340``; returns an :class:`OrbitalHessian`."""
        return self._hessian(self._given_integrals(int1e_mo, int2e_mo), one_rdm, two_rdm, int1e_mo)

    def analytic_hessian(self, one_rdm, two_rdm, mo_coeff=None):
        """Reference ``oo_energy.py:415-424``; returns an :class:`OrbitalHessian`."""
        return self._hessian(self._mo_integrals(mo_coeff), one_rdm, two_rdm, _as_tensor(one_rdm))

    def _hessian(self, ints, one_rdm, two_rdm, like):
        eng = self.engine
        d1, d2 = eng.dev(one_rdm), eng.dev(two_rdm)
        F = ints.fock_gradient(d1, d2, want_matrix=False, want_vector=False)[2]
        return OrbitalHessian(eng, ints, F, d1, d2, like)

    def full_hessian_to_matrix(self, full_hess):
        """``(N,N,N,N)`` -> ``(n_kappa, n_kappa)`` (reference ``oo_energy.py:395-402``).  Accepts the
        :class:`OrbitalHessian` of ``analytic_hessian`` (fused assembly on device) or any dense
        rank-4 array (plain gather, as in the reference)."""
        if isinstance(full_hess, OrbitalHessian):
            return _like(full_hess.matrix(), full_hess._like)
        rows, cols = np.tril_indices(self.nao, k=-1)
        part = full_hess[rows, cols, :, :][:, rows, cols]
        return part[self.params_idx, :][:, self.params_idx]

    # ------------------------------------------------------------------ batched evaluation
    def energy_gradient_hessian(self, kappa, one_rdm, two_rdm, want_hessian=True, hessian_format="dense",
                                pinned_results=False, wait=True):
        """``E``, packed gradient and Hessian matrix at ``C expm(-K(kappa_b))`` for a batch of
        rotations ``kappa (B, n_kappa)`` -- the three reference calls ``energy_from_kappa``,
        ``kappa_matrix_to_vector(analytic_gradient(mo_coeff=C'))`` and
        ``full_hessian_to_matrix(analytic_hessian(mo_coeff=C'))`` fused so that one four-index
        transform serves all three.  CUDA tensors in -> fresh CUDA tensors out.  Host tensors in (staged through
        pinned memory) -> host tensors out: ``(B,)``, ``(B, n_kappa)`` and the Hessians, which travel to the host
        on a copy stream while the next evaluation computes.

        ``hessian_format``: ``"dense"`` -> ``(B, n_kappa, n_kappa)``; ``"packed"`` -> ``(B, n_kappa (n_kappa+1)/2)``,
        the lower triangle of the symmetric matrix in ``np.tril_indices`` order (:func:`unpack_hessian` restores
        the matrix) -- half the device->host bytes, which is what bounds the end-to-end rate at N = 256.
        ``pinned_results=False`` (default): the host results are fresh tensors owned by the caller, as in the
        reference.  ``True``: they are views of the engine's pinned staging buffers -- no second copy of a 765 MB
        Hessian -- of which there are two sets used in turn: results stay valid until the call after next.
        ``wait=False`` returns a :class:`PendingEvaluation` at once; its ``wait()`` gives the results.  With at most
        two calls in flight the copies of one call overlap the computation of the next."""
        assert hessian_format in ("dense", "packed")
        eng = self.engine
        kappa = _as_tensor(kappa).detach().reshape(-1, self.n_kappa)
        one, two = _as_tensor(one_rdm).detach(), _as_tensor(two_rdm).detach()
        on_host = kappa.device.type == "cpu"
        packed = hessian_format == "packed" and want_hessian
        Coao = eng.resident_oao(self.oao_mo_coeff)
        B, nk = kappa.shape[0], self.n_kappa
        if on_host and B == 1 and not bool(kappa.any()):
            kappa = None                                   # expm(0) = 1: the rotation stage is skipped altogether
        if not on_host:
            run = eng.evaluate_graphed if self.cuda_graphs else eng.evaluate
            E, G, H = run(Coao, one, two, kappa=kappa, want_hessian=want_hessian, path=self.integral_path)
            out = (E, G, eng.pack_lower(H) if packed else H)
            return out if wait else PendingEvaluation(out, None, False)

        # ---- host face: alternate between two sets of pinned staging buffers
        self._result_slot = slot = (getattr(self, "_result_slot", -1) + 1) % 2
        shapes = {"E": (B,), "G": (B, nk), "kappa": (B, nk), "rdm1": tuple(one.shape), "rdm2": tuple(two.shape)}
        if want_hessian:
            shapes["H"] = (B, nk * (nk + 1) // 2) if packed else (B, nk, nk)
        ent = eng.result_slot(slot, shapes)
        if ent["done"] is not None:
            ent["done"].synchronize()                      # the call before last has landed (normally long ago)
        host = ent["host"]
        main = torch.cuda.current_stream(eng.device)
        # inputs: pinned staging, read by a kernel (a DMA copy on the compute stream would queue behind the
        # device->host copy of the previous call's last Hessian)
        host["rdm1"].copy_(one)
        host["rdm2"].copy_(two)
        d1, d2 = eng.upload_pinned(host["rdm1"]), eng.upload_pinned(host["rdm2"])
        kd = squarings = None
        if kappa is not None:
            host["kappa"].copy_(kappa)
            kd = eng.upload_pinned(host["kappa"])
            if self.nao > eng.lib.oo_expm_device_squarings_max_n():
                # decided from the HOST copy: the device variant ends in a scalar device->host copy, which would
                # wait behind the previous call's Hessian on the copy engine
                squarings = eng.squarings_for(kappa)
        done = torch.cuda.Event()
        if self.cuda_graphs:
            # launch-bound sizes: one graph replay, results straight from the graph's output buffers
            E, G, H = eng.evaluate_graphed(Coao, d1, d2, kappa=kd, want_hessian=want_hessian,
                                           path=self.integral_path, clone=False)
            host["E"].copy_(E, non_blocking=True)
            host["G"].copy_(G, non_blocking=True)
            if want_hessian:
                host["H"].copy_(eng.pack_lower(H) if packed else H, non_blocking=True)
            done.record(main)
        else:
            # the Hessian of evaluation b goes to pinned host memory on a copy stream while evaluation b+1 computes
            side = eng.copy_stream()
            H_dev = eng.workspace_tensor("H_batch", (B, nk, nk)) if want_hessian else None
            Hp_dev = eng.workspace_tensor(("H_packed", slot), (B, nk * (nk + 1) // 2)) if packed else None
            if want_hessian and not packed:
                main.wait_stream(side)                     # dense copies of the previous call read H_dev itself

            def ship(b):
                if not want_hessian:
                    return
                src = H_dev[b]
                if packed:
                    eng.pack_lower(H_dev[b:b + 1], out=Hp_dev[b:b + 1])
                    src = Hp_dev[b]
                ev = torch.cuda.Event()
                ev.record(main)
                side.wait_event(ev)
                with torch.cuda.stream(side):
                    host["H"][b].copy_(src, non_blocking=True)

            E, G, _ = eng.evaluate(Coao, d1, d2, kappa=kd, want_hessian=want_hessian, squarings=squarings,
                                   path=self.integral_path, H_out=H_dev, on_result=ship)
            side.wait_stream(main)
            with torch.cuda.stream(side):                  # every device->host copy of the call is on the copy stream
                host["E"].copy_(E, non_blocking=True)
                host["G"].copy_(G, non_blocking=True)
            E.record_stream(side)
            G.record_stream(side)
            done.record(side)
        ent["done"] = done
        pending = PendingEvaluation((host["E"], host["G"], host["H"] if want_hessian else None), done,
                                    copy=not pinned_results)
        return pending.wait() if wait else pending

    def energy_gradient_newton_direction(self, kappa, one_rdm, two_rdm, matrix_free=False, **newton_kwargs):
        """Device-resident Newton mode of :meth:`energy_gradient_hessian`: for every rotation of the batch the
        Hessian is built AND consumed in HBM -- ``NewtonStep.newton_step`` (one ``eigh`` on the device, the
        augmented-Hessian shift of ``utils/newton_raphson.py:78-129``) -- and only ``E (B,)``, the gradient
        ``(B, n_kappa)``, the Newton direction ``(B, n_kappa)`` and the lowest Hessian eigenvalue ``(B,)`` come
        back (on the device of ``kappa``).  ``newton_kwargs`` go to :class:`NewtonStep` (``mu, rho, lambda_min, aug``).
        ``matrix_free=True``: each rotation evaluates E and G only, and the step comes from an :class:`OrbitalHessian`
        on that rotation's transformed integrals (Davidson + deflated CG on products, ``OrbitalHessian.newton_step``):
        H is never formed, E and G are the same, the direction and eigenvalue agree to the solver tolerances."""
        eng = self.engine
        kappa = _as_tensor(kappa).detach().reshape(-1, self.n_kappa)
        dev_in = kappa.device
        opt = NewtonStep(verbose=0, **newton_kwargs)
        Coao = eng.to_padded(self.oao_mo_coeff, 2)
        d1, d2, kd = eng.dev(_as_tensor(one_rdm).detach()), eng.dev(_as_tensor(two_rdm).detach()), eng.dev(kappa)
        B = kd.shape[0]
        dk = torch.empty(B, self.n_kappa, dtype=F64, device=eng.device)
        lam = torch.empty(B, dtype=F64)
        Es, Gs = [], []
        if matrix_free:
            for b in range(B):
                d1b, d2b = d1[b:b + 1] if d1.dim() == 3 else d1, d2[b:b + 1] if d2.dim() == 5 else d2

                def step(_, ints, F, g):                         # while this rotation's integrals are current
                    dk[b], lam[b] = opt.newton_step(g, OrbitalHessian(eng, ints, F, d1b, d2b, d1b))
                E, G, _ = eng.evaluate(Coao, d1b, d2b, kappa=kd[b:b + 1], want_hessian=False, path=self.integral_path,
                                       on_integrals=step)
                Es.append(E)
                Gs.append(G)
            return (torch.cat(Es).to(dev_in), torch.cat(Gs).to(dev_in), dk.to(dev_in), lam.to(dev_in))
        H = eng.workspace_tensor("H_newton", (1, self.n_kappa, self.n_kappa))
        for b in range(B):                                   # one Hessian resident at a time
            E, G, _ = eng.evaluate(Coao, d1[b:b + 1] if d1.dim() == 3 else d1, d2[b:b + 1] if d2.dim() == 5 else d2,
                                   kappa=kd[b:b + 1], H_out=H, path=self.integral_path)
            dk[b], lam[b] = opt.newton_step(G[0], H[0])
            Es.append(E)
            Gs.append(G)
        return (torch.cat(Es).to(dev_in), torch.cat(Gs).to(dev_in), dk.to(dev_in), lam.to(dev_in))

    # ------------------------------------------------------------------ driver
    def orbital_optimization(self, one_rdm, two_rdm, conv_tol=1e-8, max_iterations=100, verbose=0,
                             matrix_free=False, **kwargs):
        """Damped-Newton orbital optimisation at fixed RDMs; mutates ``oao_mo_coeff`` and returns
        the energy trajectory (reference ``oo_energy.py:426-474``: re-base after every step,
        convergence tested only for ``n > 1``, per-iteration line printed unless ``verbose`` is None).
        ``matrix_free=True``: every iteration takes the gradient and the :class:`OrbitalHessian` at the current
        orbitals (one transform, shared through the integral cache) and ``NewtonStep`` steps on its products; the
        n_kappa^2 Hessian is never formed.  The trajectory equals the default one to the solver tolerances."""
        objective_fn = partial(self.energy_from_kappa, one_rdm=one_rdm, two_rdm=two_rdm)
        # batched form for NewtonStep(speculate=k): a list of (kappa,) tuples -> energies
        objective_fn.batched = lambda plist: self.energies_from_kappas(
            torch.stack([_as_tensor(p[0]) for p in plist]), one_rdm, two_rdm)
        opt = NewtonStep(verbose=verbose, **kwargs)
        energy_l = []
        if verbose:
            energy = self.energy_from_mo_coeff(self.mo_coeff, one_rdm, two_rdm).item()
            print(f"Starting energy: {energy:.12f}")
        one = _as_tensor(one_rdm)
        for n in range(max_iterations):
            kappa = torch.zeros(self.n_kappa, dtype=F64, device=one.device)
            # gradient and Hessian at the current orbitals from ONE fused evaluation (one transform, one graph
            # replay for small bases) instead of the reference's analytic_gradient + analytic_hessian calls
            if matrix_free:
                ints = self._mo_integrals()
                d1, d2 = self.engine.dev(one_rdm), self.engine.dev(two_rdm)
                _, _, F, _, gv = ints.fock_gradient(d1, d2, want_matrix=False)
                gradient = gv[0].to(one.device)
                # damped_newton_step in two parts: the OrbitalHessian (and its hold on the integrals) is released
                # before the line search, whose transforms then reuse the cached class buffer
                dp, lowest_eigenvalue = opt.newton_step(gradient, OrbitalHessian(self.engine, ints, F, d1, d2, d1))
                kappa, _ = opt.backtracking(objective_fn, (kappa,), dp, gradient)
            else:
                _, G, H = self.energy_gradient_hessian(kappa[None], one_rdm, two_rdm)
                gradient, hessian = G[0], H[0]
                kappa, lowest_eigenvalue = opt.damped_newton_step(objective_fn, (kappa,), gradient, hessian)
            self.oao_mo_coeff = self.get_transformed_mo(self.oao_mo_coeff, kappa)
            energy = self.energy_from_mo_coeff(self.mo_coeff, one_rdm, two_rdm).item()
            energy_l.append(energy)
            if verbose is not None:
                print(f"iter = {n:03}, energy = {energy:.12f}")
            if n > 1 and abs(energy_l[-1] - energy_l[-2]) < conv_tol:
                if verbose:
                    print("Orbital optimization finished.")
                    print("E_fin =", energy_l[-1])
                break
        return energy_l


class OO_energy_geometries:
    """Many molecular geometries of one system (same basis size, same active space) evaluated
    together -- the shape of the Berry-phase loop (``examples/Tutorial_Berry_phase.ipynb`` cell 22:
    one ``Moldata_pyscf`` / ``OO_pqc`` per geometry, each needing energy, orbital gradient and
    Hessian at its own integrals).  Every stage is ONE batched launch over the geometries.

    ``mols``: sequence of duck-typed ``Moldata_pyscf`` objects; ``oao_mo_coeff``: ``(G, N, N)`` (or
    one ``(N, N)`` matrix used for all).  ``energy_gradient_hessian(kappa, one_rdm, two_rdm)`` takes
    ``kappa (G, n_kappa)`` and RDMs shared ``(na,na)/(na^4)`` or per geometry ``(G, ...)``.  Its results are not
    differentiable: ``kappa`` and the RDMs are detached."""

    def __init__(self, mols, ncas, nelecas, oao_mo_coeff, freeze_active=False, device=None,
                 eri_symmetry="auto", cuda_graphs="auto"):
        mols = list(mols)
        self.cuda_graphs = (mols[0].nao <= OO_energy.GRAPH_MAX_NAO) if cuda_graphs == "auto" else bool(cuda_graphs)
        self._Coao_dev = self._Coao_src = None
        assert len(mols) > 0
        self.nao = mols[0].nao
        assert all(m.nao == self.nao for m in mols), "all geometries must share the basis size"
        self.ncas, self.nelecas = ncas, nelecas
        self.occ_idx, self.act_idx, self.virt_idx = mols[0].get_active_space_idx(ncas, nelecas)
        self.params_idx = non_redundant_indices(self.occ_idx, self.act_idx, self.virt_idx, freeze_active)
        self.n_kappa = len(self.params_idx)
        self.n_geometries = G = len(mols)
        stack = lambda name: torch.stack([_as_tensor(getattr(m, name)) for m in mols])
        self.engine = HotPathEngine(stack("int1e_ao"), stack("int2e_ao"), stack("oao_coeff"),
                                    np.array([m.nuc for m in mols], dtype=np.float64), self.nao,
                                    len(self.occ_idx), len(self.act_idx), self.params_idx, device=device,
                                    n_geometries=G, eri_symmetry=eri_symmetry)
        self.engine.drop_full_eri()                       # only the class path's copy of the integrals is needed
        C = _as_tensor(oao_mo_coeff).detach().to(F64)
        self.oao_mo_coeff = C if C.dim() == 3 else C[None].repeat(G, 1, 1)
        assert self.oao_mo_coeff.shape[0] == G

    def energy_gradient_hessian(self, kappa, one_rdm, two_rdm, want_hessian=True, pinned_results=False):
        """``(E (G,), gradient (G, n_kappa), Hessian (G, n_kappa, n_kappa))`` at
        ``C_g expm(-K(kappa_g))`` for every geometry ``g``; results on the device of ``kappa``.  Host results are
        fresh tensors; with ``pinned_results=True`` they are views of the reused pinned staging buffers instead
        (valid until the next call).  The whole pass is one CUDA-graph launch when ``cuda_graphs`` is on."""
        eng = self.engine
        kappa = _as_tensor(kappa).detach().reshape(self.n_geometries, self.n_kappa)
        one, two = _as_tensor(one_rdm).detach(), _as_tensor(two_rdm).detach()
        on_host = kappa.device.type == "cpu"
        src = (self.oao_mo_coeff, self.oao_mo_coeff._version)          # follows re-assignment and in-place writes
        if self._Coao_dev is None or self._Coao_src[0] is not src[0] or self._Coao_src[1] != src[1]:
            self._Coao_dev = eng.to_padded(self.oao_mo_coeff, 2, batch=self.n_geometries)
            self._Coao_src = src
        if on_host:
            kappa, one, two = (eng.stage_pinned(k, t.to(F64)) for k, t in
                               (("kappa", kappa), ("rdm1", one), ("rdm2", two)))
        if self.cuda_graphs:
            E, G, H = eng.evaluate_graphed(self._Coao_dev, one, two, kappa=kappa, want_hessian=want_hessian,
                                           path="class", clone=not on_host)
        else:
            E, G, H = eng.evaluate(self._Coao_dev, eng.dev(one), eng.dev(two), kappa=eng.dev(kappa),
                                   want_hessian=want_hessian, path="class")
        if not on_host:
            return E, G, H
        out = (eng.stage_out("E", E), eng.stage_out("G", G), eng.stage_out("H", H) if want_hessian else None)
        torch.cuda.current_stream(eng.device).synchronize()
        return out if pinned_results else tuple(None if t is None else t.clone() for t in out)

    def rotate(self, kappa):
        """``C_g <- C_g expm(-K(kappa_g))`` for every geometry (the re-basing step of the loop)."""
        eng = self.engine
        U = eng.rotation(_as_tensor(kappa).detach().reshape(self.n_geometries, self.n_kappa))
        Coao = eng.to_padded(self.oao_mo_coeff, 2, batch=self.n_geometries)
        new = torch.stack([eng.matmul(Coao[g], U[g]) for g in range(self.n_geometries)])
        self.oao_mo_coeff = eng.from_padded(new, 2).to(self.oao_mo_coeff.device)
