"""CPU: the float64 reference of the kappa adjoint that ``tests/test_gpu_kappa_adjoint.py`` compares the device with.

For U = expm(-K(kappa)) and a cotangent Ubar = df/dU, the VJP is Kbar = -L(K, Ubar) (L: Frechet derivative of exp,
``scipy.linalg.expm_frechet``), gathered as kappa_bar_j = Kbar[l_j,r_j] - Kbar[r_j,l_j].  For the energy at
C' = C U the cotangent is Ubar = -U G / 2 with G = 2 (F - F^T) the FULL gradient matrix at C' (its act-act block
included, also when those rotations are frozen).  Both are checked against torch autograd through
``torch.linalg.matrix_exp`` and the oracle energy."""
import numpy as np
import pytest
import scipy.linalg
import torch

from oracle import oo_oracle as orc
from helpers import load_case

F64 = torch.float64


def skew(kappa, pl, pr, n):
    K = np.zeros((n, n))
    K[pl, pr] = kappa
    K[pr, pl] = -kappa
    return K


def rotation_vjp_reference(kappa, pl, pr, n, Ubar):
    """kappa_bar of U = expm(-K(kappa)) for the cotangent Ubar (n x n), float64."""
    L = scipy.linalg.expm_frechet(skew(np.asarray(kappa, dtype=np.float64), pl, pr, n), np.asarray(Ubar),
                                  compute_expm=False)
    return -(L[pl, pr] - L[pr, pl])


def energy_vjp_reference(p, one_rdm, two_rdm, kappa, drop_act_act=False):
    """dE/dkappa of the oracle energy at C' = C expm(-K(kappa)) from the full gradient matrix."""
    rows, cols = np.tril_indices(p.nao, k=-1)
    pl, pr = rows[p.params_idx], cols[p.params_idx]
    U = orc.rotation_from_kappa(kappa, p.params_idx, p.nao).numpy()
    h, g = p.mo_integrals(kappa)
    G = orc.gradient_matrix(h, g, one_rdm, two_rdm, p.occ_idx, p.act_idx).numpy()
    if drop_act_act:
        act = np.asarray(p.act_idx)
        G[np.ix_(act, act)] = 0.0
    return rotation_vjp_reference(np.asarray(kappa), pl, pr, p.nao, -0.5 * U @ G)


def autograd_energy_gradient(p, one_rdm, two_rdm, kappa):
    k = torch.as_tensor(kappa, dtype=F64).clone().requires_grad_(True)
    C = p.mo_coeff @ torch.linalg.matrix_exp(-orc.kappa_to_skew_diff(k, p.params_idx, p.nao))
    hh, gg = orc.transform_1e(p.h_ao, C), orc.transform_2e(p.g_ao, C)
    c0, c1, c2 = orc.hamiltonian_coefficients(p.nuc, hh, gg, p.occ_idx, p.act_idx)
    E = orc.energy_from_coefficients(c0, c1, c2, one_rdm, two_rdm)
    return torch.autograd.grad(E, k)[0].numpy()


@pytest.mark.parametrize("norm1", [0.0, 0.3, 0.95, 2.0, 9.0, 30.0])
def test_rotation_vjp_reference_matches_autograd(norm1):
    n = 9
    rng = np.random.default_rng(int(norm1 * 10) + 1)
    pl, pr = np.tril_indices(n, k=-1)
    kappa = rng.standard_normal(len(pl))
    K = skew(kappa, pl, pr, n)
    if norm1 > 0:
        kappa *= norm1 / np.abs(K).sum(axis=0).max()
    else:
        kappa[:] = 0.0
    Ubar = rng.standard_normal((n, n))
    ref = rotation_vjp_reference(kappa, pl, pr, n, Ubar)
    k = torch.as_tensor(kappa).requires_grad_(True)
    Kt = torch.zeros(n, n, dtype=F64).index_put((torch.as_tensor(pl), torch.as_tensor(pr)), k)
    Kt = Kt.index_put((torch.as_tensor(pr), torch.as_tensor(pl)), -k)
    (torch.linalg.matrix_exp(-Kt) * torch.as_tensor(Ubar)).sum().backward()
    auto = k.grad.numpy()
    assert np.abs(ref - auto).max() <= 1e-12 * max(1.0, np.abs(auto).max())


@pytest.mark.parametrize("name", ["n7_cas44", "n13_cas22", "n8_nocore", "n13_bigkappa"])
def test_energy_vjp_reference_matches_oracle_autograd(name):
    c = load_case(name)
    p = c.oracle()
    kappa = 3.0 * c.kappa
    assert kappa.abs().max().item() > 0
    ref = energy_vjp_reference(p, c.one_rdm, c.two_rdm, kappa)
    auto = autograd_energy_gradient(p, c.one_rdm, c.two_rdm, kappa)
    assert np.abs(ref - auto).max() <= 1e-10 * max(1.0, np.abs(auto).max())


def test_frozen_active_needs_the_act_act_block():
    """With freeze_active the act-act rotations are not parameters, but that block of G still enters the adjoint."""
    c = load_case("n13_cas22")
    assert c.freeze
    p = c.oracle()
    kappa = 3.0 * c.kappa
    auto = autograd_energy_gradient(p, c.one_rdm, c.two_rdm, kappa)
    dropped = energy_vjp_reference(p, c.one_rdm, c.two_rdm, kappa, drop_act_act=True)
    assert np.abs(dropped - auto).max() > 1e-2
