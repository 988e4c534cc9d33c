"""What the matrix-free Hessian kernels compute, checked on the CPU class oracle.

For a vector v (n_kappa) with skew matrix V (V[l_j, r_j] = v_j = -V[r_j, l_j]):

    W[p,q]  = -((F + F^T) V)[p,q] + [p in I] sum_{r in I, s} T[(p r),(q s)] V[r,s]
    (H v)_j = W[l_j, r_j] - W[r_j, l_j]
    H_jj    = X(l,r,l,r) - X(l,r,r,l) - X(r,l,l,r) + X(r,l,r,l)

and the T part never needs T: with T = sum_k A_k (x) B_k over the class rows k (A_k[p,r] the RDM coefficients,
B_k[q,s] a class plane), sum_{r,s} T[(p r),(q s)] V[r,s] = sum_k sum_s B_k[q,s] M_k[p,s], M_k = A_k V_I.
"""
import numpy as np
import pytest
import torch

from helpers import load_case
from oracle import class_oracle as co
from oracle import oo_oracle as orc

DT = torch.float64
CASES = ["n7_cas44", "n7_cas44_frozen", "n8_nocore", "n11_cas43", "n13_cas22"]


def _evaluation(name):
    c = load_case(name)
    p = co.ClassProblem(c.int1e_ao, c.int2e_ao, c.oao_coeff, c.oao_mo_coeff, c.nuc, c.nelec, c.ncas, c.nelecas,
                        c.freeze)
    return c, p.at(c.kappa)


def _skew(ev, v):
    rr, cc = orc.tril_pairs(ev.N)
    L = torch.as_tensor(rr[ev.params_idx], dtype=torch.long)
    R = torch.as_tensor(cc[ev.params_idx], dtype=torch.long)
    V = torch.zeros(v.shape[1], ev.N, ev.N, dtype=DT)
    V[:, L, R] = v.T
    V[:, R, L] = -v.T
    return V, L, R


@pytest.mark.parametrize("name", CASES)
def test_hessian_vector_product_and_diagonal_identities(name):
    c, ev = _evaluation(name)
    one, two = c.one_rdm, c.two_rdm
    H = ev.hessian(one, two)
    t = ev._t_matrix(one, two)                                  # T[(p r),(q s)] as [p, r, q, s], p, r in I
    F = ev.fock_generalized(one, two)
    ni, N = ev.ni, ev.N
    v = torch.as_tensor(np.random.default_rng(3).standard_normal((H.shape[0], 3)))
    V, L, R = _skew(ev, v)
    W = -torch.einsum('px,bxq->bpq', F + F.T, V)
    W[:, :ni] += torch.einsum('prqs,brs->bpq', t, V[:, :ni])
    HV = (W[:, L, R] - W[:, R, L]).T
    scale = H.abs().max().item()
    assert (HV - H @ v).abs().max().item() <= 1e-13 * scale

    fs = F + F.T

    def x(a, b, cc, d):
        out = -fs[a, cc] * (b == d).to(DT)
        inside = (a < ni) & (cc < ni)
        tt = t[a.clamp(max=ni - 1), cc.clamp(max=ni - 1), b, d]
        return out + torch.where(inside, tt, torch.zeros_like(tt))

    diag = x(L, R, L, R) - x(L, R, R, L) - x(R, L, L, R) + x(R, L, R, L)
    assert torch.equal(diag, H.diagonal())


@pytest.mark.parametrize("name", ["n7_cas44", "n11_cas43"])
def test_plane_products_never_need_the_t_matrix(name):
    """sum_{r,s} T[(p r),(q s)] V[r,s] from the class planes one at a time: M_k = A_k V_I, then B_k M_k^T."""
    c, ev = _evaluation(name)
    one, two = c.one_rdm, c.two_rdm
    ni, N, no = ev.ni, ev.N, ev.no
    d1, d2 = orc.full_rdms(one, two, ni, np.arange(no), np.arange(no, ni))
    # rows k of A (coefficients, [k, p, r]) and B (class planes, [k, q, s]) such that T = sum_k A_k (x) B_k
    A = torch.cat([2 * (d2.permute(0, 2, 1, 3) + d2.permute(0, 3, 1, 2)).reshape(ni, ni, ni * ni).permute(2, 0, 1),
                   2 * d2.reshape(ni, ni, ni * ni).permute(2, 0, 1), 2 * d1[None]])
    B = torch.cat([ev.K.permute(1, 0, 2, 3).reshape(ni * ni, N, N), ev.J.reshape(ni * ni, N, N), ev.h[None]])
    t = ev._t_matrix(one, two)
    V = torch.as_tensor(np.random.default_rng(5).standard_normal((N, N)))
    V = V - V.T
    direct = torch.einsum('prqs,rs->pq', t, V[:ni])
    streamed = torch.zeros(ni, N, dtype=DT)
    for k in range(A.shape[0]):
        M = A[k] @ V[:ni]                                        # [p, s]
        streamed += M @ B[k].T                                   # [p, q] += sum_s M[p,s] B_k[q,s]
    assert (streamed - direct).abs().max().item() <= 1e-12 * max(1.0, direct.abs().max().item())


# ---- the float64 reference of tests/test_gpu_hessian_configs.py, pinned ------------------------------------------------
from test_gpu_hessian_configs import hessian_reference, low_rank_factors, t_reference  # noqa: E402


@pytest.mark.parametrize("name", CASES)
def test_generalised_reference_equals_the_class_oracle_on_tril_lists(name):
    """T and H written out for an arbitrary pair list reproduce ClassEvaluation.hessian on the engine's list"""
    c, ev = _evaluation(name)
    one, two = c.one_rdm, c.two_rdm
    T = t_reference(ev.h, ev.J, ev.K, one, two, ev.no, ev.na)
    rr, cc = orc.tril_pairs(ev.N)
    H = hessian_reference(T, ev.fock_generalized(one, two), ev.ni, rr[ev.params_idx], cc[ev.params_idx])
    want = ev.hessian(one, two)
    assert (H - want).abs().max().item() <= 1e-13 * want.abs().max().item()


@pytest.mark.parametrize("name", ["n7_cas44", "n11_cas43"])
def test_generalised_reference_reproduces_the_golden_hessians(name):
    c, ev = _evaluation(name)
    one, two = c.one_rdm, c.two_rdm
    T = t_reference(ev.h, ev.J, ev.K, one, two, ev.no, ev.na)
    rr, cc = orc.tril_pairs(ev.N)
    H = hessian_reference(T, ev.fock_generalized(one, two), ev.ni, rr[ev.params_idx], cc[ev.params_idx])
    assert np.abs(H.numpy() - c.ref["H"]).max() < 1e-12


def test_generalised_reference_equals_the_dense_hessian_on_any_pair_list():
    """upper-triangle, virt-virt and occ-occ pairs in random order: oo_oracle.hessian_full (dense N^4 / N^6) indexed
    at the pairs"""
    from auto_oo_b200.synthetic import random_rdms
    N, no, na = 9, 2, 3
    nI = no + na
    M, w = low_rank_factors(N, N, seed=11)
    g = torch.einsum('P,Pab,Pcd->abcd', w, M, M)
    gen = torch.Generator().manual_seed(12)
    h = torch.randn(N, N, dtype=DT, generator=gen)
    h = h + h.T
    one, two = random_rdms(na, 2, seed=3)
    occ, act = np.arange(no), np.arange(no, nI)
    H4 = orc.hessian_full(h, g, one, two, occ, act)
    F = orc.fock_generalized(h, g, one, two, occ, act)
    J = g[:, :, :nI, :nI].permute(2, 3, 0, 1)                   # J[m,n,a,b] = g'[a,b,m,n]
    K = g[:, :nI, :nI, :].permute(2, 1, 0, 3)                   # K[n,m,a,b] = g'[a,m,n,b]
    T = t_reference(h, J, K, one, two, no, na)
    rng = np.random.default_rng(4)
    rows, cols = np.tril_indices(N, k=-1)
    flip = rng.random(len(rows)) < 0.5
    L, R = np.where(flip, cols, rows), np.where(flip, rows, cols)
    perm = rng.permutation(len(L))
    L, R = L[perm], R[perm]
    H = hessian_reference(T, F, nI, L, R)
    Lt, Rt = torch.as_tensor(L), torch.as_tensor(R)
    want = H4[Lt[:, None], Rt[:, None], Lt[None, :], Rt[None, :]]
    assert (H - want).abs().max().item() <= 1e-13 * want.abs().max().item()
