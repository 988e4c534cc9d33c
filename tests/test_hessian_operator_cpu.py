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
