"""CPU: pin the oracle (oracle/oo_oracle.py) against (1) the reference's own known-answer
tests and (2) outputs of the verbatim reference stored in tests/golden (made by
oracle/make_golden.py)."""
import os

import numpy as np
import pytest
import torch

from oracle import oo_oracle as orc
from helpers import ALL_CASES, SMALL_CASES, GOLDEN, TOL_E, TOL_GH, load_case


def test_vector_to_skew_symmetric_known_answer():
    # reference test/test_oo_energy.py:188-213
    v = torch.arange(1.0, 7.0, dtype=torch.float64)
    K = orc.unpack_skew(v)
    expect = torch.tensor([[0, -1, -2, -4], [1, 0, -3, -5], [2, 3, 0, -6], [4, 5, 6, 0]], dtype=torch.float64)
    assert torch.equal(K, expect)
    assert torch.equal(orc.pack_skew(K), v)


@pytest.mark.parametrize("occ,act,virt,freeze,expect", [
    # reference test/test_oo_energy.py:216-231
    ([0, 1], [2, 3], [4, 5], False, [1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13]),
    ([0, 1], [2, 3], [4, 5], True, [1, 2, 3, 4, 6, 7, 8, 9, 10, 11, 12, 13]),
])
def test_non_redundant_indices_known_answer(occ, act, virt, freeze, expect):
    assert list(orc.non_redundant_indices(occ, act, virt, freeze)) == expect


def test_non_redundant_counts():
    for (no, na, nv) in [(0, 3, 5), (3, 4, 0), (2, 2, 2), (6, 4, 24)]:
        occ, act, virt = np.arange(no), no + np.arange(na), no + na + np.arange(nv)
        for freeze in (False, True):
            idx = orc.non_redundant_indices(occ, act, virt, freeze)
            assert len(idx) == no * na + na * nv + no * nv + (0 if freeze else na * (na - 1) // 2)


@pytest.mark.parametrize("name", ALL_CASES)
def test_oracle_matches_reference_outputs(name):
    c = load_case(name)
    p = c.oracle()
    r = c.ref
    assert np.array_equal(p.params_idx, r["params_idx"])
    U = orc.rotation_from_kappa(c.kappa, p.params_idx, c.nao)
    assert np.abs(U.numpy() - r["U"]).max() < 1e-14
    assert np.abs(p.rotated_mo(c.kappa).numpy() - r["mo_coeff_rot"]).max() < 1e-13
    c0, c1, c2 = p.active_integrals(c.kappa)
    assert abs(float(c0) - float(r["c0"])) < TOL_E
    assert np.abs(c1.numpy() - r["c1"]).max() < 1e-11
    assert np.abs(c2.numpy() - r["c2"]).max() < 1e-11
    assert abs(p.energy(c.one_rdm, c.two_rdm, c.kappa).item() - float(r["E"])) < TOL_E
    assert abs(p.energy(c.one_rdm, c.two_rdm).item() - float(r["E0"])) < TOL_E
    assert np.abs(p.gradient(c.one_rdm, c.two_rdm, c.kappa).numpy() - r["G"]).max() < TOL_GH
    assert np.abs(p.gradient(c.one_rdm, c.two_rdm).numpy() - r["G0"]).max() < TOL_GH
    # the dense N^6 form is the reference's algorithm; keep it to the sizes that finish in seconds
    H = p.hessian(c.one_rdm, c.two_rdm, c.kappa, ispace=c.nao > 13)
    assert np.abs(H.numpy() - r["H"]).max() < TOL_GH


@pytest.mark.parametrize("name", SMALL_CASES)
def test_ispace_hessian_equals_dense_form(name):
    c = load_case(name)
    p = c.oracle()
    Hd = p.hessian(c.one_rdm, c.two_rdm, c.kappa, ispace=False)
    Hi = p.hessian(c.one_rdm, c.two_rdm, c.kappa, ispace=True)
    assert (Hd - Hi).abs().max().item() < 1e-11
    assert (Hd - Hd.T).abs().max().item() < 1e-10
    assert np.abs(Hi.numpy() - c.ref["H"]).max() < TOL_GH


@pytest.mark.parametrize("name", SMALL_CASES)
def test_transforms_match_reference(name):
    c = load_case(name)
    Cp = torch.as_tensor(c.ref["mo_coeff_rot"])
    assert np.abs(orc.transform_1e(c.int1e_ao, Cp).numpy() - c.ref["int1e_mo"]).max() < 1e-12
    assert np.abs(orc.transform_2e(c.int2e_ao, Cp).numpy() - c.ref["int2e_mo"]).max() < 1e-12


def test_general_4index_transform():
    d = np.load(os.path.join(GOLDEN, "general_4index_n6.npz"))
    out = orc.transform_4index(d["M"], d["C0"], d["C1"], d["C2"], d["C3"])
    assert np.abs(out.numpy() - d["out"]).max() < 1e-12
    explicit = np.einsum('pi,qj,rk,sl,pqrs->ijkl', d["C0"], d["C1"], d["C2"], d["C3"], d["M"])
    assert np.abs(out.numpy() - explicit).max() < 1e-11


@pytest.mark.parametrize("name", ["n7_cas44", "n13_cas22", "mol_ch2nh_sto3g_cas22", "mol_h2o_sto3g_cas44"])
def test_analytic_derivatives_equal_autograd(name):
    """The reference's own strategy (test/test_oo_energy.py:415-971): analytic G/H at kappa=0
    against autograd of energy_from_kappa -- proves the fixtures obey the symmetry preconditions."""
    c = load_case(name)
    p = c.oracle()

    def energy(k):
        C = p.mo_coeff @ torch.linalg.matrix_exp(-orc.kappa_to_skew_diff(k, p.params_idx, c.nao))
        h, g = orc.transform_1e(p.h_ao, C), orc.transform_2e(p.g_ao, C)
        c0, c1, c2 = orc.hamiltonian_coefficients(p.nuc, h, g, p.occ_idx, p.act_idx)
        return orc.energy_from_coefficients(c0, c1, c2, c.one_rdm, c.two_rdm)

    k0 = torch.zeros(p.n_kappa, dtype=torch.float64)
    g_auto = torch.autograd.functional.jacobian(energy, k0)
    h_auto = torch.autograd.functional.hessian(energy, k0)
    assert (g_auto - p.gradient(c.one_rdm, c.two_rdm)).abs().max().item() < 1e-10
    assert (h_auto - p.hessian(c.one_rdm, c.two_rdm)).abs().max().item() < 1e-9


def test_odd_core_electrons_raises():
    with pytest.raises(ValueError):
        orc.active_space_idx(7, 9, 4, 4)


@pytest.mark.parametrize("no,na", [(0, 3), (1, 2), (3, 4), (6, 4), (4, 6), (10, 3), (18, 6)])
def test_hessian_sparse_row_bound(no, na):
    """The CUDA Hessian stores the non-dense part of At in ELL rows of width 2 na^2 + 2 (no+na) + 8
    (csrc/hessian_terms.cuh, ell_width).  Count the structural non-zeros of the reference's full-space
    2-RDM (full_rdms, oo_energy.py:342-379) outside the act-act block and check the bound."""
    gen = torch.Generator().manual_seed(0)
    one = torch.rand(na, na, dtype=torch.float64, generator=gen) + 0.5          # no accidental zeros
    two = torch.rand(na, na, na, na, dtype=torch.float64, generator=gen) + 0.5
    ni = no + na
    occ, act = np.arange(no), no + np.arange(na)
    d1, d2 = orc.full_rdms(one, two, ni, occ, act)
    a1 = (d2.permute(0, 2, 1, 3) + d2.permute(0, 3, 1, 2)) != 0     # [(p r),(m n)]
    a2 = d2 != 0                                                    # [(p r),(m n)] = G_prmn
    worst = 0
    for p in range(ni):
        for r in range(ni):
            nnz = int(a1[p, r].sum()) + int(a2[p, r].sum()) + int(d1[p, r] != 0)
            if p >= no and r >= no:                                  # dense block handled by the GEMM
                nnz -= int(a1[p, r][no:, no:].sum()) + int(a2[p, r][no:, no:].sum()) + int(d1[p, r] != 0)
            worst = max(worst, nnz)
    assert worst <= 2 * na * na + 2 * ni + 8, worst


@pytest.mark.parametrize("name", ALL_CASES)
def test_class_oracle_matches_reference_outputs(name):
    """oracle/class_oracle.py (the form that scales to N = 256) against the verbatim-reference fixtures."""
    from oracle.class_oracle import ClassProblem
    c = load_case(name)
    p = ClassProblem(c.int1e_ao, c.int2e_ao, c.oao_coeff, c.oao_mo_coeff, c.nuc, c.nelec, c.ncas, c.nelecas,
                     c.freeze)
    r = c.ref
    ev = p.at(c.kappa)
    c0, c1, c2 = ev.hamiltonian()
    assert abs(float(c0) - float(r["c0"])) < TOL_E
    assert np.abs(c1.numpy() - r["c1"]).max() < 1e-11 and np.abs(c2.numpy() - r["c2"]).max() < 1e-11
    assert abs(ev.energy(c.one_rdm, c.two_rdm).item() - float(r["E"])) < 1e-12 * max(1.0, abs(float(r["E"])))
    assert np.abs(ev.gradient(c.one_rdm, c.two_rdm).numpy() - r["G"]).max() < 1e-12
    assert np.abs(ev.hessian(c.one_rdm, c.two_rdm).numpy() - r["H"]).max() < 1e-12


def test_full_size_fixtures_are_pinned():
    """n114: verbatim reference, with both oracles' differences at that size recorded by the generator;
    n256: the class oracle (oracle/make_golden_large.py)."""
    d = np.load(os.path.join(GOLDEN, "n114_cas66.npz"))
    assert str(d["source"]) == "verbatim reference"
    assert d["class_oracle_vs_reference"].max() < 1e-12 and d["oo_oracle_vs_reference"].max() < 1e-12
    assert d["G"].shape == (2283,) and d["H_diag"].shape == (2283,) and float(d["H_asym"]) < 1e-10
    d = np.load(os.path.join(GOLDEN, "n256_cas1212.npz"))
    assert d["G"].shape == (9778,) and d["H_times_probes"].shape == (8, 9778) and float(d["H_asym"]) < 1e-10
