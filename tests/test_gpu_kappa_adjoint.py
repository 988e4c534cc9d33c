"""GPU: the device adjoint of kappa -> expm(-K) (``oo_kappa_rotation_vjp_f64``) and what it makes differentiable:
``energy_from_kappa``, ``kappa_to_mo_coeff`` and ``get_transformed_mo`` in kappa (the last also in ``mo_coeff``).

* The C ABI on both routes -- the single cooperative launch (8 <= ld <= 256, panels staged once or, for the dual
  products, twice) and the multi-launch chain (ld < 8, ld > 256) -- against ``scipy.linalg.expm_frechet``, with host-
  and device-chosen squaring counts, outputs between sentinel guards and a NaN-filled padding of Ubar.
* The gradient of ``energy_from_kappa`` against torch autograd of the oracle energy (``tests/test_kappa_adjoint_cpu.py``
  pins the float64 reference) on both integral paths, against the analytic gradient at kappa = 0, and against a
  4-point central difference at N = 114 and 256.
* Second derivatives in kappa raise; those in the RDMs keep working."""
import re

import numpy as np
import pytest
import torch

from auto_oo_b200 import _lib
from helpers import load_case
from test_kappa_adjoint_cpu import autograd_energy_gradient, rotation_vjp_reference, skew

pytestmark = pytest.mark.gpu
F64 = torch.float64
SENTINEL = float.fromhex("-0x1.deadbeef00000p+700")
GUARD = 64
DEV = torch.device("cuda", 0)


def _p(t):
    return 0 if t is None else t.data_ptr()


def host_squarings(kappas, pl, pr, n):
    norm = max(np.abs(skew(k, pl, pr, n)).sum(axis=0).max() for k in kappas)
    return 0 if norm <= 0.95 else int(np.ceil(np.log2(norm / 0.95)))


def abi_case(N, batch, seed):
    """kappa (batch, nk) over all tril pairs with ||K_b||_1 = 0.5, 3, 9 (batch 1: 0.5), Ubar (batch, ld, ld) with a
    NaN padding that must not be read."""
    ld = N + (N & 1)
    pl, pr = np.tril_indices(N, k=-1)
    rng = np.random.default_rng(seed)
    norms = [0.5, 3.0, 9.0][:batch]
    kappas = []
    for nb in norms:
        k = rng.standard_normal(len(pl))
        kappas.append(k * nb / np.abs(skew(k, pl, pr, N)).sum(axis=0).max())
    Ubar = np.full((batch, ld, ld), np.nan)
    Ubar[:, :N, :N] = rng.standard_normal((batch, N, N))
    return ld, pl.astype(np.int32), pr.astype(np.int32), np.array(kappas), Ubar


def call_vjp(lib, N, ld, pl, pr, kappa, Ubar, squarings, ws_bytes=None):
    batch, nk = kappa.shape
    nbytes = lib.oo_workspace_bytes(_lib.OO_WS_ROTATION_VJP, N, ld, 0, batch)
    ws = torch.full((nbytes // 8,), float("nan"), dtype=F64, device=DEV)
    buf = torch.full((batch * nk + 2 * GUARD,), SENTINEL, dtype=F64, device=DEV)
    buf[GUARD:GUARD + batch * nk] = float("nan")
    k, U = torch.as_tensor(kappa, device=DEV), torch.as_tensor(Ubar, device=DEV)
    tl, tr = torch.as_tensor(pl, device=DEV), torch.as_tensor(pr, device=DEV)
    rc = lib.oo_kappa_rotation_vjp_f64(_p(k), _p(tl), _p(tr), nk, N, ld, batch, squarings, _p(U),
                                       _p(buf) + 8 * GUARD, _p(ws), nbytes if ws_bytes is None else ws_bytes, 0)
    torch.cuda.synchronize()
    return rc, buf


ABI_N = [6, 7, 13, 34, 64, 65, 114, 128, 129, 256, 257]


@pytest.mark.parametrize("N", ABI_N)
@pytest.mark.parametrize("batch", [1, 3])
def test_abi_matches_expm_frechet(N, batch):
    lib = _lib.load()
    ld, pl, pr, kappa, Ubar = abi_case(N, batch, seed=N * 10 + batch)
    nk = len(pl)
    ref = np.stack([rotation_vjp_reference(kappa[b], pl, pr, N, Ubar[b, :N, :N]) for b in range(batch)])
    s_host = host_squarings(kappa, pl, pr, N)
    assert (s_host == 0) == (batch == 1) and (batch == 1 or s_host >= 3)
    modes = [s_host, s_host + 2] + ([-1] if 8 <= ld <= 256 else [])
    for s in modes:
        rc, buf = call_vjp(lib, N, ld, pl, pr, kappa, Ubar, s)
        assert rc == 0, (N, batch, s, rc)
        out = buf[GUARD:GUARD + batch * nk].reshape(batch, nk).cpu().numpy()
        assert np.isfinite(out).all(), f"N={N} s={s}: unwritten kappa_bar"
        assert (buf[:GUARD] == SENTINEL).all() and (buf[-GUARD:] == SENTINEL).all(), "guard zone overwritten"
        err = np.abs(out - ref).max() / np.abs(ref).max()
        assert err <= 1e-11, f"N={N} batch={batch} s={s}: rel err {err:.2e}"
        rc2, buf2 = call_vjp(lib, N, ld, pl, pr, kappa, Ubar, s)
        assert rc2 == 0 and torch.equal(buf, buf2), "repeats must be bit-identical"
    if not 8 <= ld <= 256:
        assert call_vjp(lib, N, ld, pl, pr, kappa, Ubar, -1)[0] == -2     # needs the host's squaring count


def test_abi_rejects_bad_arguments_before_any_launch():
    lib = _lib.load()
    N, batch = 34, 1
    ld, pl, pr, kappa, Ubar = abi_case(N, batch, seed=5)
    nk = len(pl)
    nbytes = lib.oo_workspace_bytes(_lib.OO_WS_ROTATION_VJP, N, ld, 0, batch)
    assert nbytes >= 14 * ld * ld * 8
    k, U = torch.as_tensor(kappa, device=DEV), torch.as_tensor(Ubar, device=DEV)
    tl, tr = torch.as_tensor(pl, device=DEV), torch.as_tensor(pr, device=DEV)
    out = torch.empty(nk, dtype=F64, device=DEV)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=DEV)
    before = lib.oo_launch_count()
    args = [_p(k), _p(tl), _p(tr), nk, N, ld, batch, -1, _p(U), _p(out), _p(ws), nbytes, 0]
    for i in (0, 1, 2, 8, 9, 10):
        bad = list(args)
        bad[i] = 0
        assert lib.oo_kappa_rotation_vjp_f64(*bad) == -1, i
    bad = list(args)
    bad[5] = 35                                                   # odd ld
    assert lib.oo_kappa_rotation_vjp_f64(*bad) == -1
    bad = list(args)
    bad[11] = nbytes - 8
    assert lib.oo_kappa_rotation_vjp_f64(*bad) == -3
    assert lib.oo_launch_count() == before


def _kernel_names(prof):
    return {e.name for e in prof.events()}


def test_both_routes_launch_the_adjoint_kernels():
    from torch.profiler import ProfilerActivity, profile
    lib = _lib.load()
    launched = {}
    for N in (6, 34, 256, 257):
        ld, pl, pr, kappa, Ubar = abi_case(N, 1, seed=N)
        s = host_squarings(kappa, pl, pr, N)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            assert call_vjp(lib, N, ld, pl, pr, kappa, Ubar, s if N in (6, 257) else -1)[0] == 0
        launched[N] = _kernel_names(prof)
    for N in (34, 256):
        assert any("expm_frechet_chain_kernel" in n for n in launched[N]), N
        assert not any("dgemm_panel_kernel" in n or "dgemm_small_kernel" in n for n in launched[N]), N
    for N in (6, 257):
        assert any("skew_gather_kernel" in n for n in launched[N]), N
        assert not any("expm_frechet_chain_kernel" in n for n in launched[N]), N


# ---------------------------------------------------------------------------------------------------- Python face
def make_oo(name, path="class"):
    from auto_oo_b200 import OO_energy
    c = load_case(name)
    return c, OO_energy(c.mol(), c.ncas, c.nelecas, oao_mo_coeff=c.oao_mo_coeff, freeze_active=c.freeze,
                        integral_path=path)


API_CASES = ["n7_cas44", "n13_cas22", "n8_nocore", "n13_bigkappa", "mol_h2o_sto3g_cas44"]


@pytest.mark.parametrize("path", ["class", "full"])
@pytest.mark.parametrize("name", API_CASES)
def test_energy_gradient_matches_oracle_autograd(name, path):
    c, oo = make_oo(name, path)
    kappa = 3.0 * c.kappa
    ref = autograd_energy_gradient(c.oracle(), c.one_rdm, c.two_rdm, kappa)
    k = kappa.clone().requires_grad_(True)
    g, = torch.autograd.grad(oo.energy_from_kappa(k, c.one_rdm, c.two_rdm), k)
    assert g.device == k.device and g.dtype == F64
    assert np.abs(g.numpy() - ref).max() <= 1e-10 * max(1.0, np.abs(ref).max())
    # kappa = 0: the analytic gradient
    k0 = torch.zeros_like(kappa, requires_grad=True)
    g0, = torch.autograd.grad(oo.energy_from_kappa(k0, c.one_rdm, c.two_rdm), k0)
    ga = oo.kappa_matrix_to_vector(oo.analytic_gradient(c.one_rdm, c.two_rdm))
    assert (g0 - ga).abs().max().item() <= 1e-13 * max(1.0, ga.abs().max().item())


def test_joint_gradients_devices_and_hold():
    c, oo = make_oo("n7_cas44")
    kappa = 3.0 * c.kappa
    k = kappa.clone().requires_grad_(True)
    one, two = c.one_rdm.clone().requires_grad_(True), c.two_rdm.clone().requires_grad_(True)
    gk, g1, g2 = torch.autograd.grad(oo.energy_from_kappa(k, one, two), (k, one, two))
    assert torch.equal(gk, torch.autograd.grad(oo.energy_from_kappa(k, c.one_rdm, c.two_rdm), k)[0])
    r1, r2 = torch.autograd.grad(oo.energy_from_kappa(kappa, one, two), (one, two))
    assert torch.equal(g1, r1) and torch.equal(g2, r2)
    # a CUDA kappa gets a CUDA gradient, equal to the CPU one
    kc = kappa.to(DEV).requires_grad_(True)
    gc, = torch.autograd.grad(oo.energy_from_kappa(kc, c.one_rdm, c.two_rdm), kc)
    assert gc.device == kc.device and (gc.cpu() - gk).abs().max().item() <= 1e-13
    # forward A, forward B, backward A: A's integrals are held
    ka = kappa.clone().requires_grad_(True)
    kb = (-2.0 * kappa).requires_grad_(True)
    Ea = oo.energy_from_kappa(ka, c.one_rdm, c.two_rdm)
    Eb = oo.energy_from_kappa(kb, c.one_rdm, c.two_rdm)
    ga, = torch.autograd.grad(Ea, ka)
    assert torch.equal(ga, gk)
    gb, = torch.autograd.grad(Eb, kb)
    ref_b = autograd_energy_gradient(c.oracle(), c.one_rdm, c.two_rdm, -2.0 * kappa)
    assert np.abs(gb.numpy() - ref_b).max() <= 1e-10 * max(1.0, np.abs(ref_b).max())


def test_rotation_vjps_match_torch_autograd():
    from oracle import oo_oracle as orc
    c, oo = make_oo("n13_cas22")
    kappa = 3.0 * c.kappa
    n = c.nao
    W = torch.randn(n, n, dtype=F64, generator=torch.Generator().manual_seed(3))
    M = torch.randn(n, n, dtype=F64, generator=torch.Generator().manual_seed(4))

    def ref_grads(fn):
        k = kappa.clone().requires_grad_(True)
        m = M.clone().requires_grad_(True)
        (fn(m, torch.linalg.matrix_exp(-orc.kappa_to_skew_diff(k, oo.params_idx, n))) * W).sum().backward()
        return k.grad, m.grad

    k = kappa.clone().requires_grad_(True)
    (oo.kappa_to_mo_coeff(k) * W).sum().backward()
    rk, _ = ref_grads(lambda m, U: U)
    assert (k.grad - rk).abs().max().item() <= 1e-11 * rk.abs().max().item()
    k = kappa.clone().requires_grad_(True)
    m = M.clone().requires_grad_(True)
    (oo.get_transformed_mo(m, k) * W).sum().backward()
    rk, rm = ref_grads(lambda m, U: m @ U)
    assert (k.grad - rk).abs().max().item() <= 1e-11 * rk.abs().max().item()
    assert (m.grad - rm).abs().max().item() <= 1e-12 * rm.abs().max().item()
    assert isinstance(oo.get_transformed_mo(M.numpy(), kappa), np.ndarray)


def test_oo_pqc_jacobian_in_theta_and_kappa():
    import auto_oo_b200
    from auto_oo_b200.synthetic import CIVectorCircuit
    from oracle import oo_oracle as orc
    c = load_case("n7_cas44")
    circ = CIVectorCircuit(c.ncas, c.nelecas, n_theta=2, seed=3)
    oo = auto_oo_b200.OO_pqc(circ, c.mol(), c.ncas, c.nelecas, oao_mo_coeff=c.oao_mo_coeff, freeze_active=c.freeze)
    p = c.oracle()
    theta = torch.tensor([0.8324, 0.2490], dtype=F64)

    def ref_energy(th, k):
        one, two = circ.get_rdms(th)
        C = p.mo_coeff @ torch.linalg.matrix_exp(-orc.kappa_to_skew_diff(k, p.params_idx, c.nao))
        hh, gg = orc.transform_1e(p.h_ao, C), orc.transform_2e(p.g_ao, C)
        c0, c1, c2 = orc.hamiltonian_coefficients(p.nuc, hh, gg, p.occ_idx, p.act_idx)
        return orc.energy_from_coefficients(c0, c1, c2, one, two)

    jac = torch.autograd.functional.jacobian
    kappa = 3.0 * c.kappa
    jt, jk = jac(oo.energy_from_parameters, (theta, kappa))
    rt, rk = jac(ref_energy, (theta, kappa))
    assert (jt - rt).abs().max().item() <= 1e-10 and (jk - rk).abs().max().item() <= 1e-10
    jt0, jk0 = jac(oo.energy_from_parameters, (theta, torch.zeros_like(kappa)))
    assert (torch.cat((jt0, jk0)) - oo.full_gradient(theta)).abs().max().item() <= 1e-11


def test_second_order_in_kappa_raises_and_in_the_rdms_works():
    c, oo = make_oo("n7_cas44")
    kappa = 3.0 * c.kappa
    with pytest.raises(RuntimeError, match="analytic_hessian"):
        torch.autograd.functional.hessian(lambda k: oo.energy_from_kappa(k, c.one_rdm, c.two_rdm), kappa)
    k = kappa.clone().requires_grad_(True)
    from auto_oo_b200.synthetic import CIVectorCircuit
    circ = CIVectorCircuit(c.ncas, c.nelecas, n_theta=2, seed=3)
    theta = torch.tensor([0.8324, 0.2490], dtype=F64)
    h_k = torch.autograd.functional.hessian(lambda th: oo.energy_from_kappa(k, *circ.get_rdms(th)), theta)
    h_0 = torch.autograd.functional.hessian(lambda th: oo.energy_from_kappa(kappa, *circ.get_rdms(th)), theta)
    assert torch.isfinite(h_0).all() and h_0.abs().max().item() > 0
    assert (h_k - h_0).abs().max().item() <= 1e-12


def test_profiler_forward_unchanged_backward_without_transform():
    from torch.profiler import ProfilerActivity, profile
    c, oo = make_oo("n13_cas22")
    kappa = 3.0 * c.kappa

    def kernels(fn):
        oo.engine._icache.clear()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        return [e.name for e in prof.events() if str(e.device_type).endswith("CUDA")
                and not re.search(r"Memcpy|Memset", e.name)]

    kernels(lambda: oo.energy_from_kappa(kappa, c.one_rdm, c.two_rdm))      # first use: one-time set-up launches
    plain = kernels(lambda: oo.energy_from_kappa(kappa, c.one_rdm, c.two_rdm))
    k = kappa.clone().requires_grad_(True)
    holder = {}
    graded = kernels(lambda: holder.setdefault("E", oo.energy_from_kappa(k, c.one_rdm, c.two_rdm)))
    assert plain == graded and len(plain) > 0
    back = kernels(lambda: holder["E"].backward())
    assert not any(re.search(r"dgemm_tn", n) for n in back), back
    assert any("expm_frechet_chain_kernel" in n for n in back)


# ---------------------------------------------------------------------------------------------------- full size
@pytest.mark.parametrize("workload", ["c6h6_ccpvdz_cas66", "synthetic_n256_cas1212"])
def test_full_size_gradient_matches_central_difference(workload):
    from auto_oo_b200 import OO_energy
    from auto_oo_b200.synthetic import CONFIG_SHAPES, SyntheticMol, random_kappa, random_rdms
    nao, nelec, ncas, nelecas = CONFIG_SHAPES[workload]
    mol = SyntheticMol(nao, nelec, seed=11, device=DEV, rng_device="cpu")
    oo = OO_energy(mol, ncas, nelecas, oao_mo_coeff=mol.random_oao_mo_coeff, device=DEV)
    one, two = (t.to(DEV) for t in random_rdms(ncas, nelecas, seed=11))
    kappa = random_kappa(oo.n_kappa, seed=11, scale=0.05).to(DEV)
    d = random_kappa(oo.n_kappa, seed=12, scale=1.0).to(DEV)
    d /= d.norm()
    k = kappa.clone().requires_grad_(True)
    g, = torch.autograd.grad(oo.energy_from_kappa(k, one, two), k)
    h = 1e-3
    E = oo.energies_from_kappas(torch.stack([kappa + t * h * d for t in (2, 1, -1, -2)]), one, two)
    fd = float((-E[0] + 8 * E[1] - 8 * E[2] + E[3]) / (12 * h))
    an = float(g @ d)
    assert abs(an - fd) <= 1e-7 * max(abs(fd), 1.0), (an, fd)
