"""GPU: the matrix-free Newton step -- Davidson for the lowest orbital-Hessian eigenpair and deflated PCG for the
shifted solve (``auto_oo_b200/krylov.py``, ``csrc/krylov.cu``) -- against the dense ``NewtonStep.newton_step``.

* the kernels (subspace eigensolver, Davidson expand and restart, PCG step) against torch references;
* ``OrbitalHessian.newton_step`` against ``NewtonStep.newton_step(g, H.matrix())`` on every golden case and route, in
  both branches (shifted, and unshifted at a converged minimum), and at the two full sizes;
* the drivers with ``matrix_free=True``, the dense path left bit-identical, which kernels launch, determinism and
  the error cases."""
import numpy as np
import pytest
import torch

from auto_oo_b200 import _lib
from helpers import ALL_CASES, load_case

pytestmark = pytest.mark.gpu
F64 = torch.float64
SEED = 11
ROUTES = ["class", "class_general", "full", "from_integrals"]


def _engine():
    from auto_oo_b200.engine import HotPathEngine
    return HotPathEngine.for_tensors(2)


def _sym(k, rng, evals=None):
    if evals is None:
        A = rng.standard_normal((k, k))
        return (A + A.T) / 2
    Q, _ = np.linalg.qr(rng.standard_normal((k, k)))
    return (Q * np.asarray(evals)) @ Q.T


# ---------------------------------------------------------------------------------------------- kernels
@pytest.mark.parametrize("batch", [1, 5])
def test_subspace_eigh_matches_torch(batch):
    eng = _engine()
    rng = np.random.default_rng(3)
    for k in list(range(1, 17)) + [23, 31, 32, 33, 47, 63, 64]:
        mats = [_sym(k, rng) for _ in range(batch)]
        if k >= 6:                                                   # repeated and clustered eigenvalues
            ev = np.sort(rng.standard_normal(k))
            ev[1:4] = ev[1]
            ev[-3:] = ev[-1] + np.array([0.0, 1e-9, 2e-9])
            mats[-1] = _sym(k, rng, ev)
        S = torch.as_tensor(np.stack(mats), device="cuda")
        w = torch.full((batch, k), np.nan, dtype=F64, device="cuda")
        Y = torch.full((batch, k, k), np.nan, dtype=F64, device="cuda")
        eng.subspace_eigh(S, k, w, Y)
        ref = torch.linalg.eigvalsh(S)
        scale = ref.abs().amax(dim=1, keepdim=True).clamp_min(1e-300)
        assert ((w - ref).abs() / scale).max().item() <= 1e-13, k
        eye = torch.eye(k, dtype=F64, device="cuda")
        assert (Y.transpose(1, 2) @ Y - eye).abs().max().item() <= 1e-13, k
        assert ((S @ Y - Y * w[:, None, :]).abs() / scale[:, :, None]).max().item() <= 1e-12, k
        assert bool((w[:, 1:] >= w[:, :-1]).all())


def _basis(n, k, rng):
    Q, _ = np.linalg.qr(rng.standard_normal((n, k)))
    return Q.T.copy()


def test_davidson_expand_against_a_cgs2_reference():
    eng = _engine()
    rng = np.random.default_rng(5)
    n, kmax = 200, 8
    M = torch.as_tensor(_sym(n, rng) + np.diag(np.linspace(-1, 5, n)), device="cuda")
    D = M.diagonal().contiguous()
    for k in (2, 5, kmax):                                           # k = kmax: thick restart to [x, x_prev]
        Vt = torch.zeros(kmax, n, dtype=F64, device="cuda")
        Vt[:k] = torch.as_tensor(_basis(n, k, rng), device="cuda")
        HVt = torch.zeros_like(Vt)
        HVt[:k] = (M @ Vt[:k].T).T
        S = torch.zeros(kmax, kmax, dtype=F64, device="cuda")
        for m in range(k):
            eng.davidson_project(Vt, m + 1, HVt[m], S[m], 1, S[:, m], kmax)
        Sref = Vt[:k] @ HVt[:k].T
        assert (S[:k, :k] - Sref).abs().max().item() <= 1e-12
        w = torch.zeros(kmax, dtype=F64, device="cuda")
        Y = torch.zeros(kmax, kmax, dtype=F64, device="cuda")
        eng.subspace_eigh(S, k, w, Y)
        yprev = torch.zeros(kmax, dtype=F64, device="cuda")
        yprev[:k - 1] = torch.as_tensor(rng.standard_normal(k - 1), device="cuda")
        yprev /= yprev.norm()
        V0, yp0 = Vt[:k].clone(), yprev.clone()
        x, hx, rn = (torch.empty(n, dtype=F64, device="cuda") for _ in range(3))
        eng.davidson_expand(Vt, HVt, k, Y, w[:1], D, S, x, hx, yprev, rn[:1], 1e-8)
        y, th = Y[:k, 0], w[0]
        if k < kmax:
            xr = Vt[:k].T @ y
            hxr = HVt[:k].T @ y
            r = hxr - th * xr
            assert abs(rn[0].item() - r.norm().item()) <= 1e-13 * max(1.0, r.norm().item())
            d = D - th
            d = torch.where(d.abs() < 1e-8, torch.where(d < 0, -1e-8, 1e-8), d)
            t = r / d
            B = Vt[:k]
            for _ in range(2):
                t = t - B.T @ (B @ t)
            t = t / t.norm()
            new = Vt[k]
            assert (x - xr).abs().max().item() <= 1e-13 and (hx - hxr).abs().max().item() <= 1e-12
            assert (B @ new).abs().max().item() <= 1e-14
            assert abs(new.norm().item() - 1.0) <= 1e-14
            assert (new - t).abs().max().item() <= 1e-10
            assert torch.equal(yprev[:k], y) and yprev[k].item() == 0.0
        else:
            # restart: rows 0, 1 = [x, x_prev made orthonormal to x], their products and projected matrix, row 2 new
            assert (Vt[0] - x).abs().max().item() == 0.0 and (HVt[0] - hx).abs().max().item() == 0.0
            assert (HVt[:2] - (M @ Vt[:2].T).T).abs().max().item() <= 1e-12
            G = Vt[:3] @ Vt[:3].T
            assert (G - torch.eye(3, dtype=F64, device="cuda")).abs().max().item() <= 1e-14
            assert (S[:2, :2] - Vt[:2] @ HVt[:2].T).abs().max().item() <= 1e-12
            c = yp0[:k] - (y @ yp0[:k]) * y
            assert (Vt[1] - V0.T @ (c / c.norm())).abs().max().item() <= 1e-12
            assert yprev[0].item() == 1.0 and yprev[1:k].abs().max().item() == 0.0


@pytest.mark.parametrize("deflate", [False, True])
def test_pcg_step_against_the_written_out_update(deflate):
    eng = _engine()
    rng = np.random.default_rng(7)
    n = 300
    A = rng.standard_normal((n, n))
    M = torch.as_tensor(A @ A.T / n + np.diag(np.linspace(0.1, 3, n)), device="cuda")
    D = M.diagonal().contiguous()
    b = torch.as_tensor(rng.standard_normal(n), device="cuda")
    sigma = 0.25
    Ms = M + sigma * torch.eye(n, dtype=F64, device="cuda")
    w = aw = None
    if deflate:
        ev, U = torch.linalg.eigh(M)
        w = U[:, 0].contiguous()
        aw = (Ms @ w).contiguous()
    x, r, p = torch.empty(n, dtype=F64, device="cuda"), b.clone(), torch.empty(n, dtype=F64, device="cuda")
    state, rn = torch.zeros(2, dtype=F64, device="cuda"), torch.empty(1, dtype=F64, device="cuda")
    eng.pcg_step(None, sigma, D, x, r, p, state, rn, w=w, aw=aw, init=True)
    # reference
    pre = D + sigma
    if deflate:
        gam = (w @ b) / (w @ aw)
        xr, rr = gam * w, b - gam * aw
    else:
        xr, rr = torch.zeros_like(b), b.clone()
    zr = rr / pre
    pr = zr - ((aw @ zr) / (w @ aw)) * w if deflate else zr.clone()
    rz = rr @ zr
    for step in range(6):
        scale = max(1.0, xr.abs().max().item())
        assert (x - xr).abs().max().item() <= 1e-12 * scale, step
        assert (r - rr).abs().max().item() <= 1e-12 * max(1.0, b.abs().max().item()), step
        assert (p - pr).abs().max().item() <= 1e-11 * max(1.0, pr.abs().max().item()), step
        assert abs(rn[0].item() - rr.norm().item()) <= 1e-12 * b.norm().item(), step
        Ap = (M @ p).contiguous()
        eng.pcg_step(Ap, sigma, D, x, r, p, state, rn, w=w, aw=aw)
        q = Ms @ pr
        a = rz / (pr @ q)
        xr = xr + a * pr
        rr = rr - a * q
        zr = rr / pre
        rz_new = rr @ zr
        pr = zr + (rz_new / rz) * pr - (((aw @ zr) / (w @ aw)) * w if deflate else 0.0)
        rz = rz_new
        if deflate:
            assert abs((w @ r).item()) <= 1e-12 * b.norm().item()


# ---------------------------------------------------------------------------------------------- Newton step
def make_oo(c, **kw):
    import auto_oo_b200
    return auto_oo_b200.OO_energy(c.mol(), c.ncas, c.nelecas, oao_mo_coeff=c.oao_mo_coeff, freeze_active=c.freeze,
                                  **kw)


def _hessian_and_gradient(c, route):
    if route == "from_integrals":
        oo = make_oo(c)
        h, g = c.oracle().mo_integrals(c.kappa)
        H = oo.analytic_hessian_from_integrals(h, g, c.one_rdm, c.two_rdm)
        Gm = oo.analytic_gradient_from_integrals(h, g, c.one_rdm, c.two_rdm)
    else:
        kw = {"class": {}, "class_general": {"eri_symmetry": "off"}, "full": {"integral_path": "full"}}[route]
        oo = make_oo(c, **kw)
        Cp = torch.as_tensor(c.ref["mo_coeff_rot"])
        H = oo.analytic_hessian(c.one_rdm, c.two_rdm, mo_coeff=Cp)
        Gm = oo.analytic_gradient(c.one_rdm, c.two_rdm, mo_coeff=Cp)
    g = torch.as_tensor(oo.kappa_matrix_to_vector(Gm.detach())).to(device="cuda", dtype=F64)
    return oo, H, g


def _check_step(H, g, lambda_min=1e-6, M=None):
    from auto_oo_b200.utils.newton_raphson import NewtonStep
    M = H.matrix() if M is None else M
    ns = NewtonStep(verbose=0, lambda_min=lambda_min)
    dp_ref, lam_ref = ns.newton_step(g, M)
    info = {}
    dp, lam = H.newton_step(g, lambda_min=lambda_min, info=info)
    assert dp.device == g.device and dp.shape == g.shape
    sigma = ns.mu + ns.rho * abs(lam_ref) if lam_ref < lambda_min else 0.0
    assert abs(lam - lam_ref) <= 1e-10, (lam, lam_ref)
    assert (dp - dp_ref).abs().max().item() <= 1e-8 * max(1.0, dp_ref.abs().max().item())
    res = (M @ dp + sigma * dp + g).norm().item()
    assert res <= 1e-10 * max(g.norm().item(), 1e-300), res
    return lam_ref < lambda_min, info


@pytest.mark.parametrize("route", ROUTES)
@pytest.mark.parametrize("name", ALL_CASES)
def test_newton_step_matches_the_dense_step(name, route):
    c = load_case(name)
    oo, H, g = _hessian_and_gradient(c, route)
    _check_step(H, g)


def _indefinite_case():
    """The first golden case whose Hessian has a negative eigenvalue at its rotated orbitals."""
    for name in ALL_CASES:
        oo, H, g = _hessian_and_gradient(load_case(name), "class")
        if torch.linalg.eigvalsh(H.matrix())[0].item() < 0:
            return oo, H, g
    pytest.fail("no golden case with an indefinite Hessian")


def test_shifted_branch_is_taken():
    oo, H, g = _indefinite_case()
    shifted, info = _check_step(H, g)
    assert shifted and info["shift"] > 0


def test_unshifted_branch_at_a_converged_minimum():
    c = load_case("n7_cas44_frozen")
    oo = make_oo(c)
    oo.orbital_optimization(c.one_rdm, c.two_rdm, conv_tol=1e-12, max_iterations=60, verbose=None)
    H = oo.analytic_hessian(c.one_rdm, c.two_rdm)
    g = torch.as_tensor(oo.kappa_matrix_to_vector(oo.analytic_gradient(c.one_rdm, c.two_rdm).detach())).cuda()
    M = H.matrix()
    lam0 = torch.linalg.eigvalsh(M)[0].item()
    assert lam0 > 0, lam0                                     # a minimum
    lambda_min = min(1e-6, 0.5 * lam0)
    shifted, info = _check_step(H, g, lambda_min=lambda_min, M=M)
    assert not shifted and info["shift"] == 0.0


# ---------------------------------------------------------------------------------------------- full sizes
def _full_size(workload):
    from auto_oo_b200 import OO_energy
    from auto_oo_b200.synthetic import CONFIG_SHAPES, SyntheticMol, random_kappa, random_rdms
    dev = torch.device("cuda", 0)
    nao, nelec, ncas, nelecas = CONFIG_SHAPES[workload]
    mol = SyntheticMol(nao, nelec, seed=SEED, device=dev, rng_device="cpu")
    oo = OO_energy(mol, ncas, nelecas, oao_mo_coeff=mol.random_oao_mo_coeff, device=dev)
    mol._B = None
    one, two = (x.to(dev) for x in random_rdms(ncas, nelecas, seed=SEED))
    kappa = random_kappa(oo.n_kappa, seed=SEED, batch=2).to(dev)
    return oo, one, two, kappa


@pytest.mark.parametrize("workload", ["c6h6_ccpvdz_cas66", "synthetic_n256_cas1212"])
def test_full_size_newton_direction(workload):
    oo, one, two, kappa = _full_size(workload)
    k1 = kappa[:1]
    E0, G0, dk0, lam0 = oo.energy_gradient_newton_direction(k1, one, two)
    oo.engine.release_workspaces()
    torch.cuda.empty_cache()
    E1, G1, dk1, lam1 = oo.energy_gradient_newton_direction(k1, one, two, matrix_free=True)     # warm
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    E1, G1, dk1, lam1 = oo.energy_gradient_newton_direction(k1, one, two, matrix_free=True)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    assert torch.equal(E0, E1) and torch.equal(G0, G1)
    assert abs(lam1[0].item() - lam0[0].item()) <= 1e-10
    assert (dk1 - dk0).abs().max().item() <= 1e-8 * max(1.0, dk0.abs().max().item())
    if oo.nao == 256:
        assert peak < 256 << 20, peak


# ---------------------------------------------------------------------------------------------- drivers
@pytest.mark.parametrize("name", ["n28_cas66", "mol_h2o_sto3g_cas44"])
def test_orbital_optimization_trajectory(name):
    c = load_case(name)
    runs = []
    for mf in (False, True):
        oo = make_oo(c)
        runs.append(oo.orbital_optimization(c.one_rdm, c.two_rdm, conv_tol=-1.0, max_iterations=8, verbose=None,
                                            matrix_free=mf))
    assert len(runs[0]) == len(runs[1]) == 8
    assert np.abs(np.array(runs[0]) - np.array(runs[1])).max() <= 1e-9, runs


def test_newton_direction_batch_of_three():
    c = load_case("n28_cas66")
    oo = make_oo(c)
    k = torch.stack([c.kappa, 0.5 * c.kappa, -c.kappa]).cuda()
    E0, G0, dk0, lam0 = oo.energy_gradient_newton_direction(k, c.one_rdm, c.two_rdm)
    E1, G1, dk1, lam1 = oo.energy_gradient_newton_direction(k, c.one_rdm, c.two_rdm, matrix_free=True)
    assert torch.equal(E0, E1) and torch.equal(G0, G1)
    assert (lam1 - lam0).abs().max().item() <= 1e-10
    for b in range(3):
        assert (dk1[b] - dk0[b]).abs().max().item() <= 1e-8 * max(1.0, dk0[b].abs().max().item())


def test_dense_newton_step_is_the_eigh_formula():
    from auto_oo_b200.utils.newton_raphson import NewtonStep
    c = load_case("n28_cas66")
    oo, H, g = _hessian_and_gradient(c, "class")
    M = H.matrix()
    ns = NewtonStep(verbose=0)
    dp, lam = ns.newton_step(g, M)
    evals, evecs = torch.linalg.eigh(M)
    low = evals[0].item()
    if low < ns.lambda_min and ns.aug:
        evals = evals + (ns.mu + ns.rho * abs(low))
    assert lam == low and torch.equal(dp, -(evecs @ ((evecs.T @ g) / evals)))


def test_only_products_and_solver_kernels_launch():
    from torch.profiler import ProfilerActivity, profile
    c = load_case("n28_cas66")
    oo = make_oo(c)
    k = c.kappa[None].cuda()
    oo.energy_gradient_newton_direction(k, c.one_rdm, c.two_rdm, matrix_free=True)            # warm
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        torch.ones(1, device="cuda").add_(1)
        oo.energy_gradient_newton_direction(k, c.one_rdm, c.two_rdm, matrix_free=True)
        torch.cuda.synchronize()
    names = [e.name for e in prof.events()]
    for kern in ("subspace_eigh_kernel", "dav_project_kernel", "dav_expand_kernel", "dav_orth_kernel",
                 "pcg_partial_kernel", "pcg_update_kernel", "hvp_plane_kernel", "hess_diag_kernel"):
        assert any(kern in n for n in names), kern
    assembly = [n for n in names if "hess_" in n and "hess_diag_kernel" not in n]
    assert not assembly, sorted(set(assembly))
    assert not [n for n in names if "syev" in n.lower()]


# ---------------------------------------------------------------------------------------------- determinism, errors
def test_repeats_are_bit_identical():
    c = load_case("n43_cas34")
    oo, H, g = _hessian_and_gradient(c, "class")
    a, la = H.newton_step(g)
    b, lb = H.newton_step(g)
    assert la == lb and torch.equal(a, b)
    (l1, x1), (l2, x2) = H.lowest_eigenpair(), H.lowest_eigenpair()
    assert l1 == l2 and np.array_equal(np.asarray(x1), np.asarray(x2))


def test_errors():
    oo, H, g = _indefinite_case()
    assert H.lowest_eigenpair()[0] < 0
    with pytest.raises(ValueError):
        H.newton_step(g, aug=False)
    with pytest.raises(RuntimeError):
        H.lowest_eigenpair(max_iter=1)
    with pytest.raises(RuntimeError):
        H.solve(-g, shift=10.0, max_iter=1)
    with pytest.raises(ValueError):
        H.newton_step(g[:-1])
    with pytest.raises(ValueError):
        H.solve(torch.zeros(g.numel() + 1, dtype=F64, device="cuda"))
    # solve() on its own: (H + shift)^-1 rhs
    M = H.matrix()
    x = H.solve(-g, shift=10.0)
    assert (M @ x + 10.0 * x + g).norm().item() <= 1e-10 * g.norm().item()


def test_abi_rejects_bad_arguments_before_any_launch():
    lib = _lib.load()
    st = torch.cuda.current_stream().cuda_stream
    n, kmax = 100, 8
    S = torch.zeros(65, 65, dtype=F64, device="cuda")
    w = torch.zeros(65, dtype=F64, device="cuda")
    Y = torch.zeros(65, 65, dtype=F64, device="cuda")
    Vt = torch.zeros(kmax, n, dtype=F64, device="cuda")
    vec = [torch.zeros(n, dtype=F64, device="cuda") for _ in range(6)]
    nb = lib.oo_workspace_bytes(_lib.OO_WS_KRYLOV, n, 1, kmax, 1)
    assert nb > 0 and lib.oo_workspace_bytes(_lib.OO_WS_KRYLOV, n, 1, 65, 1) == 0
    ws = torch.zeros(nb, dtype=torch.uint8, device="cuda")
    p = lambda t: t.data_ptr()
    n0 = lib.oo_launch_count()
    assert lib.oo_subspace_eigh_f64(p(S), 65, 65, 0, 1, p(w), 0, p(Y), 65, 0, st) == -1
    assert lib.oo_subspace_eigh_f64(None, 4, 65, 0, 1, p(w), 0, p(Y), 65, 0, st) == -1
    assert lib.oo_subspace_eigh_f64(p(S), 4, 3, 0, 1, p(w), 0, p(Y), 65, 0, st) == -1
    assert lib.oo_davidson_project_f64(p(Vt), n, n, 65, p(vec[0]), p(w), 1, None, 0, st) == -1
    assert lib.oo_davidson_project_f64(p(Vt), n - 1, n, 2, p(vec[0]), p(w), 1, None, 0, st) == -1
    args = [p(Vt), p(Vt), n, n, 2, kmax, p(Y), 65, p(w), p(vec[0]), 1e-8, p(S), 65, p(vec[1]), p(vec[2]),
            p(vec[3]), p(w), p(ws), nb, st]
    for i, bad in [(0, None), (6, None), (3, n - 1), (5, 65), (4, kmax + 1)]:
        a = list(args)
        a[i] = bad
        assert lib.oo_davidson_expand_f64(*a) == -1, i
    a = list(args)
    a[18] = nb - 1
    assert lib.oo_davidson_expand_f64(*a) == -3
    pcg = [n, p(vec[0]), 0.0, p(vec[1]), None, None, p(vec[2]), p(vec[3]), p(vec[4]), p(w), p(w[1:]), 0, p(ws), nb, st]
    a = list(pcg)
    a[1] = None
    assert lib.oo_pcg_step_f64(*a) == -1
    a = list(pcg)
    a[4] = p(vec[5])                                                      # w without aw
    assert lib.oo_pcg_step_f64(*a) == -1
    a = list(pcg)
    a[13] = nb - 1
    assert lib.oo_pcg_step_f64(*a) == -3
    assert lib.oo_launch_count() == n0
