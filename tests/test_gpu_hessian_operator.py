"""GPU: the matrix-free orbital Hessian -- ``OrbitalHessian.matvec`` (H v) and ``OrbitalHessian.diagonal`` -- and
their C ABI (``oo_class_hessian_vector_f64``, ``oo_class_hessian_diagonal_f64``, ``oo_hessian_vector_f64``,
``oo_hessian_diagonal_f64``).

* at the two full sizes against the reference digests of ``tests/golden/n114_cas66.npz`` (verbatim reference) and
  ``n256_cas1212.npz`` (class oracle): the products with the eight probe vectors and the diagonal, both integral
  routes, and the device memory a block of 8 products takes at N = 256;
* on every golden case against the formed matrix (``matrix()``), on the class path (symmetric and general
  integrals), the full path and ``analytic_hessian_from_integrals``, for numpy / CPU torch / CUDA torch inputs;
* bit-identical repeats, CUDA-graph capture, lifetime across interleaved evaluations, argument checks, which
  kernels launch, and a conjugate-gradient Newton solve that only uses ``matvec`` and ``diagonal``."""
import os

import numpy as np
import pytest
import torch

from auto_oo_b200 import _lib
from helpers import ALL_CASES, GOLDEN, TOL_GH, load_case

pytestmark = pytest.mark.gpu
F64 = torch.float64
SEED = 11                      # oracle/make_golden_large.py draws its inputs from the same seed
NV = [1, 2, 7, 33]             # 33 > 8 vectors per pass: processed in blocks, the last one partial


def make_oo(c, **kw):
    import auto_oo_b200
    return auto_oo_b200.OO_energy(c.mol(), c.ncas, c.nelecas, oao_mo_coeff=c.oao_mo_coeff, freeze_active=c.freeze,
                                  **kw)


def _probes(nk, nv, seed=0):
    return np.random.default_rng(seed).uniform(-1.0, 1.0, (nk, nv))


# ---------------------------------------------------------------------------------------------- full sizes
@pytest.mark.parametrize("workload,golden", [("c6h6_ccpvdz_cas66", "n114_cas66"),
                                             ("synthetic_n256_cas1212", "n256_cas1212")])
def test_full_size_products_and_diagonal_match_the_reference_digest(workload, golden):
    from auto_oo_b200 import OO_energy
    from auto_oo_b200.synthetic import CONFIG_SHAPES, SyntheticMol, random_kappa, random_rdms
    dev = torch.device("cuda", 0)
    nao, nelec, ncas, nelecas = CONFIG_SHAPES[workload]
    mol = SyntheticMol(nao, nelec, seed=SEED, device=dev, rng_device="cpu")
    oo = OO_energy(mol, ncas, nelecas, oao_mo_coeff=mol.random_oao_mo_coeff, device=dev)
    mol._B = None
    eng = oo.engine
    one, two = (x.to(dev) for x in random_rdms(ncas, nelecas, seed=SEED))
    kappa = random_kappa(oo.n_kappa, seed=SEED, batch=2).to(dev)
    d = np.load(os.path.join(GOLDEN, golden + ".npz"))
    assert np.array_equal(kappa[0].cpu().numpy(), d["kappa"])
    U = eng.rotation(kappa[:1])
    Cp = eng.from_padded(eng.mo_coeff(eng.to_padded(oo.oao_mo_coeff, 2), U), 2)[0]
    probes = torch.as_tensor(d["H_probes"], device=dev)                      # (8, nk)
    for path in ("class", "full"):
        oo.integral_path = path
        H = oo.analytic_hessian(one, two, mo_coeff=Cp)
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        HV = H.matvec(probes.T.contiguous())
        torch.cuda.synchronize()
        peak = torch.cuda.max_memory_allocated() - base
        assert np.abs(HV.T.cpu().numpy() - d["H_times_probes"]).max() < TOL_GH, path
        assert np.abs(H.diagonal().cpu().numpy() - d["H_diag"]).max() < TOL_GH, path
        if path == "class" and nao == 256:
            # H alone would be 765 MB, the T-matrix 1.0 GB (the full route gathers a 2 GB class layout first)
            assert peak < 256 << 20, peak
        del H, HV
        eng.release_workspaces()
        torch.cuda.empty_cache()


# ---------------------------------------------------------------------------------------------- small cases
ROUTES = ["class", "class_general", "full", "from_integrals"]


def _hessian(c, route):
    if route == "from_integrals":
        oo = make_oo(c)
        h, g = c.oracle().mo_integrals(c.kappa)
        return oo, oo.analytic_hessian_from_integrals(h, g, c.one_rdm, c.two_rdm)
    kw = {"class": {}, "class_general": {"eri_symmetry": "off"}, "full": {"integral_path": "full"}}[route]
    oo = make_oo(c, **kw)
    Cp = torch.as_tensor(c.ref["mo_coeff_rot"])
    return oo, oo.analytic_hessian(c.one_rdm, c.two_rdm, mo_coeff=Cp)


@pytest.mark.parametrize("route", ROUTES)
@pytest.mark.parametrize("name", ALL_CASES)
def test_products_and_diagonal_equal_the_formed_matrix(name, route):
    c = load_case(name)
    oo, H = _hessian(c, route)
    M = H.matrix()
    nk = M.shape[0]
    scale = M.abs().max().item()
    for nv in NV:
        V = _probes(nk, nv, seed=nv)
        ref = (M @ torch.as_tensor(V, device=M.device)).cpu().numpy()
        for kind in ("numpy", "cpu", "cuda"):
            x = V if kind == "numpy" else torch.as_tensor(V, device="cuda" if kind == "cuda" else "cpu")
            out = H.matvec(x)
            if kind == "numpy":
                assert isinstance(out, np.ndarray)
            else:
                assert torch.is_tensor(out) and out.device == x.device and out.dtype == F64
            out = out if kind == "numpy" else out.cpu().numpy()
            assert out.shape == (nk, nv)
            assert np.abs(out - ref).max() <= 1e-12 * scale, (nv, kind)
    v1 = torch.as_tensor(_probes(nk, 1)[:, 0], device="cuda")
    out1 = H.matvec(v1)
    assert out1.shape == (nk,) and (out1 - M @ v1).abs().max().item() <= 1e-12 * scale
    assert torch.equal(H.matvec(torch.zeros(nk, 3, dtype=F64, device="cuda")), torch.zeros(nk, 3, dtype=F64,
                                                                                          device="cuda"))
    diag = H.diagonal()
    diag = diag.cpu() if torch.is_tensor(diag) else torch.as_tensor(diag)
    assert (diag - M.diagonal().cpu()).abs().max().item() <= 1e-12 * scale


def test_shapes_and_empty_blocks():
    c = load_case("n7_cas44")
    oo, H = _hessian(c, "class")
    nk = oo.n_kappa
    assert H.matvec(np.zeros((nk, 0))).shape == (nk, 0)
    assert H.matvec(torch.zeros(nk, 0, dtype=F64, device="cuda")).shape == (nk, 0)
    for bad in (np.zeros(nk + 1), np.zeros((nk - 1, 2)), np.zeros((nk, 2, 2))):
        with pytest.raises(ValueError):
            H.matvec(bad)


def test_no_parameters_gives_empty_results():
    """A CAS with no core and no virtuals and frozen active rotations has n_kappa = 0."""
    from auto_oo_b200 import OO_energy
    from auto_oo_b200.synthetic import SyntheticMol, random_rdms
    mol = SyntheticMol(4, 4, seed=2)
    oo = OO_energy(mol, 4, 4, oao_mo_coeff=mol.random_oao_mo_coeff, freeze_active=True)
    assert oo.n_kappa == 0
    one, two = random_rdms(4, 4, seed=2)
    H = oo.analytic_hessian(one, two)
    assert H.matvec(torch.zeros(0, 3, dtype=F64)).shape == (0, 3)
    assert H.matvec(np.zeros(0)).shape == (0,)
    assert tuple(H.diagonal().shape) == (0,)


# ---------------------------------------------------------------------------------------------- determinism, graphs
@pytest.mark.parametrize("route", ["class", "full"])
def test_repeats_are_bit_identical_and_a_captured_product_replays(route):
    c = load_case("n43_cas34")
    oo, H = _hessian(c, route)
    nk = oo.n_kappa
    V = torch.as_tensor(_probes(nk, 9, seed=4), device="cuda")
    a, b = H.matvec(V), H.matvec(V)
    assert torch.equal(a, b)
    assert torch.equal(H.diagonal(), H.diagonal())
    static = V.clone()
    H.matvec(static)                                                  # warm-up: workspaces exist before capture
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = H.matvec(static)
    static.copy_(torch.as_tensor(_probes(nk, 9, seed=5), device="cuda"))
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, H.matvec(static))


def test_products_survive_interleaved_evaluations():
    c = load_case("n13_bigkappa")
    r = c.ref
    for path in ("class", "full"):
        oo = make_oo(c, integral_path=path)
        Cp = torch.as_tensor(r["mo_coeff_rot"])
        H = oo.analytic_hessian(c.one_rdm, c.two_rdm, mo_coeff=Cp)
        k2 = 0.3 * c.kappa
        oo.energy_from_kappa(k2, c.one_rdm, c.two_rdm)
        oo.energies_from_kappas(torch.stack([k2, 2 * k2]), c.one_rdm, c.two_rdm)
        for _ in range(3):
            oo.energy_gradient_hessian(torch.stack([k2, -k2]), c.one_rdm, c.two_rdm)
        oo.analytic_gradient(c.one_rdm, c.two_rdm)
        V = _probes(r["H"].shape[0], 5)
        assert np.abs(H.matvec(V) - r["H"] @ V).max() < TOL_GH * max(1.0, np.abs(V).sum(0).max()), path
        assert np.abs(np.asarray(H.diagonal()) - np.diagonal(r["H"])).max() < TOL_GH, path


# ---------------------------------------------------------------------------------------------- C ABI
def test_invalid_arguments_are_rejected_before_any_launch():
    lib = _lib.load()
    c = load_case("n7_cas44")
    oo, H = _hessian(c, "class")
    eng, ints = oo.engine, H._ints
    nk, ld = eng.nk, eng.ld
    V = torch.as_tensor(_probes(nk, 2), device="cuda")
    HV = torch.empty_like(V)
    nb = lib.oo_workspace_bytes(_lib.OO_WS_CLASS_HESSIAN_VECTOR, eng.na, ld, eng.nI, 2)
    assert nb > 0
    ws = torch.empty(nb, dtype=torch.uint8, device="cuda")
    cls, F = ints.cls[0].data_ptr(), H._F[0].data_ptr()
    d1, d2 = H._d1.data_ptr(), H._d2.data_ptr()
    pl, pr = eng.pair_l.data_ptr(), eng.pair_r.data_ptr()
    st = torch.cuda.current_stream().cuda_stream
    n0 = lib.oo_launch_count()
    args = [cls, F, d1, d2, eng.no, eng.na, eng.N, ld, eng.nIp, pl, pr, nk, V.data_ptr(), 2, HV.data_ptr(),
            ws.data_ptr(), nb, st]
    for i, bad in [(0, None), (12, None), (13, 0), (11, 0), (7, ld + 1), (8, eng.nIp - 1)]:
        a = list(args)
        a[i] = bad
        assert lib.oo_class_hessian_vector_f64(*a) == -1                             # OO_ERR_INVALID_ARG
    a = list(args)
    a[16] = nb - 1
    assert lib.oo_class_hessian_vector_f64(*a) == -3                                  # OO_ERR_WORKSPACE
    diag = torch.empty(nk, dtype=F64, device="cuda")
    assert lib.oo_class_hessian_diagonal_f64(cls, F, d1, d2, eng.no, eng.na, eng.N, ld, eng.nIp, pl, pr, 0,
                                             diag.data_ptr(), None, 0, st) == -1
    assert lib.oo_hessian_diagonal_f64(None, None, F, d1, d2, eng.no, eng.na, eng.N, ld, pl, pr, nk,
                                       diag.data_ptr(), ws.data_ptr(), nb, st) == -1
    assert lib.oo_launch_count() == n0
    assert lib.oo_class_hessian_vector_f64(*args) == 0
    assert lib.oo_class_hessian_diagonal_f64(cls, F, d1, d2, eng.no, eng.na, eng.N, ld, eng.nIp, pl, pr, nk,
                                             diag.data_ptr(), None, 0, st) == 0
    torch.cuda.synchronize()
    M = H.matrix()
    scale = M.abs().max().item()
    assert (HV - M @ V).abs().max().item() <= 1e-12 * scale and (diag - M.diagonal()).abs().max().item() <= 1e-12 * scale


def test_every_new_kernel_launches():
    from torch.profiler import ProfilerActivity, profile
    c = load_case("n11_cas43")
    runs = []
    for route in ("class", "full"):
        oo, H = _hessian(c, route)
        runs.append((H, torch.as_tensor(_probes(oo.n_kappa, 9), device="cuda")))
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        torch.ones(1, device="cuda").add_(1)                          # (the first kernel of a window can go unrecorded)
        for H, V in runs:
            H.matvec(V)                                               # 9 vectors: a block of 8 and a block of 1
            H.diagonal()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events()]
    count = {k: sum(k in n for n in names) for k in ("hvp_table_kernel", "hvp_scatter_kernel", "hvp_plane_kernel",
                                                     "hvp_reduce_kernel", "hvp_gather_kernel", "hess_diag_kernel",
                                                     "hess_gather_class_kernel")}
    assert all(n >= 1 for n in count.values()), count
    assert count["hvp_plane_kernel"] == 4 and count["hvp_gather_kernel"] == 4, count     # two passes per route


# ---------------------------------------------------------------------------------------------- a consumer
def test_conjugate_gradient_on_matvec_reproduces_the_newton_direction():
    """Preconditioned CG on (H + sigma I) x = -g with only matvec and diagonal: NewtonStep.newton_step's step."""
    from auto_oo_b200.utils.newton_raphson import NewtonStep
    c = load_case("n28_cas66")
    oo, H = _hessian(c, "class")
    Cp = torch.as_tensor(c.ref["mo_coeff_rot"])
    Gm = oo.analytic_gradient(c.one_rdm, c.two_rdm, mo_coeff=Cp).detach()
    g = oo.kappa_matrix_to_vector(Gm).to(device="cuda", dtype=F64)
    M = H.matrix()
    ns = NewtonStep(verbose=0)
    dp, lam0 = ns.newton_step(g, M)
    sigma = ns.mu + ns.rho * abs(lam0) if (lam0 < ns.lambda_min and ns.aug) else 0.0
    pre = torch.as_tensor(H.diagonal()).to(g.device) + sigma          # (in the array type of the RDMs: CPU here)
    assert bool((pre > 0).all())
    x = torch.zeros_like(g)
    r = -g.clone()
    z = r / pre
    p = z.clone()
    rz = torch.dot(r, z)
    for _ in range(20 * g.numel()):
        Ap = H.matvec(p) + sigma * p
        a = rz / torch.dot(p, Ap)
        x += a * p
        r -= a * Ap
        if torch.linalg.vector_norm(r) <= 1e-14 * torch.linalg.vector_norm(g):
            break
        z = r / pre
        rz_new = torch.dot(r, z)
        p = z + (rz_new / rz) * p
        rz = rz_new
    assert (x - dp).abs().max().item() < 1e-8
