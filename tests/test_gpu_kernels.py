"""GPU: every kernel group of liboo_b200.so, called through the C ABI (via HotPathEngine's
ctypes calls), against the CPU oracle and the golden outputs of the verbatim reference.
Tolerances: energy 1e-10 Ha; gradient/Hessian/matrix elements 1e-8 (BASELINE.json)."""
import os

import numpy as np
import pytest
import torch

from auto_oo_b200 import _lib
from helpers import ALL_CASES, SMALL_CASES, GOLDEN, TOL_E, TOL_GH, load_case

pytestmark = pytest.mark.gpu

F64 = torch.float64


@pytest.fixture(scope="module")
def lib():
    from auto_oo_b200 import _lib
    return _lib.load()


def engine_for(c, **kw):
    from auto_oo_b200.engine import HotPathEngine
    p = c.oracle()
    eng = HotPathEngine(c.int1e_ao, c.int2e_ao, c.oao_coeff, c.nuc, c.nao, len(p.occ_idx), c.ncas,
                        p.params_idx, **kw)
    return eng, p


# evaluation routes: the class path with / without the 8-fold ERI symmetry, and the complete transform
ROUTES = {"class": ("class", "auto"), "class_general": ("class", "off"), "full": ("full", "auto")}


def _stream():
    return torch.cuda.current_stream().cuda_stream


# ------------------------------------------------------------------ dense building blocks
@pytest.mark.parametrize("M,N,K,batch", [
    (64, 64, 64, 1), (130, 7, 9, 1), (257, 33, 50, 1), (1000, 114, 114, 1), (343, 8, 8, 3),
    (28 ** 3, 28, 28, 2), (100, 484, 201, 1), (576, 12996 // 4, 1153, 1),
    # 17-24 and 41-48 columns (the 24- and 48-wide tiles), 129-192 rows by >= 9472 columns (the 192-row tile); K = 1, 7,
    # 9, 15 mod 16 ends on a partial k-block
    (300, 20, 64, 2), (300, 20, 33, 2), (300, 20, 39, 2), (300, 20, 41, 2), (300, 20, 47, 2), (513, 45, 72, 1),
    (129, 42, 23, 3), (176, 9472, 64, 1), (176, 9472, 49, 1), (176, 9472, 55, 1), (176, 9476, 57, 1),
    (176, 9472, 63, 1),
])
def test_dgemm_tn(lib, M, N, K, batch):
    gen = torch.Generator(device="cuda").manual_seed(M * 7 + N)
    lda, ldb, ldc = M + (M & 1), N + (N & 1), N + (N & 1)
    At = torch.randn(batch, K, lda, dtype=F64, device="cuda", generator=gen)
    B = torch.randn(batch, K, ldb, dtype=F64, device="cuda", generator=gen)
    C = torch.full((batch, M, ldc), float("nan"), dtype=F64, device="cuda")
    rc = lib.oo_dgemm_tn_f64(At.data_ptr(), B.data_ptr(), C.data_ptr(), M, N, K, lda, ldb, ldc, batch,
                             K * lda, K * ldb, M * ldc, _stream())
    assert rc == 0
    ref = torch.matmul(At[:, :, :M].transpose(1, 2).cpu(), B[:, :, :N].cpu())
    err = (C[:, :, :N].cpu() - ref).abs().max().item()
    assert err < 1e-12 * K * 10, err


def test_dgemm_tn_shared_operands(lib):
    gen = torch.Generator(device="cuda").manual_seed(3)
    M, N, K, batch = 200, 20, 20, 4
    At = torch.randn(K, M, dtype=F64, device="cuda", generator=gen)
    B = torch.randn(batch, K, N, dtype=F64, device="cuda", generator=gen)
    C = torch.empty(batch, M, N, dtype=F64, device="cuda")
    assert lib.oo_dgemm_tn_f64(At.data_ptr(), B.data_ptr(), C.data_ptr(), M, N, K, M, N, N, batch,
                               0, K * N, M * N, _stream()) == 0
    ref = torch.matmul(At.T.cpu()[None], B.cpu())
    assert (C.cpu() - ref).abs().max().item() < 1e-11


@pytest.mark.parametrize("M,N,K,batch", [(45, 37, 29, 3), (46, 38, 30, 2), (114, 114, 114, 1), (256, 256, 256, 1),
                                         (64, 34, 130, 2), (34, 34, 34, 5), (8, 8, 8, 1)])
@pytest.mark.parametrize("tA,tB", [(0, 0), (1, 0), (0, 1), (1, 1)])
def test_dgemm_small_epilogue(lib, tA, tB, M, N, K, batch):
    """odd extents take the pipelined kernel, even ones (K <= 256) the one-shot panel kernel"""
    gen = torch.Generator(device="cuda").manual_seed(11)
    A = torch.randn(batch, *((K, M) if tA else (M, K)), dtype=F64, device="cuda", generator=gen)
    B = torch.randn(batch, *((N, K) if tB else (K, N)), dtype=F64, device="cuda", generator=gen)
    E = torch.randn(batch, M, N, dtype=F64, device="cuda", generator=gen)
    D = torch.empty(batch, M, N, dtype=F64, device="cuda")
    rc = lib.oo_dgemm_small_f64(tA, tB, M, N, K, 1.5, A.data_ptr(), A.shape[2], A[0].numel(),
                                B.data_ptr(), B.shape[2], B[0].numel(), -0.5, E.data_ptr(), N, M * N,
                                2.0, D.data_ptr(), N, M * N, batch, _stream())
    assert rc == 0
    opA = A.transpose(1, 2) if tA else A
    opB = B.transpose(1, 2) if tB else B
    ref = 1.5 * torch.matmul(opA.cpu(), opB.cpu()) - 0.5 * E.cpu() + 2.0 * torch.eye(M, N, dtype=F64)
    assert (D.cpu() - ref).abs().max().item() < 1e-12 * max(1, K // 16)


def test_pad_copy_roundtrip(lib):
    gen = torch.Generator(device="cuda").manual_seed(5)
    for rank in (2, 4):
        N, ld, b = 7, 8, 2
        x = torch.randn((b,) + (N,) * rank, dtype=F64, device="cuda", generator=gen)
        p = torch.full((b,) + (ld,) * rank, float("nan"), dtype=F64, device="cuda")
        y = torch.empty_like(x)
        assert lib.oo_pad_copy_f64(x.data_ptr(), p.data_ptr(), N, ld, rank, b, 1, _stream()) == 0
        assert lib.oo_pad_copy_f64(p.data_ptr(), y.data_ptr(), N, ld, rank, b, 0, _stream()) == 0
        assert torch.equal(x, y)
        sl = (slice(None),) + (slice(0, N),) * rank
        assert torch.equal(p[sl], x)
        assert float(p.sum()) == pytest.approx(float(x.sum()), rel=1e-12)   # padding is exactly zero


# ------------------------------------------------------------------ K1
@pytest.mark.parametrize("name", ALL_CASES)
def test_rotation_matches_reference(name):
    c = load_case(name)
    eng, p = engine_for(c)
    U = eng.from_padded(eng.rotation(c.kappa[None]), 2)[0].cpu().numpy()
    assert np.abs(U - c.ref["U"]).max() < 1e-13
    assert np.abs(U.T @ U - np.eye(c.nao)).max() < 1e-13
    Cp = eng.from_padded(eng.mo_coeff(eng.to_padded(c.oao_mo_coeff, 2), eng.rotation(c.kappa[None])), 2)
    assert np.abs(Cp[0].cpu().numpy() - c.ref["mo_coeff_rot"]).max() < 1e-12


def test_rotation_batched_large_norm():
    from oracle import oo_oracle as orc
    c = load_case("n13_bigkappa")
    eng, p = engine_for(c)
    gen = torch.Generator().manual_seed(1)
    kap = torch.randn(5, p.n_kappa, dtype=F64, generator=gen) * torch.tensor([0.0, 0.01, 0.3, 1.0, 3.0])[:, None]
    U = eng.from_padded(eng.rotation(kap), 2).cpu()
    for b in range(5):
        ref = orc.rotation_from_kappa(kap[b], p.params_idx, c.nao)
        assert (U[b] - ref).abs().max().item() < 2e-13


def test_expm_general_matrix(lib):
    gen = torch.Generator().manual_seed(2)
    N, ld, B = 9, 10, 3
    A = torch.randn(B, N, N, dtype=F64, generator=gen) * 0.4
    Ap = torch.zeros(B, ld, ld, dtype=F64)
    Ap[:, :N, :N] = A
    Ap = Ap.cuda()
    U = torch.empty_like(Ap)
    s = max(0, int(np.ceil(np.log2(A.abs().sum(1).max().item() / 0.95))))
    nbytes = lib.oo_workspace_bytes(1, N, ld, 0, B)
    ws = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    assert lib.oo_expm_f64(Ap.data_ptr(), -1.0, N, ld, B, s, U.data_ptr(), ws.data_ptr(), nbytes, _stream()) == 0
    ref = torch.linalg.matrix_exp(-A)
    assert (U.cpu()[:, :N, :N] - ref).abs().max().item() < 1e-12


@pytest.mark.parametrize("N", [5, 8, 31, 40, 47, 56, 64, 65, 70, 114, 130, 199, 255, 256, 258, 300])
def test_rotation_fused_and_multi_launch_routes(lib, N):
    """expm(-K) for sizes on both sides of the shared-memory limit (64: one CTA per matrix) and of the single-launch
    chain (256: one cooperative grid; above it one launch per product): explicit squaring count, and the
    device-side choice (per matrix in the fused kernel, max over the batch in the chain), against
    torch.linalg.matrix_exp."""
    from auto_oo_b200.engine import tril_pair_table
    gen = torch.Generator().manual_seed(N)
    ld = N + (N & 1)
    nk = N * (N - 1) // 2
    pl, pr = tril_pair_table(N, np.arange(nk))
    B = 4
    scale = torch.tensor([0.0, 0.02, 0.3, 2.5])[:, None] / np.sqrt(N)
    if N == 199:                                     # a batch wider than the grid: every CTA walks several tiles
        B, scale = 40, torch.linspace(0.0, 1.5, 40)[:, None] / np.sqrt(N)
    kap = torch.randn(B, nk, dtype=F64, generator=gen) * scale
    K = torch.zeros(B, N, N, dtype=F64)
    K[:, pl.astype(np.int64), pr.astype(np.int64)] = kap
    K = K - K.transpose(1, 2)
    ref = torch.linalg.matrix_exp(-K)
    s_host = max(0, int(np.ceil(np.log2(max(K.abs().sum(1).max().item(), 1e-300) / 0.95))))
    kd, pld, prd = kap.cuda(), torch.as_tensor(pl).cuda(), torch.as_tensor(pr).cuda()
    nbytes = lib.oo_workspace_bytes(1, N, ld, 0, B)
    ws = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    modes = [s_host] + ([-1] if N <= lib.oo_expm_device_squarings_max_n() else [])
    for s in modes:
        U = torch.full((B, ld, ld), float("nan"), dtype=F64, device="cuda")
        rc = lib.oo_kappa_rotation_f64(kd.data_ptr(), pld.data_ptr(), prd.data_ptr(), nk, N, ld, B, s, U.data_ptr(),
                                       ws.data_ptr(), nbytes, _stream())
        assert rc == 0
        U = U.cpu()
        assert (U[:, :N, :N] - ref).abs().max().item() < 5e-13, (N, s)
        if ld > N:
            assert U[:, N:, :].abs().max().item() == 0 and U[:, :, N:].abs().max().item() == 0
    if N > lib.oo_expm_device_squarings_max_n():      # the multi-launch route needs the host's choice
        assert lib.oo_kappa_rotation_f64(kd.data_ptr(), pld.data_ptr(), prd.data_ptr(), nk, N, ld, B, -1,
                                         U.data_ptr(), ws.data_ptr(), nbytes, _stream()) == -2


def test_expm_general_matrix_single_launch_chain(lib):
    """oo_expm_f64 on dense (not skew) matrices of 100 rows: the cooperative chain with an explicit squaring count."""
    gen = torch.Generator().manual_seed(12)
    N, ld, B = 99, 100, 3
    A = torch.randn(B, N, N, dtype=F64, generator=gen) * (0.6 / np.sqrt(N))
    Ap = torch.zeros(B, ld, ld, dtype=F64)
    Ap[:, :N, :N] = A
    Ap = Ap.cuda()
    U = torch.full_like(Ap, float("nan"))
    s = max(0, int(np.ceil(np.log2(A.abs().sum(1).max().item() / 0.95))))
    nbytes = lib.oo_workspace_bytes(1, N, ld, 0, B)
    ws = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    for sign in (-1.0, 1.0):
        assert lib.oo_expm_f64(Ap.data_ptr(), sign, N, ld, B, s, U.data_ptr(), ws.data_ptr(), nbytes, _stream()) == 0
        ref = torch.linalg.matrix_exp(sign * A)
        assert (U.cpu()[:, :N, :N] - ref).abs().max().item() < 1e-12
        assert U[:, N:, :].abs().max().item() == 0 and U[:, :, N:].abs().max().item() == 0


def test_graph_replay_above_the_shared_memory_limit():
    """70 orbitals: the rotation is the cooperative single-launch chain with the squaring count chosen on the device;
    it is captured into the evaluation's CUDA graph like any other launch, and replays follow new kappa values
    (small and large norm: different squaring counts through the same graph)."""
    from auto_oo_b200 import OO_energy
    from auto_oo_b200.synthetic import SyntheticMol, random_rdms
    dev = torch.device("cuda", 0)
    mol = SyntheticMol(70, 20, seed=8, device=dev)
    oo = OO_energy(mol, 4, 4, oao_mo_coeff=mol.random_oao_mo_coeff, device=dev)
    eng = oo.engine
    assert eng.N <= eng.lib.oo_expm_device_squarings_max_n()
    one, two = random_rdms(4, 4, seed=8, device=dev)
    Coao = eng.to_padded(oo.oao_mo_coeff, 2)
    gen = torch.Generator().manual_seed(9)
    for trial, amp in enumerate([0.01, 0.02, 1.0, 0.003]):
        kap = (torch.randn(2, eng.nk, dtype=F64, generator=gen) * amp).cuda()
        Eg, Gg, Hg = eng.evaluate_graphed(Coao, one, two, kappa=kap)
        E, G, H = eng.evaluate(Coao, one, two, kappa=kap)
        assert torch.equal(Eg, E) and torch.equal(Gg, G) and torch.equal(Hg, H)
        s = eng.squarings_for(kap)
        Es, Gs, Hs = eng.evaluate(Coao, one, two, kappa=kap, squarings=s)          # host-chosen count: same arithmetic
        assert torch.equal(Es, E) and torch.equal(Hs, H)
    assert len(eng._ws["graphs"]) == 1


def test_graph_replay_equals_direct_evaluation():
    """evaluate_graphed (one CUDA-graph launch per call) against evaluate, across changing inputs, batch sizes
    and interleaved non-graph calls that share the workspaces."""
    c = load_case("n28_cas66")
    eng, p = engine_for(c)
    Coao = eng.to_padded(c.oao_mo_coeff, 2)
    d1, d2 = eng.dev(c.one_rdm), eng.dev(c.two_rdm)
    gen = torch.Generator().manual_seed(4)
    for trial, B in enumerate([1, 3, 1, 3, 8]):
        kap = (torch.randn(B, p.n_kappa, dtype=F64, generator=gen) * 0.05).cuda()
        Eg, Gg, Hg = eng.evaluate_graphed(Coao, d1 * (1 + 0.01 * trial), d2, kappa=kap)   # first sight of B: direct
        if trial == 2:                                   # a non-graph call with a larger batch re-sizes workspaces
            eng.evaluate(Coao, d1, d2, kappa=torch.zeros(16, p.n_kappa, dtype=F64, device="cuda"))
        E, G, H = eng.evaluate(Coao, d1 * (1 + 0.01 * trial), d2, kappa=kap)
        assert torch.equal(Eg, E) and torch.equal(Gg, G) and torch.equal(Hg, H)
    assert len(eng._ws["graphs"]) == 2 and len(eng._ws["graph_seen"]) == 3        # B = 1, 3 captured; B = 8 seen once
    eng.evaluate_graphed(Coao, d1, d2, kappa=None, want_hessian=False)
    Eg, Gg, Hg = eng.evaluate_graphed(Coao, d1, d2, kappa=None, want_hessian=False)
    E, G, _ = eng.evaluate(Coao, d1, d2, want_hessian=False)
    assert Hg is None and torch.equal(Eg, E) and torch.equal(Gg, G)
    # outputs too large to pin inside a graph: the call falls back to the direct path
    eng.GRAPH_MAX_OUTPUT_BYTES = 1
    try:
        n_graphs = len(eng._ws["graphs"])
        kap = (torch.randn(2, p.n_kappa, dtype=F64, generator=gen) * 0.05).cuda()
        Ef, Gf, Hf = eng.evaluate_graphed(Coao, d1, d2, kappa=kap)
        E, G, H = eng.evaluate(Coao, d1, d2, kappa=kap)
        assert torch.equal(Ef, E) and torch.equal(Hf, H) and len(eng._ws["graphs"]) == n_graphs
    finally:
        del eng.GRAPH_MAX_OUTPUT_BYTES
    ref = c.ref
    E, G, H = eng.evaluate_graphed(Coao, d1, d2, kappa=c.kappa[None].cuda())
    assert abs(E.item() - float(ref["E"])) < TOL_E
    assert np.abs(G[0].cpu().numpy() - ref["G"]).max() < TOL_GH and np.abs(H[0].cpu().numpy() - ref["H"]).max() < TOL_GH


@pytest.mark.parametrize("name", ["n11_cas43", "n34_cas44", "n43_cas34"])
def test_hessian_output_guards_stay_untouched(name, lib):
    """(compute-sanitizer is not available on the GPU pool.)  The Hessian is written into the middle of a larger
    buffer whose guard zones hold a bit pattern; every assembly kernel (per-thread, row-tiled, bulk-async
    streamed) must leave the guards alone and fill every element in between."""
    c = load_case(name)
    eng, p = engine_for(c)
    Coao = eng.to_padded(c.oao_mo_coeff, 2)
    d1, d2 = eng.dev(c.one_rdm), eng.dev(c.two_rdm)
    nk, B, pad = eng.nk, 2, 4096
    kap = torch.stack([c.kappa, 0.5 * c.kappa]).cuda()
    sentinel = float.fromhex("-0x1.deadbeef00000p+700")
    ref = None
    for mode in (1, 2):
        big = torch.full((B * nk * nk + 2 * pad,), sentinel, dtype=F64, device="cuda")
        H = big[pad:pad + B * nk * nk].view(B, nk, nk)
        try:
            eng.flags = 2 * mode                      # OO_FLAG_HESSIAN_ASSEMBLE_PER_ELEMENT / _TILED
            eng.evaluate(Coao, d1, d2, kappa=kap, H_out=H)
        finally:
            eng.flags = 0
        torch.cuda.synchronize()
        assert bool((big[:pad] == sentinel).all()) and bool((big[-pad:] == sentinel).all())
        assert not bool((H == sentinel).any())
        ref = H.clone() if ref is None else ref
        assert (H - ref).abs().max().item() < 1e-11
    assert np.abs(ref[0].cpu().numpy() - c.ref["H"]).max() < TOL_GH


# ------------------------------------------------------------------ K2
@pytest.mark.parametrize("name", SMALL_CASES)
def test_integral_transforms_match_reference(name):
    c = load_case(name)
    eng, p = engine_for(c)
    Cp = eng.to_padded(c.ref["mo_coeff_rot"], 2)
    h = eng.from_padded(eng.int1e_transform(Cp), 2)[0].cpu().numpy()
    g = eng.from_padded(eng.int2e_transform(Cp), 4)[0].cpu().numpy()
    assert np.abs(h - c.ref["int1e_mo"]).max() < 1e-11
    assert np.abs(g - c.ref["int2e_mo"]).max() < 1e-11


def test_general_4index_four_matrices():
    from auto_oo_b200.engine import HotPathEngine
    d = np.load(os.path.join(GOLDEN, "general_4index_n6.npz"))
    eng = HotPathEngine(np.zeros((6, 6)), d["M"], np.eye(6), 0.0, 6, 0, 6, [0])
    Cs = [eng.to_padded(d[k], 2) for k in ("C0", "C1", "C2", "C3")]
    out = eng.from_padded(eng.int2e_transform(*Cs), 4)[0].cpu().numpy()
    assert np.abs(out - d["out"]).max() < 1e-11


@pytest.mark.parametrize("name", ["n28_cas66", "n43_cas34"])
def test_int2e_transform_vs_oracle_and_identity(name):
    from oracle import oo_oracle as orc
    c = load_case(name)
    eng, p = engine_for(c)
    Cp = eng.to_padded(c.ref["mo_coeff_rot"], 2)
    g = eng.from_padded(eng.int2e_transform(Cp), 4)[0].cpu()
    ref = orc.transform_2e(c.int2e_ao, c.ref["mo_coeff_rot"])
    assert (g - ref).abs().max().item() < 1e-10
    ident = eng.to_padded(np.eye(c.nao), 2)
    g_id = eng.from_padded(eng.int2e_transform(ident), 4)[0].cpu().numpy()
    assert np.array_equal(g_id, np.asarray(c.int2e_ao))     # exact: sums of x*1 and x*0


def test_int2e_transform_batched_kappa_sweep():
    from oracle import oo_oracle as orc
    c = load_case("n11_cas43")
    eng, p = engine_for(c)
    gen = torch.Generator().manual_seed(4)
    kap = torch.randn(3, p.n_kappa, dtype=F64, generator=gen) * 0.1
    C = eng.mo_coeff(eng.to_padded(c.oao_mo_coeff, 2), eng.rotation(kap))
    g = eng.from_padded(eng.int2e_transform(C), 4).cpu()
    for b in range(3):
        ref = orc.transform_2e(c.int2e_ao, p.rotated_mo(kap[b]))
        assert (g[b] - ref).abs().max().item() < 1e-11


# ------------------------------------------------------------------ K3 / K4
@pytest.mark.parametrize("route", list(ROUTES))
@pytest.mark.parametrize("name", ALL_CASES)
def test_full_evaluation_matches_reference(name, route):
    c = load_case(name)
    path, sym = ROUTES[route]
    eng, p = engine_for(c, eri_symmetry=sym)
    if path == "class":
        assert eng.eri_is_symmetric() == (sym == "auto")          # every fixture is 8-fold symmetric
    E, G, H = eng.evaluate(eng.to_padded(c.oao_mo_coeff, 2), c.one_rdm, c.two_rdm, kappa=c.kappa[None],
                           path=path)
    assert abs(E.item() - float(c.ref["E"])) < TOL_E
    assert np.abs(G[0].cpu().numpy() - c.ref["G"]).max() < TOL_GH
    assert np.abs(H[0].cpu().numpy() - c.ref["H"]).max() < TOL_GH
    E0, G0, _ = eng.evaluate(eng.to_padded(c.oao_mo_coeff, 2), c.one_rdm, c.two_rdm, want_hessian=False,
                             path=path)
    assert abs(E0.item() - float(c.ref["E0"])) < TOL_E
    assert np.abs(G0[0].cpu().numpy() - c.ref["G0"]).max() < TOL_GH


@pytest.mark.parametrize("name", ["n7_cas44", "n8_nocore", "n11_cas43", "n28_cas66"])
def test_active_hamiltonian_and_fock_stages(name):
    from oracle import oo_oracle as orc
    c = load_case(name)
    eng, p = engine_for(c)
    Cp = eng.to_padded(c.ref["mo_coeff_rot"], 2)
    h, g = eng.mo_integrals(Cp)
    c0, c1, c2 = eng.active_hamiltonian(h, g)
    assert abs(c0.item() - float(c.ref["c0"])) < TOL_E
    assert np.abs(c1[0].cpu().numpy() - c.ref["c1"]).max() < 1e-11
    assert np.abs(c2[0].cpu().numpy() - c.ref["c2"]).max() < 1e-11
    d1, d2 = eng.dev(c.one_rdm), eng.dev(c.two_rdm)
    FI, FA, F, Gm, gv = eng.fock_gradient(h, g, d1, d2)
    ho, go = p.mo_integrals(c.kappa)
    for got, ref in ((FI, orc.fock_core(ho, go, p.occ_idx)),
                     (FA, orc.fock_active(go, c.one_rdm, p.act_idx)),
                     (F, orc.fock_generalized(ho, go, c.one_rdm, c.two_rdm, p.occ_idx, p.act_idx)),
                     (Gm, orc.gradient_matrix(ho, go, c.one_rdm, c.two_rdm, p.occ_idx, p.act_idx))):
        assert (eng.from_padded(got, 2)[0].cpu() - ref).abs().max().item() < 1e-10
    assert np.abs(gv[0].cpu().numpy() - c.ref["G"]).max() < TOL_GH


@pytest.mark.parametrize("name", ["n7_cas44", "n11_cas43"])
def test_gradient_vjp_matches_autograd(name):
    """Adjoint of (gamma, Gamma) -> G (what jacobian(orbital_gradient, theta) needs, oo_pqc.py:113-123)."""
    from oracle import oo_oracle as orc
    c = load_case(name)
    eng, p = engine_for(c)
    h, g = eng.mo_integrals(eng.to_padded(c.ref["mo_coeff_rot"], 2))
    d1, d2 = eng.dev(c.one_rdm), eng.dev(c.two_rdm)
    FI, FA, F, Gm, gv = eng.fock_gradient(h, g, d1, d2)
    gen = torch.Generator().manual_seed(8)
    Gbar = torch.randn(c.nao, c.nao, dtype=F64, generator=gen)
    g1, g2 = eng.fock_gradient_vjp(g[0], FI[0], eng.to_padded(Gbar, 2))
    ho, go = p.mo_integrals(c.kappa)
    one = c.one_rdm.clone().requires_grad_(True)
    two = c.two_rdm.clone().requires_grad_(True)
    Gref = orc.gradient_matrix(ho, go, one, two, p.occ_idx, p.act_idx)
    r1, r2 = torch.autograd.grad((Gref * Gbar).sum(), (one, two))
    assert (g1.cpu() - r1).abs().max().item() < 1e-10
    assert (g2.cpu() - r2).abs().max().item() < 1e-10


@pytest.mark.parametrize("sym", ["auto", "auto-pair", "off"])
@pytest.mark.parametrize("name", ["n7_cas44", "n8_nocore", "n13_cas22", "n28_cas66", "mol_ch2nh_sto3g_cas44"])
def test_class_transform_equals_slices_of_full_transform(name, sym):
    """J[m,n,a,b] = g'[a,b,m,n], K[n,m,a,b] = g'[a,m,n,b] and the h' row of the class buffer, through the
    symmetric class transform (AO integrals 8-fold packed, or with one pair packed) and the general one."""
    c = load_case(name)
    packing = "pair" if sym == "auto-pair" else "8fold"
    sym = sym.split("-")[0]
    eng, p = engine_for(c, eri_symmetry=sym, eri_packing=packing)
    assert eng.eri_is_symmetric() == (sym == "auto")
    Cp = eng.to_padded(c.ref["mo_coeff_rot"], 2)
    cls = eng.class_integrals(Cp)[0].cpu()
    g = eng.from_padded(eng.int2e_transform(Cp), 4)[0].cpu()
    h = eng.from_padded(eng.int1e_transform(Cp), 2)[0].cpu()
    N, nI, nIp = c.nao, eng.nI, eng.nIp
    K = cls[:nIp * nIp].reshape(nIp, nIp, eng.ld, eng.ld)[:nI, :nI, :N, :N]
    J = cls[nIp * nIp:2 * nIp * nIp].reshape(nIp, nIp, eng.ld, eng.ld)[:nI, :nI, :N, :N]
    assert (J - g[:, :, :nI, :nI].permute(2, 3, 0, 1)).abs().max().item() < 1e-11
    assert (K - g[:, :nI, :nI, :].permute(2, 1, 0, 3)).abs().max().item() < 1e-11
    assert (cls[-1][:N, :N] - h).abs().max().item() < 1e-12
    if eng.ld > N:                                       # zero padding survives
        assert cls[:, N:, :].abs().max().item() == 0.0 and cls[:, :, N:].abs().max().item() == 0.0
    if sym == "auto":                                    # class-pair packing fused into the quarter-2 epilogue vs a separate pass
        try:
            eng.flags = _lib.OO_FLAG_CLASS_UNFUSED_PACK
            cls_u = eng.class_integrals(Cp)[0].cpu()
        finally:
            eng.flags = 0
        assert torch.equal(cls_u, cls)


def test_eri_symmetry_defect_and_pair_packing(lib):
    c = load_case("n11_cas43")
    eng, _ = engine_for(c)
    ld = eng.ld
    assert eng.eri_is_symmetric() and max(eng.eri_defect[:2]) <= 1e-13 * eng.eri_defect[2]
    assert abs(eng.eri_defect[2] - np.abs(c.int2e_ao).max()) < 1e-15
    ldp = int(lib.oo_pair_ld(ld))
    g = eng.g_ao.cpu()
    rows, cols = np.tril_indices(ld)                              # p >= q, pq = p(p+1)/2 + q
    assert eng.eri_packing == "8fold"                             # default: both pairs packed, g8[(r>=s), (p>=q)]
    g8 = eng.packed_eri().cpu()
    assert g8.shape == (len(rows), ldp) and ldp % 2 == 0 and ldp >= ld * (ld + 1) // 2
    assert torch.equal(g8[:, :len(rows)], g[rows, cols][:, rows, cols])
    assert g8[:, len(rows):].abs().max().item() == 0.0 if ldp > len(rows) else True
    eng.g_packed, eng.eri_packing = None, "pair"                  # one pair packed, g[r, s, (p>=q)]
    gp = eng.packed_eri().cpu()
    assert gp.shape == (ld, ld, ldp)
    assert torch.equal(gp[:, :, :len(rows)], g[:, :, rows, cols])
    assert gp[:, :, len(rows):].abs().max().item() == 0.0 if ldp > len(rows) else True
    # break each symmetry in turn: the defect reports it and the engine falls back to the general route
    for kind in (0, 1):
        g2 = torch.as_tensor(c.int2e_ao).clone()
        if kind == 0:
            g2[3, 1, 2, 5] += 1e-6                                # (pq|rs) != (qp|rs)
        else:
            g2[3, 1, 2, 5] += 1e-6
            g2[1, 3, 2, 5] += 1e-6                                # pq-symmetric, but (pq|rs) != (rs|pq)
        from auto_oo_b200.engine import HotPathEngine
        p = c.oracle()
        e2 = HotPathEngine(c.int1e_ao, g2, c.oao_coeff, c.nuc, c.nao, len(p.occ_idx), c.ncas, p.params_idx)
        assert not e2.eri_is_symmetric()
        assert abs(e2.eri_defect[kind] - 1e-6) < 1e-12
        if kind == 1:
            assert e2.eri_defect[0] == 0.0


def test_asymmetric_integrals_take_the_general_class_route():
    """No symmetry of M is assumed by the reference's transform (oo_energy.py:21-30); for a tensor without
    the 8-fold symmetry the class path must still equal slices of the complete transform."""
    from auto_oo_b200.engine import HotPathEngine
    gen = torch.Generator().manual_seed(3)
    N, no, na = 9, 2, 3
    g = torch.randn(N, N, N, N, dtype=F64, generator=gen)
    C = torch.randn(N, N, dtype=F64, generator=gen)
    eng = HotPathEngine(np.eye(N), g, np.eye(N), 0.0, N, no, na, [0])
    assert not eng.eri_is_symmetric()
    Cp = eng.to_padded(C, 2)
    cls = eng.class_integrals(Cp)[0].cpu()
    gm = torch.einsum('pi,qj,rk,sl,pqrs->ijkl', C, C, C, C, g)
    nI, nIp, ld = no + na, eng.nIp, eng.ld
    K = cls[:nIp * nIp].reshape(nIp, nIp, ld, ld)[:nI, :nI, :N, :N]
    J = cls[nIp * nIp:2 * nIp * nIp].reshape(nIp, nIp, ld, ld)[:nI, :nI, :N, :N]
    assert (J - gm[:, :, :nI, :nI].permute(2, 3, 0, 1)).abs().max().item() < 1e-11
    assert (K - gm[:, :nI, :nI, :].permute(2, 1, 0, 3)).abs().max().item() < 1e-11


def test_transpose_kernel(lib):
    gen = torch.Generator(device="cuda").manual_seed(21)
    x = torch.randn(100, 37, dtype=F64, device="cuda", generator=gen)
    y = torch.empty(37, 100, dtype=F64, device="cuda")
    assert lib.oo_transpose_f64(x.data_ptr(), y.data_ptr(), 100, 37, _stream()) == 0
    assert torch.equal(y, x.T)


@pytest.mark.parametrize("name", ["n7_cas44", "n11_cas43"])
def test_class_path_stages_and_vjp(name):
    from oracle import oo_oracle as orc
    c = load_case(name)
    eng, p = engine_for(c)
    ints = eng.integrals(eng.to_padded(c.ref["mo_coeff_rot"], 2), kind="class")
    c0, c1, c2 = ints.active_hamiltonian()
    assert abs(c0.item() - float(c.ref["c0"])) < TOL_E
    assert np.abs(c1[0].cpu().numpy() - c.ref["c1"]).max() < 1e-11
    assert np.abs(c2[0].cpu().numpy() - c.ref["c2"]).max() < 1e-11
    d1, d2 = eng.dev(c.one_rdm), eng.dev(c.two_rdm)
    FI, FA, F, Gm, gv = ints.fock_gradient(d1, d2)
    ho, go = p.mo_integrals(c.kappa)
    for got, ref in ((FI, orc.fock_core(ho, go, p.occ_idx)), (FA, orc.fock_active(go, c.one_rdm, p.act_idx)),
                     (F, orc.fock_generalized(ho, go, c.one_rdm, c.two_rdm, p.occ_idx, p.act_idx))):
        assert (eng.from_padded(got, 2)[0].cpu() - ref).abs().max().item() < 1e-10
    gen = torch.Generator().manual_seed(8)
    Gbar = torch.randn(c.nao, c.nao, dtype=F64, generator=gen)
    g1, g2 = ints.fock_gradient_vjp(FI, eng.to_padded(Gbar, 2))
    one = c.one_rdm.clone().requires_grad_(True)
    two = c.two_rdm.clone().requires_grad_(True)
    Gref = orc.gradient_matrix(ho, go, one, two, p.occ_idx, p.act_idx)
    r1, r2 = torch.autograd.grad((Gref * Gbar).sum(), (one, two))
    assert (g1.cpu() - r1).abs().max().item() < 1e-10 and (g2.cpu() - r2).abs().max().item() < 1e-10


def test_batched_class_path_matches_per_evaluation_results():
    """kappa batch through the batched launches (class path) == one evaluation at a time, and per-evaluation
    RDMs (stride != 0) are honoured."""
    c = load_case("n11_cas43")
    eng, p = engine_for(c)
    gen = torch.Generator().manual_seed(12)
    B = 5
    kap = torch.randn(B, p.n_kappa, dtype=F64, generator=gen) * 0.1
    one = c.one_rdm[None] + 0.01 * torch.randn(B, c.ncas, c.ncas, dtype=F64, generator=gen)
    one = 0.5 * (one + one.transpose(1, 2))
    two = c.two_rdm[None].repeat(B, 1, 1, 1, 1) * torch.linspace(0.8, 1.2, B, dtype=F64)[:, None, None, None, None]
    Coao = eng.to_padded(c.oao_mo_coeff, 2)
    E, G, H = eng.evaluate(Coao, one, two, kappa=kap, path="class")
    for b in range(B):
        e1, g1, h1 = eng.evaluate(Coao, one[b], two[b], kappa=kap[b:b + 1], path="class")
        assert abs(E[b].item() - e1.item()) < 1e-12
        assert (G[b] - g1[0]).abs().max().item() < 1e-12 and (H[b] - h1[0]).abs().max().item() < 1e-12
        e, gvec, hm = p.evaluate(one[b], two[b], kap[b])
        assert abs(E[b].item() - e.item()) < TOL_E
        assert (G[b].cpu() - gvec).abs().max().item() < TOL_GH
        assert (H[b].cpu() - hm).abs().max().item() < TOL_GH


def test_batched_evaluation_equals_single():
    c = load_case("n13_cas22")
    eng, p = engine_for(c)
    gen = torch.Generator().manual_seed(6)
    kap = torch.randn(4, p.n_kappa, dtype=F64, generator=gen) * 0.05
    Coao = eng.to_padded(c.oao_mo_coeff, 2)
    E, G, H = eng.evaluate(Coao, c.one_rdm, c.two_rdm, kappa=kap)
    for b in range(4):
        e, gvec, hm = p.evaluate(c.one_rdm, c.two_rdm, kap[b])
        assert abs(E[b].item() - e.item()) < TOL_E
        assert (G[b].cpu() - gvec).abs().max().item() < TOL_GH
        assert (H[b].cpu() - hm).abs().max().item() < TOL_GH


# ------------------------------------------------------------------ multi-GPU orchestration on the CUDA GEMM
@pytest.mark.parametrize("mode", ["reduce_scatter", "all_to_all"])
def test_slab_transform_world1_on_cuda_gemm(mode):
    """world_size 1: the slab-parallel driver on the sm_100a GEMM must reproduce the single-GPU
    transform (the world_size 2 exchange is covered on CPU/gloo and by tools/slab_transform_check.py)."""
    from auto_oo_b200.distributed import SlabTransform
    from auto_oo_b200.engine import HotPathEngine
    n = 12
    gen = torch.Generator(device="cuda").manual_seed(17)
    g = torch.randn(n, n, n, n, dtype=F64, device="cuda", generator=gen)
    Cs = [torch.randn(n, n, dtype=F64, device="cuda", generator=gen) for _ in range(4)]
    ref = HotPathEngine.for_tensors(n).int2e_transform(*Cs, g_ao=g)[0]
    st = SlabTransform(n, mode=mode)
    out = st(st.take_slab(g), *Cs)
    assert torch.equal(out, ref)          # same kernel, same summation order: bit-identical
    cpu = torch.einsum('pi,qj,rk,sl,pqrs->ijkl', *[c.cpu() for c in Cs], g.cpu())
    assert (out.cpu() - cpu).abs().max().item() < 1e-10


@pytest.mark.parametrize("name", ["n7_cas44", "n7_cas44_frozen", "n8_nocore", "n11_cas43", "n28_cas66", "n34_cas44"])
def test_class_hessian_sparse_and_dense_routes_agree(name, lib):
    """oo_class_hessian_f64: dense act-act block + sparse remainder (default) against the single
    dense GEMM over all of At (OO_FLAG_HESSIAN_DENSE), and both against the verbatim reference."""
    c = load_case(name)
    eng, p = engine_for(c)
    ints = eng.integrals(eng.to_padded(c.ref["mo_coeff_rot"], 2), kind="class")
    d1, d2 = eng.dev(c.one_rdm), eng.dev(c.two_rdm)
    F = ints.fock_gradient(d1, d2, want_matrix=False, want_vector=False)[2]
    Hs = ints.hessian(F, d1, d2).clone()
    try:
        eng.flags = _lib.OO_FLAG_HESSIAN_DENSE
        Hd = ints.hessian(F, d1, d2).clone()
    finally:
        eng.flags = 0
    assert (Hs - Hd).abs().max().item() < 1e-11
    try:                                                  # occ-occ columns one by one instead of in pairs
        eng.flags = _lib.OO_FLAG_HESSIAN_SPMM_UNPAIRED
        Hu = ints.hessian(F, d1, d2).clone()
    finally:
        eng.flags = 0
    assert (Hs - Hu).abs().max().item() < 1e-11
    assert np.abs(Hs.cpu().numpy() - c.ref["H"]).max() < TOL_GH
    assert np.abs(Hd.cpu().numpy() - c.ref["H"]).max() < TOL_GH
    # assembly: row-tiled / shared-memory-transposed (default) against one thread per element; a pair list that
    # is not sorted by row (reversed) takes the per-thread form inside the tiled kernel
    N = c.nao
    rev = torch.arange(eng.nk - 1, -1, -1, device=eng.device)
    idx = torch.arange(N, device=eng.device, dtype=torch.int32)
    flat = (eng.pair_l.long() * N + eng.pair_r.long())
    for mode in (1, 2):                                   # 1: per-thread kernel, 2: row-tiled kernel (0: by size)
        try:
            eng.flags = 2 * mode                      # OO_FLAG_HESSIAN_ASSEMBLE_PER_ELEMENT / _TILED
            Hp = ints.hessian(F, d1, d2).clone()
            Hr = ints.hessian(F, d1, d2, pair_l=eng.pair_l[rev].contiguous(), pair_r=eng.pair_r[rev].contiguous())
            # every (row, column) pair, the list OrbitalHessian.dense() passes: rows sorted, columns 0..N-1
            Hall = ints.hessian(F, d1, d2, pair_l=idx.repeat_interleave(N).contiguous(),
                                pair_r=idx.repeat(N).contiguous())
        finally:
            eng.flags = 0
        assert (Hs - Hp).abs().max().item() < 1e-11
        assert (Hr - Hs[rev][:, rev]).abs().max().item() < 1e-11
        assert (Hall[flat][:, flat] - Hs).abs().max().item() < 1e-11


@pytest.mark.parametrize("nao,nelec,ncas,nelecas,freeze", [
    (5, 4, 1, 2, False), (5, 4, 1, 2, True), (6, 2, 2, 2, False), (9, 10, 3, 2, False), (12, 6, 5, 4, True),
    (3, 2, 3, 2, False), (4, 8, 1, 2, False), (66, 20, 3, 2, False)])
def test_unusual_orbital_spaces_against_the_oracle(nao, nelec, ncas, nelecas, freeze):
    """one active orbital, no core, no virtuals, every orbital active, odd sizes, N just above the fused-expm
    limit: E, gradient and Hessian of the class path and of the complete transform against the CPU oracle"""
    from auto_oo_b200.engine import HotPathEngine
    from auto_oo_b200.synthetic import SyntheticMol, random_rdms, random_kappa
    from oracle import oo_oracle as orc
    mol = SyntheticMol(nao, nelec, seed=nao + ncas)
    occ, act, virt = mol.get_active_space_idx(ncas, nelecas)
    pidx = orc.non_redundant_indices(occ, act, virt, freeze)
    if len(pidx) == 0:
        pytest.skip("no non-redundant rotation")
    prob = orc.OracleProblem(mol.int1e_ao, mol.int2e_ao, mol.oao_coeff, mol.random_oao_mo_coeff, mol.nuc, nelec, ncas,
                             nelecas, freeze)
    one, two = random_rdms(ncas, nelecas, seed=3)
    kap = random_kappa(len(pidx), seed=3, scale=0.2)
    Eo, Go, Ho = prob.evaluate(one, two, kap, ispace=nao > 13)
    eng = HotPathEngine(mol.int1e_ao, mol.int2e_ao, mol.oao_coeff, mol.nuc, nao, len(occ), ncas, pidx)
    Coao = eng.to_padded(mol.random_oao_mo_coeff, 2)
    for path in ("class", "full"):
        E, G, H = eng.evaluate(Coao, one, two, kappa=kap[None], path=path)
        assert abs(E.item() - float(Eo)) < TOL_E, path
        assert (G[0].cpu() - Go).abs().max().item() < TOL_GH, path
        assert (H[0].cpu() - Ho).abs().max().item() < TOL_GH, path


@pytest.mark.parametrize("nao,nelec,ncas,nelecas", [(64, 64, 4, 4), (70, 100, 6, 6), (56, 36, 4, 4), (60, 60, 4, 4),
                                                    (57, 44, 6, 6), (129, 40, 4, 4), (40, 32, 4, 4), (60, 80, 4, 4),
                                                    (62, 80, 6, 6), (64, 84, 6, 6), (64, 88, 6, 6)])
def test_class_transform_with_wide_class_index(nao, nelec, ncas, nelecas):
    """Class index nIp in (16, 64]: exercises the 24/32/40/48/64-wide GEMM tiles, every triangular quarter-2
    configuration (nI = 18, 20, 32, 34, 42 .. 47; 54 takes the rectangular GEMM), an odd basis size and, at 129
    orbitals, the staged 128 x 128 class-expand epilogue with a ragged edge (small fixtures only reach the 16-wide
    tile).  A batch of three kappas: where nIp is 18 .. 24 or 42 .. 48 the first two share one quarter-1 GEMM (36 .. 48
    or 84 .. 96 columns) and the third runs alone.  Class tensors must equal slices of the full transform, E / G / H
    of both paths must agree, and every member must match the CPU class oracle."""
    from auto_oo_b200.engine import HotPathEngine
    from auto_oo_b200.synthetic import SyntheticMol, random_rdms, random_kappa
    from oracle import class_oracle
    from oracle import oo_oracle as orc
    mol = SyntheticMol(nao, nelec, seed=11)
    occ, act, virt = mol.get_active_space_idx(ncas, nelecas)
    pidx = orc.non_redundant_indices(occ, act, virt, False)
    eng = HotPathEngine(mol.int1e_ao, mol.int2e_ao, mol.oao_coeff, mol.nuc, nao, len(occ), ncas, pidx)
    one, two = random_rdms(ncas, nelecas, seed=2)
    k0 = random_kappa(len(pidx), seed=2, scale=0.05)
    kap = torch.stack([k0, random_kappa(len(pidx), seed=3, scale=0.05), -0.5 * k0])
    Coao = eng.to_padded(mol.random_oao_mo_coeff, 2)
    C = eng.mo_coeff(Coao, eng.rotation(kap))
    cls = eng.class_integrals(C)
    g = eng.int2e_transform(C)
    nI, nIp, ld = eng.nI, eng.nIp, eng.ld
    for b in range(3):
        K = cls[b, :nIp * nIp].reshape(nIp, nIp, ld, ld)[:nI, :nI]
        J = cls[b, nIp * nIp:2 * nIp * nIp].reshape(nIp, nIp, ld, ld)[:nI, :nI]
        assert (J - g[b][:, :, :nI, :nI].permute(2, 3, 0, 1)).abs().max().item() < 1e-10, b
        assert (K - g[b][:, :nI, :nI, :].permute(2, 1, 0, 3)).abs().max().item() < 1e-10, b
    del cls, g
    Ec, Gc, Hc = eng.evaluate(Coao, one, two, kappa=kap, path="class")
    Ef, Gf, Hf = eng.evaluate(Coao, one, two, kappa=kap, path="full")
    assert (Ec - Ef).abs().max().item() < TOL_E
    assert (Gc - Gf).abs().max().item() < TOL_GH and (Hc - Hf).abs().max().item() < TOL_GH
    ref = class_oracle.ClassProblem(mol.int1e_ao, mol.int2e_ao, mol.oao_coeff, mol.random_oao_mo_coeff, mol.nuc,
                                    nelec, ncas, nelecas, False)
    for b in range(3):
        Eo, Go, Ho = ref.evaluate(one, two, kap[b])
        assert abs(Ec[b].item() - Eo.item()) < TOL_E, b
        assert (Gc[b].cpu() - Go).abs().max().item() < TOL_GH, b
        assert (Hc[b].cpu() - Ho).abs().max().item() < TOL_GH, b
    prob = orc.OracleProblem(mol.int1e_ao, mol.int2e_ao, mol.oao_coeff, mol.random_oao_mo_coeff, mol.nuc,
                             nelec, ncas, nelecas, False)
    assert abs(Ec[0].item() - prob.energy(one, two, kap[0]).item()) < TOL_E
    assert (Gc[0].cpu() - prob.gradient(one, two, kap[0])).abs().max().item() < TOL_GH


def test_hessian_operand_reuse_follows_the_rdms():
    """A kappa sweep at fixed RDMs reuses the RDM-only operands of the class Hessian (sparse table, C-block
    coefficients, pair runs) left in the workspace; new RDM tensors, or an in-place write into the same ones, rebuild
    them -- and a CUDA-graph replay never skips them."""
    c = load_case("n28_cas66")
    eng, p = engine_for(c)
    Coao = eng.to_padded(c.oao_mo_coeff, 2)
    d1, d2 = eng.dev(c.one_rdm), eng.dev(c.two_rdm)
    kap = torch.stack([c.kappa, 0.5 * c.kappa, -c.kappa]).cuda()
    n0 = eng.lib.oo_launch_count()
    _, _, H0 = eng.evaluate(Coao, d1, d2, kappa=kap[:1])
    n1 = eng.lib.oo_launch_count()
    _, _, H1 = eng.evaluate(Coao, d1, d2, kappa=kap[1:2])                    # same RDM tensors: fewer launches
    n2 = eng.lib.oo_launch_count()
    assert n2 - n1 < n1 - n0
    assert np.abs(H0[0].cpu().numpy() - c.ref["H"]).max() < TOL_GH
    d1b, d2b = (1.1 * d1).contiguous(), (0.9 * d2).contiguous()             # different RDMs
    ref = eng.evaluate(Coao, d1b, d2b, kappa=kap[1:2])[2].clone()
    d1.copy_(d1b)                                                            # in-place write: version counter moves
    d2.copy_(d2b)
    assert torch.equal(eng.evaluate(Coao, d1, d2, kappa=kap[1:2])[2], ref)
    assert not torch.equal(ref, H1)
    for _ in range(3):                                                       # third call replays a captured graph
        Eg, Gg, Hg = eng.evaluate_graphed(Coao, d1b, d2b, kappa=kap[1:2])
    assert torch.equal(Hg, ref)
    E2, G2, H2 = eng.evaluate_graphed(Coao, eng.dev(c.one_rdm), eng.dev(c.two_rdm), kappa=kap[:1])   # replay, new RDM values
    assert np.abs(H2[0].cpu().numpy() - c.ref["H"]).max() < TOL_GH


def test_class_transform_is_reproducible_bit_for_bit():
    """The staged epilogues and bulk-copy pipelines of the class transform hand shared-memory buffers back and forth
    between warps; a buffer overwritten under a pending read would show up as a sporadic difference between
    repetitions of the same transform (tools/transform_stress.py runs the long version)."""
    from auto_oo_b200.engine import HotPathEngine
    from auto_oo_b200.synthetic import SyntheticMol
    from oracle import oo_oracle as orc
    nao, nelec, ncas, nelecas = 114, 42, 6, 6
    mol = SyntheticMol(nao, nelec, seed=3)
    occ, act, virt = mol.get_active_space_idx(ncas, nelecas)
    eng = HotPathEngine(mol.int1e_ao, mol.int2e_ao, mol.oao_coeff, mol.nuc, nao, len(occ), ncas,
                        orc.non_redundant_indices(occ, act, virt, False))
    C = eng.mo_coeff(eng.to_padded(mol.random_oao_mo_coeff, 2))
    ref = eng.class_integrals(C).clone()
    out = torch.empty_like(ref)
    for _ in range(60):
        eng.class_integrals(C, out=out)
        assert torch.equal(out, ref)
    eng.flags = _lib.OO_FLAG_CLASS_DIRECT_STORES
    try:
        direct = eng.class_integrals(C)
    finally:
        eng.flags = 0
    assert (direct - ref).abs().max().item() <= 1e-12 * ref.abs().max().item()
