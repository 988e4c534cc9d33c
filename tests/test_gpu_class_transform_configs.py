"""The symmetric class transform (``oo_class_transform_sym_f64`` and its slab form) at every tile configuration its
host dispatch can pick, called through the C ABI with hand-built inputs and compared with a float64 CPU reference.

Which kernels run depends on ``nIp`` (the class index count, even), the batch and the flags: the quarter-1 tile
(16 / 24 / 32 / 40 / 48 / 64 / wider columns, and 36 .. 48 or 84 .. 96 columns when two evaluations that share the
integrals go through one GEMM), the triangular quarter 2 (``nIp`` 18 .. 48, four configurations) or the rectangular
one, the slab route of the sharded evaluation and, at ``ld = 256``, the Coulomb quarter 4 that computes only the
lower half of each symmetric block.  The sweep below reaches each of them at small sizes; one test asserts with
``torch.profiler`` that it does.

References: ``oracle.class_oracle.class_integrals`` (plain CPU torch, pinned on the verbatim reference) on random
8-fold symmetric integrals, and at ``ld = 256`` an exact closed form for low-rank integrals ``g = 0.3 B B^T``.
Class buffers sit inside a larger allocation filled with a bit pattern, and the workspace is filled with NaN before
every unsharded call (the slab calls share one workspace, as in a sharded evaluation): every K and J element must be
written and right, the zero padding exact, the h' row and the guard zones untouched."""
import re

import numpy as np
import pytest
import torch

from auto_oo_b200 import _lib
from auto_oo_b200.distributed import pair_slab_range
from oracle import class_oracle

F64 = torch.float64
SENTINEL = float.fromhex("-0x1.deadbeef00000p+700")
PAD = 4096                                  # guard doubles on each side of the class buffers
REL_TOL = 1e-12                             # per element, relative to max |reference|
E8 = _lib.OO_FLAG_CLASS_ERI_8FOLD
OO_ERR_INVALID_ARG = -1

# basis size -> class index counts.  Quarter 1 alone: 2 8 16 -> 16 columns, 18 .. 24 -> 24, 26 32 -> 32, 34 40 -> 40,
# 42 .. 48 -> 48, 50 64 -> 64, 66 -> 128; two evaluations in one GEMM: 18 20 -> 40, 22 24 -> 48, 42 44 -> 88,
# 46 48 -> 96.  Triangular quarter 2: 18 .. 24, 26 .. 32, 34 .. 40, 42 .. 48; rectangular below 18 and above 48.
SWEEP = {67: (2, 16, 20, 24, 32, 40, 44, 48, 64, 66), 58: (8, 18, 22, 26, 34, 42, 46, 50)}
SWEEP_POINTS = [(N, nIp) for N, nIps in SWEEP.items() for nIp in nIps]


def _stream():
    return torch.cuda.current_stream().cuda_stream


def tri_index(ld):
    """(ld, ld) packed pair index: T[p, q] = max(p,q) (max(p,q) + 1) / 2 + min(p,q), the order of np.tril_indices."""
    i = torch.arange(ld)
    hi, lo = torch.maximum(i[:, None], i[None, :]), torch.minimum(i[:, None], i[None, :])
    return hi * (hi + 1) // 2 + lo


def pair_ld(ld):
    n = ld * (ld + 1) // 2
    return n + (n & 1)


def random_eri_8fold(N, ld, gen):
    """(g8, g): random 8-fold packed integrals g8[RS][PQ] (npair x pair_ld(ld); symmetric in RS <-> PQ, zero for pairs
    with the padding orbital and in the padding column) and the ld^4 tensor g[p,q,r,s] = g8[RS(r,s)][PQ(p,q)]."""
    npair = ld * (ld + 1) // 2
    T = tri_index(ld)
    live = torch.zeros(npair, dtype=F64)
    live[T[:N, :N].reshape(-1)] = 1.0
    A = torch.randn(npair, npair, dtype=F64, generator=gen)
    A = 0.5 * (A + A.T) * live[:, None] * live[None, :]
    g8 = torch.zeros(npair, pair_ld(ld), dtype=F64)
    g8[:, :npair] = A
    flat = T.reshape(-1)
    return g8, A[flat][:, flat].reshape(ld, ld, ld, ld)


def random_coefficients(N, ld, gen):
    """non-orthogonal N x N coefficients in an ld x ld zero-padded matrix"""
    C = torch.zeros(ld, ld, dtype=F64)
    C[:N, :N] = torch.randn(N, N, dtype=F64, generator=gen) / np.sqrt(N) + torch.eye(N, dtype=F64)
    return C


def low_rank_reference(B, C, nIp):
    """(K, J) of g[p,q,r,s] = 0.3 sum_P B[p,q,P] B[r,s,P] in O(R N^3): with M_P = C^T B_P C,
    J[m,n,a,b] = 0.3 sum_P M_P[a,b] M_P[m,n] and K[n,m,a,b] = g'[a,m,n,b] = 0.3 sum_P M_P[a,m] M_P[n,b]."""
    R, ld = B.shape[2], C.shape[0]
    M = C.T @ B.permute(2, 0, 1) @ C                                    # (R, ld, ld)
    J = 0.3 * (M[:, :nIp, :nIp].reshape(R, -1).T @ M.reshape(R, -1)).reshape(nIp, nIp, ld, ld)
    K = 0.3 * torch.einsum('Pam,Pnb->nmab', M[:, :, :nIp], M[:, :nIp, :])
    return K, J


def workspace(lib, N, ld, nIp, batch):
    nbytes = lib.oo_workspace_bytes(_lib.OO_WS_CLASS_TRANSFORM_SYM, N, ld, nIp, batch)
    return torch.empty((nbytes + 7) // 8, dtype=F64, device="cuda")


def run_sym(lib, ws, g, strideG, C, N, ld, nIp, batch, flags):
    """One oo_class_transform_sym_f64 call into a guarded class buffer (batch, 2 nIp^2 + 1, ld, ld); NaN workspace."""
    rows = 2 * nIp * nIp + 1
    n = batch * rows * ld * ld
    big = torch.full((n + 2 * PAD,), SENTINEL, dtype=F64, device="cuda")
    cls = big[PAD:PAD + n].view(batch, rows, ld, ld)
    ws.fill_(float("nan"))
    rc = lib.oo_class_transform_sym_f64(g.data_ptr(), strideG, C.data_ptr(), ld * ld if batch > 1 else 0, N, ld, nIp,
                                        batch, cls.data_ptr(), ws.data_ptr(), ws.numel() * 8, flags, _stream())
    assert rc == 0, (N, nIp, batch, flags, rc)
    assert bool((big[:PAD] == SENTINEL).all()) and bool((big[-PAD:] == SENTINEL).all()), "guard zone written"
    assert bool((cls[:, -1] == SENTINEL).all()), "h' row written"
    return cls


def check_classes(cls_b, ref, N, nIp, what):
    """K and J rows of one class buffer against the reference (K, J) (indices >= nIp of the reference ignored)."""
    ld, nI2 = cls_b.shape[-1], nIp * nIp
    for name, got, want in (("K", cls_b[:nI2], ref[0][:nIp, :nIp]), ("J", cls_b[nI2:2 * nI2], ref[1][:nIp, :nIp])):
        got = got.reshape(nIp, nIp, ld, ld)
        assert bool(torch.isfinite(got).all()), (what, name, "not every element written")
        scale = want.abs().max().item()
        err = (got - want).abs().max().item()
        assert err <= REL_TOL * scale, (what, name, err, scale)
        if ld > N:                                          # padding orbital: exactly zero
            assert got[:, :, N:].abs().max().item() == 0.0 and got[:, :, :, N:].abs().max().item() == 0.0, (what, name)


class Group:
    """Inputs and references of one basis size: integrals g (shared) and gb (a second geometry), three coefficient
    matrices, and the reference classes of (g, C0), (g, C1), (g, C2), (gb, C1) at the largest nIp of the sweep
    (J and K at m, n < nIp read only the first nIp columns of C, so smaller nIp are slices)."""

    def __init__(self, lib, N, nmax):
        self.N, self.ld = N, N + (N & 1)
        ld = self.ld
        gen = torch.Generator().manual_seed(1000 + N)
        g8, g = random_eri_8fold(N, ld, gen)
        g8b, gb = random_eri_8fold(N, ld, gen)
        C = torch.stack([random_coefficients(N, ld, gen) for _ in range(3)])
        zero_h = torch.zeros(ld, ld, dtype=F64)
        self.ref = {}
        for key, (gg, Cb) in {(0, 0): (g, C[0]), (0, 1): (g, C[1]), (0, 2): (g, C[2]), (1, 1): (gb, C[1])}.items():
            _, J, K = class_oracle.class_integrals(zero_h, gg, Cb, nmax)
            self.ref[key] = (K.cuda(), J.cuda())
        self.g8 = g8.cuda()
        self.g8s = torch.stack([g8, g8b]).cuda()               # per-geometry integrals (strideG != 0)
        self.C = C.cuda()
        gd = g.cuda()                                           # pair-packed form g[r, s, (p >= q)], by the library
        self.gpairs = torch.empty(ld, ld, pair_ld(ld), dtype=F64, device="cuda")
        assert lib.oo_pack_eri_pairs_f64(gd.data_ptr(), self.gpairs.data_ptr(), ld, _stream()) == 0
        del gd
        self.ws = workspace(lib, N, ld, nmax, 3)

    def run(self, lib, nIp, batch, flags=E8, g=None, strideG=0):
        return run_sym(lib, self.ws, self.g8 if g is None else g, strideG, self.C, self.N, self.ld, nIp, batch, flags)


@pytest.fixture(scope="module")
def lib():
    return _lib.load()


class Groups(dict):
    """the Group of each basis size of the sweep, built on first use"""

    def __init__(self, lib):
        super().__init__()
        self.lib = lib

    def __missing__(self, N):
        self[N] = Group(self.lib, N, max(SWEEP[N]))
        return self[N]


@pytest.fixture(scope="module")
def groups(lib):
    gs = Groups(lib)
    yield gs
    gs.clear()
    torch.cuda.empty_cache()


# ------------------------------------------------------------------ 1. every configuration against the reference
@pytest.mark.gpu
@pytest.mark.parametrize("N,nIp", SWEEP_POINTS)
def test_class_transform_sym_against_float64_reference(lib, groups, N, nIp):
    grp = groups[N]
    ref = grp.ref
    c1 = grp.run(lib, nIp, 1)
    check_classes(c1[0], ref[0, 0], N, nIp, "batch 1")
    c2 = grp.run(lib, nIp, 2)                        # one pair (where the class range allows)
    for b in range(2):
        check_classes(c2[b], ref[0, b], N, nIp, f"batch 2 member {b}")
    c3 = grp.run(lib, nIp, 3)                        # a pair and an odd single
    for b in range(3):
        check_classes(c3[b], ref[0, b], N, nIp, f"batch 3 member {b}")
    cg = grp.run(lib, nIp, 2, g=grp.g8s, strideG=grp.g8s[0].numel())    # integrals per geometry: never paired
    check_classes(cg[0], ref[0, 0], N, nIp, "per-geometry member 0")
    check_classes(cg[1], ref[1, 1], N, nIp, "per-geometry member 1")
    scale = c3[:, :-1].abs().max().item()
    for flag, bitwise in ((_lib.OO_FLAG_CLASS_Q1_UNPAIRED, True),      # same k order per element
                          (_lib.OO_FLAG_CLASS_Q2_RECTANGULAR, True),
                          (_lib.OO_FLAG_CLASS_DIRECT_STORES, False),
                          (_lib.OO_FLAG_CLASS_UNFUSED_PACK, False)):
        cv = grp.run(lib, nIp, 3, flags=E8 | flag)
        for b in range(3):
            check_classes(cv[b], ref[0, b], N, nIp, f"flag {flag} member {b}")
        if bitwise:
            assert torch.equal(cv, c3), flag
        else:
            assert (cv[:, :-1] - c3[:, :-1]).abs().max().item() <= REL_TOL * scale, flag
    cp = grp.run(lib, nIp, 3, flags=0, g=grp.gpairs)                    # one pair packed instead of both
    for b in range(3):
        check_classes(cp[b], ref[0, b], N, nIp, f"pair-packed member {b}")


# ------------------------------------------------------------------ 2. the slab route on one device
def slab_cuts(ldp):
    """balanced cuts for 2, 3 and 5 ranks, and a ragged one: a 2-column slab, a 50-column slab (narrower than one
    128-row tile), boundaries that are not multiples of 16"""
    cuts = [[pair_slab_range(ldp, w, r) for r in range(w)] for w in (2, 3, 5)]
    x, y = 16 * (ldp // 40) + 10, 16 * (ldp // 20) + 6
    cuts.append([(0, 2), (2, 52), (52, x), (x, y), (y, ldp)])
    for c in cuts:
        assert c[0][0] == 0 and c[-1][1] == ldp and all(a[1] == b[0] for a, b in zip(c, c[1:]))
        assert all(lo % 2 == 0 and hi % 2 == 0 and hi > lo for lo, hi in c)
    return cuts


@pytest.mark.gpu
@pytest.mark.parametrize("N,nIp", [(67, 16), (58, 26), (58, 46), (67, 64)])
def test_slab_shares_sum_to_the_unsharded_transform(lib, groups, N, nIp):
    """oo_class_transform_sym_slab_f64 once per slab of pair columns, each slab a contiguous copy, ONE workspace for
    all calls (as the engine uses it): the shares sum to the unsharded class buffer and to the reference."""
    grp = groups[N]
    ld, ws, nI2 = grp.ld, grp.ws, nIp * nIp
    ldp = grp.g8.shape[1]
    for batch in (1, 2):
        full = grp.run(lib, nIp, batch)[:, :-1]
        scale = full.abs().max().item()
        ws.fill_(float("nan"))
        cls = torch.empty(batch, 2 * nI2 + 1, ld, ld, dtype=F64, device="cuda")
        for cuts in slab_cuts(ldp):
            acc = torch.zeros(batch, 2 * nI2, ld, ld, dtype=F64, device="cuda")
            for lo, hi in cuts:
                slab = grp.g8[:, lo:hi].contiguous()
                cls.fill_(SENTINEL)
                rc = lib.oo_class_transform_sym_slab_f64(slab.data_ptr(), hi - lo, lo, hi - lo, grp.C.data_ptr(),
                                                         ld * ld if batch > 1 else 0, N, ld, nIp, batch,
                                                         cls.data_ptr(), ws.data_ptr(), ws.numel() * 8, 0, _stream())
                assert rc == 0, (cuts, lo, hi)
                assert bool((cls[:, -1] == SENTINEL).all()), "h' row written"
                assert not bool((cls[:, :-1] == SENTINEL).any()), ("share not written everywhere", lo, hi)
                acc += cls[:, :-1]
            err = (acc - full).abs().max().item()
            assert err <= REL_TOL * scale, (batch, cuts, err, scale)
            for b in range(batch):
                check_classes(acc[b], grp.ref[0, b], N, nIp, f"slabs {cuts} member {b}")
    # documented refusals: the unfused packing passes and the per-stage runs have no slab form
    slab = grp.g8[:, :ldp // 2].contiguous()
    for flags in (_lib.OO_FLAG_CLASS_UNFUSED_PACK, _lib.OO_FLAG_CLASS_STAGE(0), _lib.OO_FLAG_CLASS_STAGE(3),
                  _lib.OO_FLAG_CLASS_STAGE(6)):
        rc = lib.oo_class_transform_sym_slab_f64(slab.data_ptr(), ldp // 2, 0, ldp // 2, grp.C.data_ptr(), 0, N, ld,
                                                 nIp, 1, cls.data_ptr(), ws.data_ptr(), ws.numel() * 8, flags,
                                                 _stream())
        assert rc == OO_ERR_INVALID_ARG, flags


# ------------------------------------------------------------------ 3. ld = 256: the symmetric-block Coulomb quarter 4
def test_low_rank_reference_equals_the_class_oracle():
    """the closed form used at ld = 256 against class_oracle.class_integrals on the full tensor (odd N, padded)"""
    N, ld, R = 9, 10, 5
    gen = torch.Generator().manual_seed(5)
    B = torch.zeros(ld, ld, R, dtype=F64)
    b = torch.randn(N, N, R, dtype=F64, generator=gen)
    B[:N, :N] = 0.5 * (b + b.transpose(0, 1))
    C = random_coefficients(N, ld, gen)
    g = 0.3 * torch.einsum('pqP,rsP->pqrs', B, B)
    for nIp in (2, 4, ld):
        _, J, K = class_oracle.class_integrals(torch.zeros(ld, ld, dtype=F64), g, C, nIp)
        Kr, Jr = low_rank_reference(B, C, nIp)
        assert (Kr - K).abs().max().item() <= 1e-13 * K.abs().max().item()
        assert (Jr - J).abs().max().item() <= 1e-13 * J.abs().max().item()
        assert Kr[:, :, N:].abs().max().item() == 0.0 and Jr[:, :, :, N:].abs().max().item() == 0.0


class LowRank:
    """8-fold packed g8 = 0.3 Bp Bp^T at ld = 256 (8.7 GB), formed on the device from the symmetric factor
    B[p,q,P] packed over np.tril_indices(ld) (as SyntheticMol.int2e_packed_slab does): no N^4 tensor anywhere."""

    def __init__(self, N, R=12):
        self.N, self.ld = N, 256
        ld = self.ld
        gen = torch.Generator().manual_seed(N)
        b = torch.randn(N, N, R, dtype=F64, generator=gen)
        self.B = torch.zeros(ld, ld, R, dtype=F64)
        self.B[:N, :N] = 0.5 * (b + b.transpose(0, 1)) / np.sqrt(R)
        self.C = torch.stack([random_coefficients(N, ld, gen) for _ in range(2)])
        rows, cols = np.tril_indices(ld)
        Bp = self.B.cuda()[torch.as_tensor(rows, device="cuda"), torch.as_tensor(cols, device="cuda")]
        npair = len(rows)
        self.g8 = torch.zeros(npair, pair_ld(ld), dtype=F64, device="cuda")
        for i in range(0, npair, 4096):
            self.g8[i:i + 4096, :npair] = torch.matmul(Bp[i:i + 4096], Bp.T).mul_(0.3)
        del Bp


@pytest.fixture(scope="module", params=[255, 256])
def low_rank(request):
    lr = LowRank(request.param)
    yield lr
    del lr.g8
    torch.cuda.empty_cache()


@pytest.mark.gpu
@pytest.mark.parametrize("nIp", [4, 18])
def test_symmetric_block_coulomb_quarter_four_at_ld_256(lib, low_rank, nIp):
    """ld % 128 == 0 and ld >= 256: the staged Coulomb quarter 4 computes the tiles on and below the diagonal of every
    symmetric 256 x 256 block and mirrors them; the direct stores compute every tile.  Batch 2 (a pair at nIp = 18)."""
    lr = low_rank
    N, ld = lr.N, lr.ld
    refs = [tuple(t.cuda() for t in low_rank_reference(lr.B, lr.C[b], nIp)) for b in range(2)]
    ws = workspace(lib, N, ld, nIp, 2)
    C = lr.C.cuda()
    for flags in (E8, E8 | _lib.OO_FLAG_CLASS_DIRECT_STORES):
        cls = run_sym(lib, ws, lr.g8, 0, C, N, ld, nIp, 2, flags)
        for b in range(2):
            check_classes(cls[b], refs[b], N, nIp, f"flags {flags} member {b}")
        del cls
    del ws
    torch.cuda.empty_cache()


# ------------------------------------------------------------------ 4. coverage is asserted
_Q1_TILES = ["256,16,16,8,1,4,0", "256,32,16,8,1,4,3", "256,32,16,8,1,4,0", "256,48,16,8,1,4,5", "256,48,16,8,1,4,0",
             "256,64,16,4,2,4,0", "128,128,16,2,4,4,0", "128,96,16,8,1,4,11", "128,96,16,8,1,4,0"]
EXPECTED_KERNELS = ([f"dgemm_tn_kernel<TnCfg<{t}>,2,1," for t in _Q1_TILES]          # quarter 1 from g8 (AMODE 1)
                    + [f"dgemm_tn_tri_kernel<TriCfg<{c},4>>" for c in ("32,3", "32,4", "48,5", "48,6")]
                    + ["dgemm_tn_kernel<TnCfg<192,64,16,4,2,4,0>,0,"])               # Hessian C block shape


def _kernel_key(name):
    return re.sub(r"\s+", "", re.sub(r"\(anonymous namespace\)::", "", name).replace("oo::", ""))


@pytest.mark.gpu
def test_the_sweep_launches_every_tile_configuration(lib, groups):
    """A subset of the sweep under torch.profiler: every quarter-1 tile (single and paired), every triangular quarter-2
    configuration and the 192-row GEMM tile must actually run.  A dispatch change that moves one out of reach of
    these tests fails here."""
    from torch.profiler import ProfilerActivity, profile
    g58, g67 = groups[58], groups[67]
    M, Nc, K = 176, 9472, 40
    gen = torch.Generator(device="cuda").manual_seed(1)
    At = torch.randn(K, M, dtype=F64, device="cuda", generator=gen)
    Bm = torch.randn(K, Nc, dtype=F64, device="cuda", generator=gen)
    Cm = torch.empty(M, Nc, dtype=F64, device="cuda")
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for nIp in (8, 18, 22, 26, 34, 42, 46, 50):
            g58.run(lib, nIp, 3)
        g67.run(lib, 66, 3)
        assert lib.oo_dgemm_tn_f64(At.data_ptr(), Bm.data_ptr(), Cm.data_ptr(), M, Nc, K, M, Nc, Nc, 1, 0, 0, 0,
                                   _stream()) == 0
        torch.cuda.synchronize()
    names = {_kernel_key(e.name) for e in prof.events()}
    missing = [k for k in EXPECTED_KERNELS if not any(k in n for n in names)]
    assert not missing, (missing, sorted(n for n in names if "dgemm" in n))
    assert (Cm.cpu() - At.T.cpu() @ Bm.cpu()).abs().max().item() < 1e-12 * K * 10
