"""The orbital Hessian (``oo_class_hessian_f64``, ``oo_hessian_f64``) and its matrix-free operator (the Hessian-vector
product and the diagonal, class-buffer and (h', g') forms) at every route their host dispatch can pick, called through
the C ABI with hand-built inputs and compared with a float64 reference written out from the definition.

What runs depends on (no, na), ld, the batch, the flags and the pair list:
  * the G blocks of the T-matrix: ``hess_group_kernel<8|16|24>`` (passes of CH result columns: two passes at na > 12)
    below ld^2 = 4096 or with more than 24 G-block columns, ``hess_group_stream_kernel<1|2|3>`` above (256-column
    tiles, ragged when ld^2 mod 256 != 0, CTAs whose item range crosses from one occupied orbital to the next);
  * the occ-occ remainder: ``hess_spmm_pair_kernel`` (no >= 2) and ``hess_spmm_kernel``, with shared or per-evaluation
    RDMs in a batch;
  * the assembly: one thread per element (N <= 64), the row-tiled kernel (its strip, its per-thread form for unsorted
    lists and for strips over 2080 entries, i.e. nI > 64) and the streamed kernel for the rows outside I (uniform
    pair lists only; partial last row tile);
  * the product: ``nvc`` vectors per pass (8 up to nI = 25, 7 at 26, 3 at 66), ragged last passes, ld mod 32 != 0.
The shapes below reach each of these at small sizes; one test asserts with ``torch.profiler`` that they launch.

Inputs: low-rank 8-fold-symmetric MO integrals g'[a,b,c,d] = sum_P w_P M_P[a,b] M_P[c,d] (zero beyond N), a symmetric
h', a non-symmetric F (the kernels read it only through F + F^T and F_ac) and the RDMs of ``random_rdms``, which have
the symmetries the formulas assume.  Outputs sit inside a sentinel-filled allocation and are NaN-filled before every
call, as is the workspace: every element must be written and finite, the guard zones untouched.

Reference (shares no code with ``auto_oo_b200``), for an ARBITRARY pair list (l_j, r_j):
  T[(p r),(q s)] = 2 sum_mn (G_pmrn + G_pmnr) g'[q,m,n,s] + 2 sum_mn G_prmn g'[q,s,m,n] + 2 gamma_pr h'_qs,
  X(a,b,c,d)     = -(F_ac + F_ca) delta_bd + [a, c in I] T[(a c),(b d)],
  H[j,k]         = X(l_j,r_j,l_k,r_k) - X(l_j,r_j,r_k,l_k) - X(r_j,l_j,l_k,r_k) + X(r_j,l_j,r_k,l_k),
with gamma, G the full-space RDMs of ``oracle.oo_oracle.full_rdms``; H V and diag(H) are taken from it.  The large
contractions run as float64 matmuls (cuBLAS, independent of this library).  ``tests/test_hessian_operator_cpu.py``
pins this reference on the class oracle, the golden Hessians and ``oo_oracle.hessian_full``."""
import re

import numpy as np
import pytest
import torch

from auto_oo_b200 import _lib
from auto_oo_b200.synthetic import random_rdms
from oracle import oo_oracle as orc

F64 = torch.float64
SENTINEL = float.fromhex("-0x1.deadbeef00000p+700")
PAD = 4096                                  # guard doubles on each side of every output
REL_TOL = 1e-12                             # per element, relative to max |reference| of the call
RANK = 8                                    # terms of the low-rank integrals

# (N, ld, no, na): what each shape reaches
SHAPES = {
    (40, 40, 5, 3): "hess_group_kernel<8>, per-element assembly, pair spmm",
    (40, 40, 4, 7): "hess_group_kernel<16>, odd nI",
    (40, 40, 3, 10): "hess_group_kernel<24>, one pass",
    (40, 40, 2, 13): "hess_group_kernel<24>, two passes (26 columns)",
    # (the G-block coefficients are the same for every occupied orbital, so a CTA that spans two is checked through its
    #  per-orbital row offsets and output rows, not through its coefficient reload)
    (66, 68, 9, 3): "hess_group_stream_kernel<1>: 19 tiles per orbital, the last one ragged (68^2 = 18 * 256 + 16); "
                    "171 items on at most 148 SMs = 2 per CTA, so CTA 9 spans orbitals 0 and 1; streamed assembly "
                    "with a partial last row tile and ld > N",
    (66, 66, 1, 6): "hess_group_stream_kernel<2>, no = 1 (no pair kernel), nI = 7 -> rows_in = 8",
    (66, 72, 2, 12): "hess_group_stream_kernel<3>, padding columns ld > N",
    (66, 66, 0, 5): "no occupied orbitals: no G blocks, no pair kernel",
    (66, 66, 2, 13): "na > 12 at ld >= 64: hess_group_kernel<24>, two passes",
    (130, 130, 20, 6): "several streamed row tiles, nvc = 7",
    (129, 130, 60, 6): "nI = 66 > 64: strip overflow -> per-thread row tiles, no streamed assembly, nvc = 3, "
                       "ragged last row tile",
}
SHAPE_IDS = [f"N{N}-ld{ld}-no{no}-na{na}" for N, ld, no, na in SHAPES]
SMALL, STREAMED = (40, 40, 5, 3), (66, 68, 9, 3)      # one shape below and one above ld = 64


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _ptr(t):
    return 0 if t is None else t.data_ptr()


# ------------------------------------------------------------------ reference
def t_reference(h, J, K, one, two, no, na):
    """T[p, r, q, s] = T[(p r),(q s)] for p, r in I (nI, nI, ld, ld).  J[m,n,a,b] = g'[a,b,m,n] and
    K[n,m,a,b] = g'[a,m,n,b] for m, n in I (nI, nI, ld, ld); h' (ld, ld); active-space RDMs."""
    nI, ld = no + na, h.shape[0]
    dev = h.device
    d1, d2 = orc.full_rdms(one.cpu(), two.cpu(), nI, np.arange(no), np.arange(no, nI))
    d1, d2 = d1.to(dev), d2.to(dev)
    a1 = (d2.permute(0, 2, 1, 3) + d2.permute(0, 3, 1, 2)).reshape(nI * nI, nI * nI)     # [(p r),(m n)] G_pmrn + G_pmnr
    a2 = d2.reshape(nI * nI, nI * nI)                                                    # [(p r),(m n)] G_prmn
    kc = K.permute(1, 0, 2, 3).reshape(nI * nI, ld * ld)                                 # [(m n),(q s)] g'[q,m,n,s]
    jc = J.reshape(nI * nI, ld * ld)                                                     # [(m n),(q s)] g'[q,s,m,n]
    t = 2.0 * (a1 @ kc + a2 @ jc) + 2.0 * torch.outer(d1.reshape(-1), h.reshape(-1))
    return t.reshape(nI, nI, ld, ld)


def hessian_reference(T, F, nI, L, R, rows=None):
    """H[j, k] for the pair list (L, R) (any order, any pairs), rows j of `rows` (default all)."""
    fs = F + F.T
    L = torch.as_tensor(L, dtype=torch.long, device=T.device)
    R = torch.as_tensor(R, dtype=torch.long, device=T.device)
    Lj, Rj = (L, R) if rows is None else (L[rows], R[rows])

    def x(a, b, c, d):                              # a, b: (nj, 1) row indices; c, d: (1, nk) column indices
        out = -fs[a, c] * (b == d).to(F64)
        inside = (a < nI) & (c < nI)
        t = T[a.clamp(max=nI - 1), c.clamp(max=nI - 1), b, d]
        return out + torch.where(inside, t, torch.zeros_like(t))

    a, b = Lj[:, None], Rj[:, None]
    c, d = L[None, :], R[None, :]
    return x(a, b, c, d) - x(a, b, d, c) - x(b, a, c, d) + x(b, a, d, c)


# ------------------------------------------------------------------ inputs
def low_rank_factors(N, ld, seed, R=RANK):
    """(M, w): symmetric random M_P (zero beyond N) and unequal weights w_P"""
    gen = torch.Generator().manual_seed(seed)
    m = torch.randn(R, N, N, dtype=F64, generator=gen) / np.sqrt(N)
    M = torch.zeros(R, ld, ld, dtype=F64)
    M[:, :N, :N] = m + m.transpose(1, 2)
    w = 0.25 + torch.rand(R, dtype=F64, generator=gen)
    return M, w


def classes_from_factors(M, w, nI):
    """(J, K) over m, n < nI: J[m,n,a,b] = sum w M[a,b] M[m,n], K[n,m,a,b] = sum w M[a,m] M[n,b]"""
    R, ld = M.shape[0], M.shape[1]
    J = ((M[:, :nI, :nI].reshape(R, -1).T * w) @ M.reshape(R, -1)).reshape(nI, nI, ld, ld)
    K = torch.einsum('P,Pam,Pnb->nmab', w, M[:, :, :nI], M[:, :nI, :])
    return J, K


def class_buffer(h, J, K, nIp):
    """[K rows (n, m) (nIp^2); J rows (m, n) (nIp^2); h' row], rows with m or n >= nI zero"""
    nI, ld = J.shape[0], h.shape[0]
    Kp = torch.zeros(nIp, nIp, ld, ld, dtype=F64, device=h.device)
    Jp = torch.zeros_like(Kp)
    Kp[:nI, :nI], Jp[:nI, :nI] = K, J
    return torch.cat([Kp.reshape(nIp * nIp, ld, ld), Jp.reshape(nIp * nIp, ld, ld), h[None]]).contiguous()


class Evaluation:
    """One evaluation: integrals from seed, F, RDMs (given or drawn), its class buffer and reference T."""

    def __init__(self, N, ld, no, na, seed, rdms=None):
        self.N, self.ld, self.no, self.na = N, ld, no, na
        self.nI = no + na
        self.nIp = self.nI + (self.nI & 1)
        M, w = low_rank_factors(N, ld, seed)
        gen = torch.Generator().manual_seed(seed + 1)
        h = torch.zeros(ld, ld, dtype=F64)
        x = torch.randn(N, N, dtype=F64, generator=gen)
        h[:N, :N] = x + x.T
        F = torch.zeros(ld, ld, dtype=F64)
        F[:N, :N] = torch.randn(N, N, dtype=F64, generator=gen)
        self.one, self.two = rdms if rdms is not None else random_rdms(na, min(na, 4), seed=seed)
        self.M, self.w = M.cuda(), w.cuda()
        self.h, self.F = h.cuda(), F.cuda()
        J, K = classes_from_factors(self.M, self.w, self.nI)
        self.cls = class_buffer(self.h, J, K, self.nIp)
        self.T = t_reference(self.h, J, K, self.one, self.two, no, na)
        self.d1, self.d2 = self.one.cuda().contiguous(), self.two.cuda().contiguous()

    def g_full(self):
        """the complete g' (ld^4) on the device"""
        R, ld = self.M.shape[0], self.ld
        Mf = self.M.reshape(R, -1)
        return ((Mf.T * self.w) @ Mf).reshape(ld, ld, ld, ld)

    def hessian(self, L, R):
        return hessian_reference(self.T, self.F, self.nI, L, R)


def engine_pairs(N, no, na, frozen=False):
    """the engine's non-redundant list, np.tril_indices order"""
    rows, cols = orc.tril_pairs(N)
    idx = orc.non_redundant_indices(np.arange(no), np.arange(no, no + na), np.arange(no + na, N), frozen)
    return rows[idx].astype(np.int32), cols[idx].astype(np.int32)


def hvp_vectors_per_pass(nI):
    """vectors per pass of the product (hvp_layout: the largest nvc <= 8 whose shared-memory plan fits 200 KB)"""
    def smem(c):
        ncol = nI * c
        return (4 * 32 * 36 + ncol * 36 + (ncol + 7) // 8 * 8 * 36 + nI * 32 * c) * 8
    return max(c for c in range(1, 9) if smem(c) <= 200 * 1024)


# ------------------------------------------------------------------ calls through the C ABI
def guarded(n):
    """(whole, view): n NaN doubles between two sentinel guard zones"""
    big = torch.full((n + 2 * PAD,), SENTINEL, dtype=F64, device="cuda")
    big[PAD:PAD + n] = float("nan")
    return big, big[PAD:PAD + n]


def check_output(big, out, ref, what):
    torch.cuda.synchronize()
    assert bool((big[:PAD] == SENTINEL).all()) and bool((big[-PAD:] == SENTINEL).all()), (what, "guard zone written")
    assert bool(torch.isfinite(out).all()), (what, "not every element written")
    scale = ref.abs().max().item()
    err = (out.reshape(ref.shape) - ref).abs().max().item()
    assert err <= REL_TOL * scale, (what, err, scale)


def workspace(lib, kind, N, ld, nI, batch):
    nbytes = lib.oo_workspace_bytes(kind, N, ld, nI, batch)
    assert nbytes > 0
    return torch.full(((nbytes + 7) // 8,), float("nan"), dtype=F64, device="cuda")


def dev_pairs(L, R):
    return (torch.as_tensor(np.ascontiguousarray(L), dtype=torch.int32, device="cuda"),
            torch.as_tensor(np.ascontiguousarray(R), dtype=torch.int32, device="cuda"))


def class_hessian(lib, evs, L, R, flags=0, per_eval_rdms=False, ws=None, expect=None, what=""):
    """oo_class_hessian_f64 on the batch `evs` (class buffers and F per member); returns the workspace for a reuse"""
    e0, batch = evs[0], len(evs)
    nk = len(L)
    pl, pr = dev_pairs(L, R)
    cls = torch.stack([e.cls for e in evs]).contiguous()
    F = torch.stack([e.F for e in evs]).contiguous()
    if per_eval_rdms:
        d1 = torch.stack([e.d1 for e in evs]).contiguous()
        d2 = torch.stack([e.d2 for e in evs]).contiguous()
        sd1, sd2 = e0.na ** 2, e0.na ** 4
    else:
        d1, d2, sd1, sd2 = e0.d1, e0.d2, 0, 0
    if ws is None:
        ws = workspace(lib, _lib.OO_WS_CLASS_HESSIAN, e0.na, e0.ld, e0.nI, batch)
    big, H = guarded(batch * nk * nk)
    rc = lib.oo_class_hessian_f64(cls.data_ptr(), F.data_ptr(), d1.data_ptr(), sd1, d2.data_ptr(), sd2, e0.no, e0.na,
                                  e0.N, e0.ld, e0.nIp, batch, pl.data_ptr(), pr.data_ptr(), nk, H.data_ptr(),
                                  ws.data_ptr(), ws.numel() * 8, flags, _stream())
    assert rc == 0, (what, flags, rc)
    H = H.view(batch, nk, nk)
    for b, e in enumerate(evs):
        ref = e.hessian(L, R) if expect is None else expect[b]
        check_output(big, H[b], ref, f"{what} flags {flags} member {b}")
    return ws


def class_hessian_vector(lib, ev, L, R, nv, H_ref, what="", seed=0):
    nk = len(L)
    pl, pr = dev_pairs(L, R)
    V = torch.randn(nk, nv, dtype=F64, device="cuda", generator=torch.Generator(device="cuda").manual_seed(seed))
    ws = workspace(lib, _lib.OO_WS_CLASS_HESSIAN_VECTOR, ev.na, ev.ld, ev.nI, nv)
    big, HV = guarded(nk * nv)
    rc = lib.oo_class_hessian_vector_f64(ev.cls.data_ptr(), ev.F.data_ptr(), ev.d1.data_ptr(), ev.d2.data_ptr(),
                                         ev.no, ev.na, ev.N, ev.ld, ev.nIp, pl.data_ptr(), pr.data_ptr(), nk,
                                         V.data_ptr(), nv, HV.data_ptr(), ws.data_ptr(), ws.numel() * 8, _stream())
    assert rc == 0, (what, nv, rc)
    check_output(big, HV, H_ref @ V, f"{what} H V, nv = {nv}")


def class_hessian_diagonal(lib, ev, L, R, H_ref, what=""):
    nk = len(L)
    pl, pr = dev_pairs(L, R)
    big, diag = guarded(nk)
    rc = lib.oo_class_hessian_diagonal_f64(ev.cls.data_ptr(), ev.F.data_ptr(), ev.d1.data_ptr(), ev.d2.data_ptr(),
                                           ev.no, ev.na, ev.N, ev.ld, ev.nIp, pl.data_ptr(), pr.data_ptr(), nk,
                                           diag.data_ptr(), 0, 0, _stream())
    assert rc == 0, (what, rc)
    check_output(big, diag, H_ref.diagonal(), f"{what} diagonal")


@pytest.fixture(scope="module")
def lib():
    return _lib.load()


class Evaluations(dict):
    """the Evaluation of each shape (seeded by its position), built on first use"""

    def __missing__(self, shape):
        N, ld, no, na = shape
        self[shape] = Evaluation(N, ld, no, na, seed=100 + list(SHAPES).index(shape))
        return self[shape]


@pytest.fixture(scope="module")
def evals():
    ev = Evaluations()
    yield ev
    ev.clear()
    torch.cuda.empty_cache()


# ------------------------------------------------------------------ 1. every shape, the engine's list
@pytest.mark.gpu
@pytest.mark.parametrize("shape", list(SHAPES), ids=SHAPE_IDS)
def test_class_hessian_product_and_diagonal_against_float64_reference(lib, evals, shape):
    ev = evals[shape]
    L, R = engine_pairs(ev.N, ev.no, ev.na)
    H_ref = ev.hessian(L, R)
    class_hessian(lib, [ev], L, R, what=SHAPES[shape])
    nvc = hvp_vectors_per_pass(ev.nI)
    for nv in (1, nvc, nvc + 1, 2 * nvc + 1):
        class_hessian_vector(lib, ev, L, R, nv, H_ref, what=SHAPES[shape], seed=nv)
    class_hessian_diagonal(lib, ev, L, R, H_ref, what=SHAPES[shape])


def test_vectors_per_pass_of_the_product():
    """the pass widths the shapes above rely on (and the ones hvp_layout documents)"""
    assert [hvp_vectors_per_pass(n) for n in (8, 15, 25, 26, 32, 40, 53, 66, 70, 101)] == [8, 8, 8, 7, 6, 5, 3, 3, 2, 1]


# ------------------------------------------------------------------ 2. the (h', g') forms: the gathered class layout
@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(40, 40, 4, 7), (40, 40, 5, 3)], ids=["odd-nI", "even-nI"])
def test_full_tensor_forms_against_float64_reference(lib, evals, shape):
    """oo_hessian_f64, oo_hessian_vector_f64 and oo_hessian_diagonal_f64 gather the class layout out of the complete
    g' (at odd nI with the zero row and column nI of the padded class index)"""
    ev = evals[shape]
    L, R = engine_pairs(ev.N, ev.no, ev.na)
    nk = len(L)
    pl, pr = dev_pairs(L, R)
    H_ref = ev.hessian(L, R)
    g = ev.g_full()
    ws = workspace(lib, _lib.OO_WS_HESSIAN, ev.N, ev.ld, ev.nI, 1)
    big, H = guarded(nk * nk)
    rc = lib.oo_hessian_f64(ev.h.data_ptr(), g.data_ptr(), ev.F.data_ptr(), ev.d1.data_ptr(), ev.d2.data_ptr(), ev.no,
                            ev.na, ev.N, ev.ld, pl.data_ptr(), pr.data_ptr(), nk, H.data_ptr(), ws.data_ptr(),
                            ws.numel() * 8, 0, _stream())
    assert rc == 0
    check_output(big, H, H_ref, "oo_hessian_f64")
    for nv in (1, 9):
        V = torch.randn(nk, nv, dtype=F64, device="cuda", generator=torch.Generator(device="cuda").manual_seed(nv))
        ws = workspace(lib, _lib.OO_WS_HESSIAN_VECTOR, ev.na, ev.ld, ev.nI, nv)
        big, HV = guarded(nk * nv)
        rc = lib.oo_hessian_vector_f64(ev.h.data_ptr(), g.data_ptr(), ev.F.data_ptr(), ev.d1.data_ptr(),
                                       ev.d2.data_ptr(), ev.no, ev.na, ev.N, ev.ld, pl.data_ptr(), pr.data_ptr(), nk,
                                       V.data_ptr(), nv, HV.data_ptr(), ws.data_ptr(), ws.numel() * 8, _stream())
        assert rc == 0
        check_output(big, HV, H_ref @ V, f"oo_hessian_vector_f64 nv = {nv}")
    ws = workspace(lib, _lib.OO_WS_HESSIAN_DIAGONAL, ev.N, ev.ld, ev.nI, 1)
    big, diag = guarded(nk)
    rc = lib.oo_hessian_diagonal_f64(ev.h.data_ptr(), g.data_ptr(), ev.F.data_ptr(), ev.d1.data_ptr(),
                                     ev.d2.data_ptr(), ev.no, ev.na, ev.N, ev.ld, pl.data_ptr(), pr.data_ptr(), nk,
                                     diag.data_ptr(), ws.data_ptr(), ws.numel() * 8, _stream())
    assert rc == 0
    check_output(big, diag, H_ref.diagonal(), "oo_hessian_diagonal_f64")


# ------------------------------------------------------------------ 3. every Hessian flag
FLAGS = [_lib.OO_FLAG_HESSIAN_DENSE, _lib.OO_FLAG_HESSIAN_ASSEMBLE_PER_ELEMENT, _lib.OO_FLAG_HESSIAN_ASSEMBLE_TILED,
         _lib.OO_FLAG_HESSIAN_ASSEMBLE_UNSTREAMED, _lib.OO_FLAG_HESSIAN_GROUP_UNSTREAMED,
         _lib.OO_FLAG_HESSIAN_SPMM_UNPAIRED]


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [SMALL, STREAMED], ids=["ld40", "ld68"])
@pytest.mark.parametrize("flag", FLAGS)
def test_every_hessian_flag_against_float64_reference(lib, evals, shape, flag):
    """each A/B route on its own (ASSEMBLE_TILED at N <= 64 forces the row-tiled and streamed assembly there)"""
    ev = evals[shape]
    L, R = engine_pairs(ev.N, ev.no, ev.na)
    class_hessian(lib, [ev], L, R, flags=flag, what=SHAPES[shape])


# ------------------------------------------------------------------ 4. batches: class buffers, F and RDMs per member
@pytest.mark.gpu
@pytest.mark.parametrize("shape", [SMALL, STREAMED], ids=["ld40", "ld68"])
@pytest.mark.parametrize("per_eval_rdms", [False, True], ids=["shared-rdms", "rdms-per-evaluation"])
def test_batch_of_three_and_operand_reuse(lib, shape, per_eval_rdms):
    """batch 3 with a class buffer and F per member and the RDMs shared (strides 0) or per member; then, with
    OO_FLAG_HESSIAN_REUSE_OPERANDS, new class buffers and F at the same RDMs and pair list.  (The reuse call keeps the
    workspace of the first: the RDM-only operands and the pair runs it holds are what the flag reuses.)
    The occ-occ columns that hess_spmm_pair_kernel forms have RDM-independent coefficients (Kronecker terms of the
    full-space 2-RDM), so which member's sparse table it reads cannot show in the output; the other sparse columns,
    the C block and the G blocks do depend on the member's RDMs."""
    N, ld, no, na = shape
    shared = random_rdms(na, min(na, 4), seed=50)
    evs = [Evaluation(N, ld, no, na, seed=200 + b, rdms=None if per_eval_rdms else shared) for b in range(3)]
    L, R = engine_pairs(N, no, na)
    ws = class_hessian(lib, evs, L, R, per_eval_rdms=per_eval_rdms, what="batch 3")
    again = [Evaluation(N, ld, no, na, seed=300 + b, rdms=(e.one, e.two)) for b, e in enumerate(evs)]
    class_hessian(lib, again, L, R, flags=_lib.OO_FLAG_HESSIAN_REUSE_OPERANDS, per_eval_rdms=per_eval_rdms, ws=ws,
                  what="batch 3, operands reused")


# ------------------------------------------------------------------ 5. pair lists other than the engine's
def _rows(L, R):
    """{l: [r, ...]} of a list"""
    out = {}
    for l, r in zip(L.tolist(), R.tolist()):
        out.setdefault(l, []).append(r)
    return out


def _from_rows(rows):
    L = np.array([l for l in sorted(rows) for _ in rows[l]], dtype=np.int32)
    R = np.array([r for l in sorted(rows) for r in rows[l]], dtype=np.int32)
    return L, R


def pair_lists(N, no, na):
    """name -> (L, R) at one N > 64 shape"""
    nI = no + na
    rng = np.random.default_rng(7)
    L, R = engine_pairs(N, no, na)
    lists = {"frozen-active": engine_pairs(N, no, na, frozen=True)}
    keep = np.sort(rng.choice(len(L), size=len(L) * 3 // 5, replace=False))
    lists["random-subset"] = (L[keep], R[keep])                       # row order, gaps inside rows: unstructured
    perm = rng.permutation(len(L))
    lists["shuffled"] = (L[perm], R[perm])
    rows = _rows(L, R)
    for l, extra in ((nI + 3, 2), (nI + 20, 5), (N - 1, N - 1 - nI)):  # consecutive virt-virt columns nI .. :
        rows[l] = rows[l] + list(range(nI, nI + extra))                  # structured, not uniform
    lists["virt-virt"] = _from_rows(rows)
    # Rows inside I may hold a pair (p, q) with q >= rows_in while the rows outside keep the uniform layout of the
    # streamed assembly (columns 0 .. S-1, S < nI): p >= S keeps every unordered pair unique.  Hessian elements
    # H[(p, q), (q, s)] then need the Fock term of -X(p,q,s,r) at q == r inside the streamed kernel.
    S = nI - 2
    rows = {l: [r for r in cols if r < S] if l >= nI else cols for l, cols in _rows(L, R).items()}
    rows[nI - 2], rows[nI - 1] = [nI + 18], [nI + 8, nI + 9]
    lists["upper-triangle"] = _from_rows(rows)
    return lists


def issue_upper_list(N):
    """nI = 3: (1, 0), (2, 5), then (l, 0), (l, 1) for every l >= 4 -- row-sorted, consecutive columns, the layout
    the streamed assembly accepts, with the pair (2, 5) above the diagonal"""
    L = [1, 2] + [l for l in range(4, N) for _ in (0, 1)]
    R = [0, 5] + [r for _ in range(4, N) for r in (0, 1)]
    return np.array(L, dtype=np.int32), np.array(R, dtype=np.int32)


def _check_list(L, R):
    """what the product and the diagonal require: l != r, every unordered pair at most once"""
    key = np.minimum(L, R).astype(np.int64) * 100000 + np.maximum(L, R)
    assert (L != R).all() and len(np.unique(key)) == len(key)


PAIR_LIST_NAMES = ["frozen-active", "random-subset", "shuffled", "virt-virt", "upper-triangle"]


@pytest.mark.gpu
@pytest.mark.parametrize("name", PAIR_LIST_NAMES)
def test_pair_lists_against_float64_reference(lib, evals, name):
    """the C ABI takes any pair list: hess_pair_runs_kernel picks the structured, unstructured or streamed assembly
    on the device; the product and the diagonal take any list of distinct unordered pairs"""
    ev = evals[STREAMED]
    L, R = pair_lists(ev.N, ev.no, ev.na)[name]
    _check_list(L, R)
    H_ref = ev.hessian(L, R)
    for flags in (0, _lib.OO_FLAG_HESSIAN_ASSEMBLE_UNSTREAMED):
        class_hessian(lib, [ev], L, R, flags=flags, what=name)
    class_hessian_vector(lib, ev, L, R, 3, H_ref, what=name)
    class_hessian_diagonal(lib, ev, L, R, H_ref, what=name)


@pytest.mark.gpu
def test_upper_triangle_pair_in_a_streamed_layout(lib):
    """no = 1, na = 2, N = 66: the list (1,0), (2,5), (l,0), (l,1) for l >= 4 passes the streamed layout check, and
    H[(2,5),(5,s)] holds F_2s + F_s2 from the q == r term of the assembly"""
    ev = Evaluation(66, 66, 1, 2, seed=400)
    L, R = issue_upper_list(ev.N)
    _check_list(L, R)
    H_ref = ev.hessian(L, R)
    assert (L[4:6] == 5).all() and (ev.F[2, :2] + ev.F[:2, 2]).abs().min().item() > 0.0   # k = (5,0), (5,1)
    for flags in (0, _lib.OO_FLAG_HESSIAN_ASSEMBLE_UNSTREAMED, _lib.OO_FLAG_HESSIAN_ASSEMBLE_PER_ELEMENT):
        class_hessian(lib, [ev], L, R, flags=flags, what="upper-triangle nI = 3")
    class_hessian_vector(lib, ev, L, R, 2, H_ref, what="upper-triangle nI = 3")
    class_hessian_diagonal(lib, ev, L, R, H_ref, what="upper-triangle nI = 3")


# ------------------------------------------------------------------ 6. coverage is asserted
EXPECTED_KERNELS = ([f"hess_group_kernel<{c}>" for c in (8, 16, 24)]
                    + [f"hess_group_stream_kernel<{c}>" for c in (1, 2, 3)]
                    + ["hess_spmm_pair_kernel", "hess_spmm_kernel", "hess_assemble_kernel",
                       "hess_assemble_rows_kernel", "hess_assemble_stream_kernel", "hess_diag_kernel"]
                    + [f"hvp_{k}_kernel" for k in ("table", "scatter", "plane", "reduce", "gather")])


def _kernel_key(name):
    return re.sub(r"\s+", "", re.sub(r"\(anonymous namespace\)::", "", name).replace("oo::", ""))


@pytest.mark.gpu
def test_the_shapes_launch_every_hessian_kernel(lib, evals):
    """The routes of the shapes above under torch.profiler: every template instance of the G-block kernels, both
    sparse kernels, all three assembly kernels and the matrix-free kernels must run.  A dispatch change that moves one
    out of reach of these tests fails here.  (The streamed assembly returns at once on a list it cannot take; the
    NaN-filled output of the tests above catches that.)"""
    from torch.profiler import ProfilerActivity, profile
    shapes = [SMALL, (40, 40, 4, 7), (40, 40, 3, 10), STREAMED, (66, 66, 1, 6), (66, 72, 2, 12)]
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for shape in shapes:
            ev = evals[shape]
            L, R = engine_pairs(ev.N, ev.no, ev.na)
            H_ref = ev.hessian(L, R)
            class_hessian(lib, [ev], L, R, what=SHAPES[shape])
        class_hessian_vector(lib, ev, L, R, 2, H_ref, what=SHAPES[shape])
        class_hessian_diagonal(lib, ev, L, R, H_ref, what=SHAPES[shape])
        torch.cuda.synchronize()
    names = {_kernel_key(e.name) for e in prof.events()}
    launched = {k: [n for n in names if re.search(re.escape(k) + r"(?![\w<])", n)] for k in EXPECTED_KERNELS}
    missing = [k for k, hits in launched.items() if not hits]
    assert not missing, (missing, sorted(n for n in names if "hess" in n or "hvp" in n))
