"""Device-resident orchestration of the hot path on one B200.

``HotPathEngine`` owns the padded AO integrals in HBM and drives the C-ABI library
(``include/oo_b200.h``) on torch's current CUDA stream.  torch is used only for
device memory, streams and index tables; every arithmetic step is a kernel of
``liboo_b200.so``.  All N-sized tensors live in the padded layout (leading dimension
``ld`` = N rounded up to even, zero padding) that the TMA descriptors require.
"""
from __future__ import annotations

import math as _math
import weakref

import numpy as np
import torch

from . import _lib

F64 = torch.float64


def _p(t):
    return 0 if t is None else t.data_ptr()


def pad_even(n):
    return n + (n & 1)


def tril_pair_table(nao, params_idx):
    """(row, col) of every non-redundant rotation, in kappa order (oo_energy.py:63-94)."""
    rows, cols = np.tril_indices(nao, k=-1)
    pidx = np.asarray(params_idx, dtype=np.int64)
    return rows[pidx].astype(np.int32), cols[pidx].astype(np.int32)


class _DeviceLib:
    """The ctypes library with every call made under the engine's CUDA device: kernels launch on the
    CURRENT device, so an engine built with ``device="cuda:1"`` must not depend on what the caller's current
    device happens to be."""

    def __init__(self, lib, index):
        self._lib, self._index = lib, int(index)

    def __getattr__(self, name):
        fn, idx = getattr(self._lib, name), self._index

        def call(*args):
            if torch.cuda.current_device() == idx:
                return fn(*args)
            with torch.cuda.device(idx):
                return fn(*args)

        call.__name__ = name
        setattr(self, name, call)                         # bound once per entry point
        return call


class _Hold:
    """Token of a lazy consumer (an ``OrbitalHessian``, the autograd context of a gradient) of a set of
    transformed integrals: while one is alive the engine does not recycle that buffer for the next transform."""
    __slots__ = ("__weakref__",)


class _IntegralsKey:
    """What a cached set of transformed integrals was computed from: a tag ("mo": the matrix IS the MO
    coefficients, "oao": OAO->MO coefficients to be multiplied by S^-1/2, "C": a padded device matrix), the source
    tensor (kept alive, so its identity + version counter is a valid sync-free hit test) with a private copy of its
    values, and optionally a rotation vector.  Host tensors are compared on the host; only a DEVICE tensor that is
    not the very object seen last costs a device comparison (one synchronisation)."""

    def __init__(self, tag, src, kappa=None):
        self.tag, self.src, self.version = tag, src, src._version
        self.value = src.detach().clone()
        self.kappa = None if kappa is None else kappa.detach().clone()

    def matches(self, tag, src, kappa=None):
        if tag != self.tag or (kappa is None) != (self.kappa is None):
            return False
        if kappa is not None and not (kappa.shape == self.kappa.shape and kappa.device == self.kappa.device
                                      and torch.equal(kappa, self.kappa)):
            return False
        if src is self.src and src._version == self.version:
            return True
        if src.shape != self.value.shape or src.device != self.value.device or src.dtype != self.value.dtype:
            return False
        return bool(torch.equal(src.detach(), self.value))


class MOIntegrals:
    """Transformed integrals of ONE set of MO coefficients on the device, in either representation:
    ``kind="full"`` -- (h', g') with the complete ld^4 tensor of the four-index transform, or
    ``kind="class"`` -- the class buffer [K; J; h'] of the partial transform.  Both give the same
    numbers to every consumer (energy, Fock matrices, gradient, adjoint, Hessian)."""

    def __init__(self, eng, kind, h=None, g=None, cls=None):
        self.eng, self.kind, self.h, self.g, self.cls = eng, kind, h, g, cls
        self._holds = weakref.WeakSet()

    def hold(self):
        """A token for a consumer that will read these integrals LATER (``OrbitalHessian.matrix``, a gradient's
        ``backward``): as long as the token lives, the engine allocates a new buffer for the next transform
        instead of overwriting this one, so interleaved calls stay as safe as with the reference's dense values."""
        tok = _Hold()
        self._holds.add(tok)
        return tok

    @property
    def held(self):
        return len(self._holds) > 0

    def active_hamiltonian(self):
        if self.kind == "class":
            return self.eng.class_active_hamiltonian(self.cls)
        return self.eng.active_hamiltonian(self.h, self.g)

    def fock_gradient(self, d1, d2, want_matrix=True, want_vector=True):
        if self.kind == "class":
            return self.eng.class_fock_gradient(self.cls, d1, d2, want_matrix, want_vector)
        return self.eng.fock_gradient(self.h, self.g, d1, d2, want_matrix, want_vector)

    def fock_gradient_vjp(self, FI, Gbar):
        if self.kind == "class":
            return self.eng.class_fock_gradient_vjp(self.cls[0], FI[0], Gbar)
        return self.eng.fock_gradient_vjp(self.g[0], FI[0], Gbar)

    def hessian(self, F, d1, d2, pair_l=None, pair_r=None):
        if self.kind == "class":
            return self.eng.class_hessian(self.cls, F, d1, d2, pair_l=pair_l, pair_r=pair_r)[0]
        return self.eng.hessian(self.h[0], self.g[0], F[0], d1, d2, pair_l=pair_l, pair_r=pair_r)

    def hessian_vector(self, F, d1, d2, V):
        if self.kind == "class":
            return self.eng.class_hessian_vector(self.cls[0], F[0], d1, d2, V)
        return self.eng.hessian_vector(self.h[0], self.g[0], F[0], d1, d2, V)

    def hessian_diagonal(self, F, d1, d2):
        if self.kind == "class":
            return self.eng.class_hessian_diagonal(self.cls[0], F[0], d1, d2)
        return self.eng.hessian_diagonal(self.h[0], self.g[0], F[0], d1, d2)


class HotPathEngine:
    _tensor_engines = {}

    @classmethod
    def for_tensors(cls, nao, device=None):
        """An engine without resident integrals, for the module-level transform functions
        (``int1e_transform``, ``general_4index_transform``); cached per (size, device)."""
        if not torch.cuda.is_available():
            raise _lib.OOError("auto_oo_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        key = (int(nao), str(dev))
        if key not in cls._tensor_engines:
            cls._tensor_engines[key] = cls(None, None, None, 0.0, nao, 0, max(1, min(2, int(nao))), [], device=dev)
        return cls._tensor_engines[key]

    # relative 8-fold-symmetry defect of the AO integrals below which the symmetric class transform is used
    SYMMETRY_TOL = 1e-13

    def __init__(self, int1e_ao, int2e_ao, oao_coeff, nuc, nao, no, na, params_idx, device=None,
                 n_geometries=0, eri_symmetry="auto", eri_packing="8fold", pair_shard=None, eri_packed8=None):
        """``eri_symmetry``: "auto" measures the 8-fold symmetry of ``int2e_ao`` on the device at first use and
        takes the symmetric class transform (half the quarter-1 work, packed AO integrals) when it holds to
        round-off, the general one otherwise; "off" always takes the general one.
        ``eri_packing``: how the symmetric route keeps the AO integrals in HBM -- "8fold": both pairs packed,
        g8[(r>=s), (p>=q)] (an eighth of N^4; quarter 1 unpacks in its producer), "pair": g[r, s, (p>=q)] (half).
        ``eri_packed8``: the AO integrals already in the 8-fold packed layout ``g8[RS][PQ]`` (``(ld(ld+1)/2, pair_ld)``,
        e.g. from ``io.load_problem(..., eri="packed")``) with ``int2e_ao=None``: the N^4 tensor is never formed; the
        complete four-index transform is then unavailable, energy / gradient / Hessian run the symmetric class path.
        ``pair_shard``: ``None`` or a :class:`auto_oo_b200.distributed.PairShard` -- ONE evaluation spread over the
        ranks of a process group: this rank keeps only its slab of pair columns of the 8-fold packed integrals
        (``int2e_ao`` may then be the slab itself, see ``PairShard``), computes its additive share of the class
        buffer and all-reduces it over NVLink; energy, gradient and Hessian are then formed on every rank.
        ``n_geometries`` > 0: ``int1e_ao (G,N,N)``, ``int2e_ao (G,N,N,N,N)``, ``oao_coeff (G,N,N)``,
        ``nuc (G,)`` hold one molecule geometry each (same orbital classes); evaluation ``b`` of a
        batch then uses geometry ``b`` (class path only)."""
        if not torch.cuda.is_available():
            raise _lib.OOError("auto_oo_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.lib = _DeviceLib(_lib.load(), self.device.index)
        self.flags = 0                                 # OO_FLAG_* variant switches passed with every call (A/B tests)
        self.N = int(nao)
        self.ld = pad_even(self.N)
        self.no, self.na = int(no), int(na)
        self.nI = self.no + self.na
        self.n_geom = int(n_geometries)
        G = self.n_geom if self.n_geom > 0 else None
        self.nuc = float(nuc) if G is None else 0.0
        pl, pr = tril_pair_table(self.N, params_idx)
        self.nk = len(pl)
        self.pair_l = torch.as_tensor(pl, device=self.device)
        self.pair_r = torch.as_tensor(pr, device=self.device)
        self._pair_host = (torch.as_tensor(pl).long(), torch.as_tensor(pr).long())   # for host-side decisions
        with torch.cuda.device(self.device):
            self.h_ao = None if int1e_ao is None else self.to_padded(int1e_ao, 2, batch=G)
            self.X = None if oao_coeff is None else self.to_padded(oao_coeff, 2, batch=G)
            slab_in = pair_shard is not None and pair_shard.slab_given
            self.g_ao = None if (int2e_ao is None or slab_in) else self.to_padded(int2e_ao, 4, batch=G)
            self.nuc_dev = None if G is None else self.dev(np.asarray(nuc, dtype=np.float64).reshape(G))
        self.nIp = pad_even(self.nI)                   # class index padded to even (TMA strides)
        self.g_pairT = None                            # g_ao[p,q,r,s] stored as [r,s,p,q]; built on first use
        self.g_packed = None                           # packed AO integrals when they are 8-fold symmetric
        assert eri_packing in ("8fold", "pair")
        self.eri_packing = eri_packing
        self.pair_shard = pair_shard
        if pair_shard is not None:
            assert self.n_geom == 0 and eri_packing == "8fold", "a pair shard is one problem on 8-fold packed integrals"
            pair_shard.bind(self)
            if pair_shard.slab_given:                  # the caller handed over this rank's slab, not the N^4 tensor
                self.g_packed = self.dev(int2e_ao)
                self.g_ao = None
        self.eri_symmetry = eri_symmetry
        self._eri_symmetric = None if eri_symmetry == "auto" else False
        if pair_shard is not None:
            self._eri_symmetric = True                 # the slab layout IS the symmetric representation
        if eri_packed8 is not None:
            assert int2e_ao is None and pair_shard is None and self.n_geom == 0 and eri_packing == "8fold"
            rows = self.ld * (self.ld + 1) // 2
            self.g_packed = self.dev(eri_packed8)
            if tuple(self.g_packed.shape) != (rows, rows + (rows & 1)):
                raise ValueError(f"eri_packed8 must be ({rows}, {rows + (rows & 1)}) for {self.N} orbitals")
            self._eri_symmetric = True
        self.eri_defect = None
        self._ws = {}
        self._icache = {}                              # kind -> (_IntegralsKey | None, MOIntegrals)

    # ------------------------------------------------------------------ plumbing
    @property
    def stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    def _check(self, rc, what):
        _lib.check(rc, what)

    def dev(self, x):
        """float64 contiguous tensor on the engine's device (no copy if already there)."""
        if not torch.is_tensor(x):
            x = torch.as_tensor(np.ascontiguousarray(x))
        return x.detach().to(device=self.device, dtype=F64).contiguous()

    def to_padded(self, x, rank, batch=None):
        """dense (.., N^rank) -> zero padded (.., ld^rank) on device."""
        x = self.dev(x)
        N, ld = self.N, self.ld
        b = 1 if batch is None else batch
        if N == ld:
            out = x.reshape((b,) + (ld,) * rank)        # already in the padded layout: no copy
            return out if batch is not None else out[0]
        out = torch.empty((b,) + (ld,) * rank, dtype=F64, device=self.device)
        self._check(self.lib.oo_pad_copy_f64(_p(x), _p(out), N, ld, rank, b, 1, self.stream), "pad_copy")
        return out if batch is not None else out[0]

    def from_padded(self, x, rank):
        """padded (ld^rank) or (B, ld^rank) -> dense, on device."""
        N, ld = self.N, self.ld
        batched = x.dim() == rank + 1
        b = x.shape[0] if batched else 1
        if N == ld:
            return x
        out = torch.empty((b,) + (N,) * rank, dtype=F64, device=self.device)
        self._check(self.lib.oo_pad_copy_f64(_p(x.contiguous()), _p(out), N, ld, rank, b, 0, self.stream),
                    "pad_copy")
        return out if batched else out[0]

    def workspace(self, key, nbytes):
        buf = self._ws.get(key)
        if buf is None or buf.numel() < nbytes:
            self._ws[key] = buf = None                       # the old block goes back to the allocator first
            buf = torch.empty(int(nbytes), dtype=torch.uint8, device=self.device)
            self._ws[key] = buf
        return buf

    def stage_in(self, key, host_tensor):
        """Host -> device through a reused pinned buffer (asynchronous on the current stream)."""
        buf = self._ws.get(("pin_in", key))
        if buf is None or buf.shape != host_tensor.shape:
            buf = torch.empty(host_tensor.shape, dtype=F64, pin_memory=True)
            self._ws[("pin_in", key)] = buf
        buf.copy_(host_tensor)
        return buf.to(self.device, non_blocking=True)

    def stage_pinned(self, key, host_tensor):
        """Copy a host tensor into a reused pinned buffer and return that buffer (source of an async H2D copy)."""
        buf = self._ws.get(("pin_in", key))
        if buf is None or buf.shape != host_tensor.shape:
            buf = torch.empty(host_tensor.shape, dtype=F64, pin_memory=True)
            self._ws[("pin_in", key)] = buf
        buf.copy_(host_tensor)
        return buf

    def pinned(self, key, shape):
        buf = self._ws.get(("pin_out", key))
        if buf is None or tuple(buf.shape) != tuple(shape):
            buf = torch.empty(tuple(shape), dtype=F64, pin_memory=True)
            self._ws[("pin_out", key)] = buf
        return buf

    def copy_stream(self):
        st = self._ws.get("copy_stream")
        if st is None:
            st = self._ws["copy_stream"] = torch.cuda.Stream(self.device)
        return st

    def stage_out(self, key, dev_tensor):
        """Device -> reused pinned host buffer (asynchronous; caller synchronises the stream)."""
        buf = self._ws.get(("pin_out", key))
        if buf is None or buf.shape != dev_tensor.shape:
            buf = torch.empty(dev_tensor.shape, dtype=F64, pin_memory=True)
            self._ws[("pin_out", key)] = buf
        buf.copy_(dev_tensor, non_blocking=True)
        return buf

    def pack_lower(self, H, out=None):
        """Lower triangles (np.tril_indices order) of symmetric device matrices ``H (B, n, n)`` -> ``(B, n(n+1)/2)``."""
        H = H if H.dim() == 3 else H[None]
        B, n = H.shape[0], H.shape[1]
        P = out if out is not None else torch.empty(B, n * (n + 1) // 2, dtype=F64, device=self.device)
        if n > 0 and B > 0:
            self._check(self.lib.oo_pack_lower_f64(_p(H), n, B, _p(P), self.stream), "pack_lower")
        return P

    def upload_pinned(self, pinned):
        """Device copy of a PINNED host tensor made by a kernel that reads the host memory directly (no DMA-engine
        copy on the compute stream -- see ``oo_copy_f64``)."""
        out = torch.empty(tuple(pinned.shape), dtype=F64, device=self.device)
        self._check(self.lib.oo_copy_f64(pinned.data_ptr(), _p(out), pinned.numel(), self.stream), "copy")
        return out

    def resident_oao(self, oao_mo_coeff):
        """Padded device copy of ``OO_energy.oao_mo_coeff``, re-uploaded only when the tensor object or its version
        counter changes (callers re-assign it or write into it: oo_pqc.py:191, Berry cell 22)."""
        if not torch.is_tensor(oao_mo_coeff):                  # (a numpy array assigned by the caller: no version counter)
            return self.to_padded(oao_mo_coeff, 2)
        ent = self._ws.get("oao_dev")
        if ent is None or ent[0] is not oao_mo_coeff or ent[1] != oao_mo_coeff._version:
            ent = (oao_mo_coeff, oao_mo_coeff._version, self.to_padded(oao_mo_coeff, 2))
            self._ws["oao_dev"] = ent
        return ent[2]

    def result_slot(self, slot, shapes):
        """One of the two alternating sets of host-result staging buffers of ``energy_gradient_hessian``:
        pinned tensors of the given shapes (dict name -> shape) plus a completion event, rebuilt when a shape
        changes.  Two sets let the device->host copies of one call overlap the computation of the next."""
        ent = self._ws.get(("slot", slot))
        if ent is None or ent["shapes"] != shapes:
            self._ws[("slot", slot)] = None
            ent = {"shapes": dict(shapes), "done": None,
                   "host": {k: torch.empty(tuple(v), dtype=F64, pin_memory=True) for k, v in shapes.items()}}
            self._ws[("slot", slot)] = ent
        return ent

    def workspace_tensor(self, key, shape):
        """Reused float64 device buffer of the given shape."""
        buf = self._ws.get(("t", key))
        if buf is None or tuple(buf.shape) != tuple(shape):
            self._ws[("t", key)] = None
            buf = torch.empty(tuple(shape), dtype=F64, device=self.device)
            self._ws[("t", key)] = buf
        return buf

    def release_workspaces(self):
        self._ws.clear()
        self._icache.clear()

    # ------------------------------------------------------------------ K1
    def squarings_for(self, kappa):
        """s = max(0, ceil(log2(||K||_1 / 0.95))) from the packed parameters (max over a batch)."""
        k = kappa.detach().abs().reshape(-1, self.nk).to(F64)
        if self.nk == 0:
            return 0
        if k.device.type == "cpu":
            colsum = torch.zeros(k.shape[0], self.N, dtype=F64)
            pl, pr = self._pair_host
        else:
            colsum = torch.zeros(k.shape[0], self.N, dtype=F64, device=k.device)
            pl, pr = self.pair_l.long(), self.pair_r.long()
        colsum.index_add_(1, pl, k)
        colsum.index_add_(1, pr, k)
        norm1 = float(colsum.max())
        if not _math.isfinite(norm1):
            raise ValueError("kappa contains non-finite values")
        if norm1 <= 0.95:
            return 0
        return int(_math.ceil(_math.log2(norm1 / 0.95)))

    def rotation(self, kappa, squarings=None):
        """kappa (B, nk) on device -> U (B, ld, ld) = expm(-K(kappa))."""
        kappa = self.dev(kappa).reshape(-1, self.nk)
        B = kappa.shape[0]
        if squarings is None:
            # small bases: the fused kernel applies the rule per matrix on the device (no host round trip)
            squarings = -1 if self.N <= self.lib.oo_expm_device_squarings_max_n() else self.squarings_for(kappa)
        U = torch.empty(B, self.ld, self.ld, dtype=F64, device=self.device)
        nbytes = self.lib.oo_workspace_bytes(_lib.OO_WS_ROTATION, self.N, self.ld, 0, B)
        ws = self.workspace("rot", nbytes)
        self._check(self.lib.oo_kappa_rotation_f64(_p(kappa), _p(self.pair_l), _p(self.pair_r), self.nk,
                                                   self.N, self.ld, B, int(squarings), _p(U), _p(ws),
                                                   nbytes, self.stream), "kappa_rotation")
        return U

    def rotation_vjp(self, kappa, Ubar, squarings=None):
        """kappa (B, nk), Ubar (B, ld, ld) on device -> kappa_bar (B, nk): the vector-Jacobian product of
        :meth:`rotation` for the cotangent ``Ubar = dE/dU`` (only its N x N block is read)."""
        kappa = self.dev(kappa).reshape(-1, self.nk)
        B = kappa.shape[0]
        Ubar = Ubar.reshape(B, self.ld, self.ld).contiguous()
        if squarings is None:
            # the single-launch adjoint (8 <= ld <= 256) chooses s on the device; the multi-launch one needs it here
            squarings = -1 if 8 <= self.ld <= self.lib.oo_expm_device_squarings_max_n() else self.squarings_for(kappa)
        kbar = torch.empty(B, self.nk, dtype=F64, device=self.device)
        nbytes = self.lib.oo_workspace_bytes(_lib.OO_WS_ROTATION_VJP, self.N, self.ld, 0, B)
        ws = self.workspace("rot_vjp", nbytes)
        self._check(self.lib.oo_kappa_rotation_vjp_f64(_p(kappa), _p(self.pair_l), _p(self.pair_r), self.nk,
                                                       self.N, self.ld, B, int(squarings), _p(Ubar), _p(kbar),
                                                       _p(ws), nbytes, self.stream), "kappa_rotation_vjp")
        return kbar

    def mo_coeff(self, oao_mo_coeff, U=None):
        """C' = X C_oao U  (padded, batched over U; one X per evaluation for geometry batches)."""
        Coao = oao_mo_coeff if oao_mo_coeff.dim() == 3 else oao_mo_coeff[None]
        B = max(Coao.shape[0], 1 if U is None else U.shape[0])
        if self.n_geom:
            assert B == self.n_geom, "a geometry batch evaluates exactly one rotation per geometry"
        out = torch.empty(B, self.ld, self.ld, dtype=F64, device=self.device)
        nbytes = self.lib.oo_workspace_bytes(_lib.OO_WS_INT1E, self.N, self.ld, 0, B)
        ws = self.workspace("i1e", nbytes)
        mat = self.ld * self.ld
        sC = mat if Coao.shape[0] > 1 else 0
        sU = 0 if U is None or U.shape[0] == 1 else mat
        self._check(self.lib.oo_mo_coeff_f64(_p(self.X), mat if self.n_geom > 1 else 0, _p(Coao), sC, _p(U), sU,
                                             self.N, self.ld, B,
                                             _p(out), _p(ws), nbytes, self.stream), "mo_coeff")
        return out

    # ------------------------------------------------------------------ K2
    def int1e_transform(self, C, h_ao=None, geo=(0, None)):
        C = C if C.dim() == 3 else C[None]
        B = C.shape[0]
        out = torch.empty(B, self.ld, self.ld, dtype=F64, device=self.device)
        nbytes = self.lib.oo_workspace_bytes(_lib.OO_WS_INT1E, self.N, self.ld, 0, B)
        ws = self.workspace("i1e", nbytes)
        mat = self.ld * self.ld
        if h_ao is None:
            h, sh = self._geo(self.h_ao, geo[0], geo[0] + B)
        else:
            h, sh = h_ao, 0
        self._check(self.lib.oo_int1e_transform_f64(_p(h), sh, _p(C), mat if B > 1 else 0, self.N, self.ld, B,
                                                    _p(out), _p(ws), nbytes, self.stream), "int1e_transform")
        return out

    def int2e_transform(self, C0, C1=None, C2=None, C3=None, g_ao=None, out=None):
        """g'[b] from padded coefficient matrices (B, ld, ld); g_ao shared unless (B, ld^4) given."""
        C0 = C0 if C0.dim() == 3 else C0[None]
        Cs = [C0] + [C0 if c is None else (c if c.dim() == 3 else c[None]) for c in (C1, C2, C3)]
        B = C0.shape[0]
        ld = self.ld
        g = self.g_ao if g_ao is None else g_ao
        if g is None:
            raise _lib.OOError("the complete four-index transform needs the dense AO integrals (this engine only holds "
                               "their packed / sharded form: use the class path)")
        strideG = ld ** 4 if (g.dim() == 5 and g.shape[0] > 1) else 0
        if out is None:
            out = torch.empty((B, ld, ld, ld, ld), dtype=F64, device=self.device)
        nbytes = self.lib.oo_workspace_bytes(_lib.OO_WS_INT2E, self.N, ld, 0, B)
        ws = self.workspace("i2e", nbytes)
        self._check(self.lib.oo_int2e_transform_f64(_p(g), strideG, _p(Cs[0]), _p(Cs[1]), _p(Cs[2]),
                                                    _p(Cs[3]), ld * ld if B > 1 else 0, self.N, ld, B,
                                                    _p(out), _p(ws), nbytes, self.stream), "int2e_transform")
        return out

    # ------------------------------------------------------------------ cache of transformed integrals
    def _recycle(self, kind):
        """The big buffer of the last transform of this kind (class buffer / g') for reuse, or None when there is
        none or a lazy consumer still holds it (:meth:`MOIntegrals.hold`): the cache entry is dropped either way."""
        ent = self._icache.pop(kind, None)
        if ent is None or ent[1].held:
            return None
        return ent[1].cls if kind == "class" else ent[1].g

    def _park(self, kind, buf):
        """Keep a scratch buffer of :meth:`evaluate` for the next transform (no key: never a cache hit)."""
        if buf is not None and buf.shape[0] == 1:
            self._icache[kind] = (None, MOIntegrals(self, kind, cls=buf) if kind == "class"
                                  else MOIntegrals(self, kind, g=buf))

    def integrals_for(self, kind, tag, src, make_C, kappa=None):
        """:class:`MOIntegrals` of kind "class" / "full", cached under (tag, src[, kappa]) -- see
        :class:`_IntegralsKey`; ``make_C()`` supplies the padded (ld, ld) MO coefficients on a miss."""
        ent = self._icache.get(kind)
        if ent is not None and ent[0] is not None and ent[0].matches(tag, src, kappa):
            return ent[1]
        C = make_C().reshape(1, self.ld, self.ld)
        buf = self._recycle(kind)
        if kind == "class":
            ints = MOIntegrals(self, "class", cls=self.class_integrals(C, out=buf))
        else:
            ints = MOIntegrals(self, "full", h=self.int1e_transform(C), g=self.int2e_transform(C, out=buf))
        self._icache[kind] = (_IntegralsKey(tag, src, kappa), ints)
        return ints

    def integrals(self, C, kind="class"):
        """:class:`MOIntegrals` for one padded device matrix C (ld, ld), cached by identity / value of C."""
        return self.integrals_for(kind, "C", C, lambda: C)

    def mo_integrals(self, C):
        """(h', g') for padded C (ld, ld) or (B, ld, ld); a single matrix goes through the cache."""
        C = C if C.dim() == 3 else C[None]
        if C.shape[0] == 1:
            ints = self.integrals(C[0], kind="full")
            return ints.h, ints.g
        return self.int1e_transform(C), self.int2e_transform(C)

    # ------------------------------------------------------------------ class (partial-transform) path
    def pair_transposed_eri(self):
        """g_pairT[r,s,p,q] = g_ao[p,q,r,s] (one HBM-bound transpose, once per problem)."""
        if self.g_pairT is None:
            ld2 = self.ld * self.ld
            out = torch.empty_like(self.g_ao)
            src, dst = self.g_ao.reshape(-1, ld2, ld2), out.reshape(-1, ld2, ld2)
            for i in range(src.shape[0]):
                self._check(self.lib.oo_transpose_f64(_p(src[i]), _p(dst[i]), ld2, ld2, self.stream), "transpose")
            self.g_pairT = out
        return self.g_pairT

    def eri_is_symmetric(self):
        """True when every resident AO tensor has (pq|rs) = (qp|rs) = (rs|pq) to round-off (measured once
        on the device; ``eri_defect`` keeps (max |g_pqrs - g_qprs|, max |g_pqrs - g_rspq|, max |g|))."""
        if self._eri_symmetric is None:
            g = self.g_ao.reshape(-1, self.ld ** 4)
            worst = torch.zeros(3, dtype=F64, device=self.device)
            d = torch.empty(3, dtype=F64, device=self.device)
            for i in range(g.shape[0]):
                self._check(self.lib.oo_eri_symmetry_defect_f64(_p(g[i]), self.ld, _p(d), self.stream),
                            "eri_symmetry_defect")
                worst = torch.maximum(worst, d)
            dpq, dpair, amax = (float(x) for x in worst.cpu())
            self.eri_defect = (dpq, dpair, amax)
            self._eri_symmetric = max(dpq, dpair) <= self.SYMMETRY_TOL * max(amax, 1e-300)
        return self._eri_symmetric

    def packed_eri(self):
        """The symmetric route's copy of the AO integrals over the ld padded orbitals (row = packed pair p >= q,
        padded to even): ``eri_packing="8fold"`` g8[(r>=s), (pq)], ``"pair"`` g[r, s, (pq)]."""
        if self.g_packed is None and self.pair_shard is not None:
            # full tensor given (small problems, tests): pack all of it, keep this rank's columns
            sh, self.pair_shard = self.pair_shard, None
            try:
                full = self.packed_eri()
            finally:
                self.pair_shard = sh
            self.g_packed = full[:, sh.pq_lo:sh.pq_lo + sh.slab_ld].contiguous()
            del full
        if self.g_packed is None:
            ldp = int(self.lib.oo_pair_ld(self.ld))
            g = self.g_ao.reshape(-1, self.ld ** 4)
            if self.eri_packing == "8fold":
                out = torch.empty(g.shape[0], self.ld * (self.ld + 1) // 2, ldp, dtype=F64, device=self.device)
                pack, what = self.lib.oo_pack_eri_8fold_f64, "pack_eri_8fold"
            else:
                out = torch.empty(g.shape[0], self.ld, self.ld, ldp, dtype=F64, device=self.device)
                pack, what = self.lib.oo_pack_eri_pairs_f64, "pack_eri_pairs"
            for i in range(g.shape[0]):
                self._check(pack(_p(g[i]), _p(out[i]), self.ld, self.stream), what)
            self.g_packed = out if self.n_geom else out[0]
        return self.g_packed

    def _geo(self, t, lo, hi):
        """(tensor, per-evaluation stride) of a per-problem / per-geometry resident tensor for the
        evaluations [lo, hi) of a batch."""
        if self.n_geom == 0:
            return t, 0
        sl = t[lo:hi]
        return sl, (sl[0].numel() if hi - lo > 1 else 0)

    def drop_full_eri(self):
        """Free g_ao (and the full-transform buffers) once the class path's own copy exists (the packed
        tensor for symmetric integrals, the pair-transposed one otherwise).  The full four-index transform API then needs ``g_ao=`` again."""
        if self.eri_is_symmetric():
            self.packed_eri()
        else:
            self.pair_transposed_eri()
        self.g_ao = None
        self._icache.pop("full", None)
        self._ws.pop("i2e", None)

    def class_rows(self):
        return 2 * self.nIp * self.nIp + 1

    def class_integrals(self, C, out=None, geo_lo=0):
        """Class buffers [K rows; J rows; h' row] for padded C (ld, ld) or (B, ld, ld):
        returns (B, 2 nIp^2 + 1, ld, ld); every GEMM step is one batched launch."""
        C = C.reshape(-1, self.ld, self.ld)
        B, ld, nIp, rows = C.shape[0], self.ld, self.nIp, self.class_rows()
        cls = out if out is not None and out.shape[0] == B else torch.empty(B, rows, ld, ld, dtype=F64,
                                                                           device=self.device)
        if self.pair_shard is not None:
            sh = self.pair_shard
            nbytes = self.lib.oo_workspace_bytes(_lib.OO_WS_CLASS_TRANSFORM_SYM, self.N, ld, self.nI, B)
            ws = self.workspace("cls", nbytes)
            self._check(self.lib.oo_class_transform_sym_slab_f64(_p(self.packed_eri()), sh.slab_ld, sh.pq_lo, sh.pq_cnt,
                                                                 _p(C), ld * ld if B > 1 else 0, self.N, ld, nIp, B,
                                                                 _p(cls), _p(ws), nbytes, self.flags, self.stream),
                        "class_transform_sym_slab")
            # sum of the ranks' shares of the K and J rows (the whole contiguous buffer goes through the collective;
            # its last row, h', is written below)
            sh.all_reduce(cls)
        elif self.eri_is_symmetric():
            nbytes = self.lib.oo_workspace_bytes(_lib.OO_WS_CLASS_TRANSFORM_SYM, self.N, ld, self.nI, B)
            ws = self.workspace("cls", nbytes)
            gp, sg = self._geo(self.packed_eri(), geo_lo, geo_lo + B)
            flags = self.flags | (_lib.OO_FLAG_CLASS_ERI_8FOLD if self.eri_packing == "8fold" else 0)
            self._check(self.lib.oo_class_transform_sym_f64(_p(gp), sg, _p(C), ld * ld if B > 1 else 0,
                                                            self.N, ld, nIp, B, _p(cls), _p(ws), nbytes,
                                                            flags, self.stream), "class_transform_sym")
        else:
            nbytes = self.lib.oo_workspace_bytes(_lib.OO_WS_CLASS_TRANSFORM, self.N, ld, self.nI, B)
            ws = self.workspace("cls", nbytes)
            gp, sg = self._geo(self.pair_transposed_eri(), geo_lo, geo_lo + B)
            self._check(self.lib.oo_class_transform_f64(_p(gp), sg, _p(C), ld * ld if B > 1 else 0,
                                                        self.N, ld, nIp, B, _p(cls), _p(ws), nbytes, self.stream),
                        "class_transform")
        if B == 1:                                           # h' = C^T h C straight into the last row
            nb1 = self.lib.oo_workspace_bytes(_lib.OO_WS_INT1E, self.N, ld, 0, 1)
            ws1 = self.workspace("i1e", nb1)
            h1, _ = self._geo(self.h_ao, geo_lo, geo_lo + 1)
            self._check(self.lib.oo_int1e_transform_f64(_p(h1), 0, _p(C), 0, self.N, ld, 1, _p(cls[0, rows - 1]),
                                                        _p(ws1), nb1, self.stream), "int1e_transform")
        else:                                                # batched: dense scratch, then a strided device copy
            cls[:, rows - 1].copy_(self.int1e_transform(C, geo=(geo_lo, None)))
        return cls

    def class_active_hamiltonian(self, cls, geo_lo=0):
        na, B = self.na, cls.shape[0]
        nuc_b = None if self.n_geom == 0 else self.nuc_dev[geo_lo:geo_lo + B]
        c0 = torch.empty(B, dtype=F64, device=self.device)
        c1 = torch.empty(B, na, na, dtype=F64, device=self.device)
        c2 = torch.empty(B, na, na, na, na, dtype=F64, device=self.device)
        self._check(self.lib.oo_class_active_hamiltonian_f64(_p(cls), self.no, na, self.N, self.ld, self.nIp, B,
                                                             self.nuc, _p(nuc_b), _p(c0), _p(c1), _p(c2),
                                                             self.stream),
                    "class_active_hamiltonian")
        return c0, c1, c2

    def class_fock_gradient(self, cls, d1, d2, want_matrix=True, want_vector=True):
        ld, B = self.ld, cls.shape[0]
        s1, s2 = self._rdm_strides(d1, d2, B)
        FI = torch.empty(B, ld, ld, dtype=F64, device=self.device)
        FA = torch.empty_like(FI)
        F = torch.empty_like(FI)
        G = torch.empty_like(FI) if want_matrix else None
        gv = torch.empty(B, self.nk, dtype=F64, device=self.device) if want_vector else None
        self._check(self.lib.oo_class_fock_gradient_f64(_p(cls), _p(d1), s1, _p(d2), s2, self.no, self.na, self.N,
                                                        ld, self.nIp, B, _p(self.pair_l), _p(self.pair_r),
                                                        self.nk, _p(FI), _p(FA), _p(F), _p(G), _p(gv),
                                                        self.stream), "class_fock_gradient")
        return FI, FA, F, G, gv

    def class_fock_gradient_vjp(self, cls, FI, Gbar):
        na = self.na
        g1 = torch.empty(na, na, dtype=F64, device=self.device)
        g2 = torch.empty(na, na, na, na, dtype=F64, device=self.device)
        self._check(self.lib.oo_class_fock_gradient_vjp_f64(_p(cls), _p(FI), _p(Gbar), self.no, na, self.N,
                                                            self.ld, self.nIp, _p(g1), _p(g2), self.stream),
                    "class_fock_gradient_vjp")
        return g1, g2

    def class_hessian(self, cls, F, d1, d2, out=None, pair_l=None, pair_r=None):
        """Hessians (B, nk, nk) of the B evaluations in cls (B, rows, ld, ld), F (B, ld, ld)."""
        pl = self.pair_l if pair_l is None else pair_l
        pr = self.pair_r if pair_r is None else pair_r
        nk = int(pl.numel())
        B = cls.shape[0]
        H = out if out is not None else torch.empty(B, nk, nk, dtype=F64, device=self.device)
        if nk == 0:
            return H
        s1, s2 = self._rdm_strides(d1, d2, B)
        nbytes = self.lib.oo_workspace_bytes(_lib.OO_WS_CLASS_HESSIAN, self.na, self.ld, self.nI, B)
        ws = self.workspace("chess", nbytes)
        # operands that depend on the RDMs / the pair list alone stay in the workspace: reuse them when the very same
        # tensors (kept alive here, so neither address can be recycled; unchanged version counters) come again
        key = (ws.data_ptr(), B, self.flags, d1.data_ptr(), d1._version, d2.data_ptr(), d2._version, pl.data_ptr(),
               pr.data_ptr(), nk)
        prev = self._ws.get("chess_key")
        # (never inside a CUDA-graph capture: a replay sees new RDM values in the same static buffers)
        reuse = prev is not None and prev[0] == key and not self._ws.get("capturing", False)
        flags = self.flags | (_lib.OO_FLAG_HESSIAN_REUSE_OPERANDS if reuse else 0)
        self._ws["chess_key"] = (key, d1, d2, pl, pr)
        self._check(self.lib.oo_class_hessian_f64(_p(cls), _p(F), _p(d1), s1, _p(d2), s2, self.no, self.na, self.N,
                                                  self.ld, self.nIp, B, _p(pl), _p(pr), nk, _p(H), _p(ws), nbytes,
                                                  flags, self.stream), "class_hessian")
        return H

    def class_hessian_vector(self, cls, F, d1, d2, V, out=None):
        """H V (nk, nv) of ONE evaluation, cls (rows, ld, ld), F (ld, ld), V (nk, nv) device tensors, without
        forming H."""
        nk, nv = V.shape
        HV = out if out is not None else torch.empty(nk, nv, dtype=F64, device=self.device)
        if nk == 0 or nv == 0:
            return HV
        nbytes = self.lib.oo_workspace_bytes(_lib.OO_WS_CLASS_HESSIAN_VECTOR, self.na, self.ld, self.nI, nv)
        ws = self.workspace("hvp", nbytes)
        self._check(self.lib.oo_class_hessian_vector_f64(_p(cls), _p(F), _p(d1), _p(d2), self.no, self.na, self.N,
                                                         self.ld, self.nIp, _p(self.pair_l), _p(self.pair_r), nk,
                                                         _p(V), nv, _p(HV), _p(ws), nbytes, self.stream),
                    "class_hessian_vector")
        return HV

    def class_hessian_diagonal(self, cls, F, d1, d2):
        """diag(H) (nk,) of ONE evaluation from its class buffer."""
        diag = torch.empty(self.nk, dtype=F64, device=self.device)
        if self.nk == 0:
            return diag
        self._check(self.lib.oo_class_hessian_diagonal_f64(_p(cls), _p(F), _p(d1), _p(d2), self.no, self.na, self.N,
                                                           self.ld, self.nIp, _p(self.pair_l), _p(self.pair_r),
                                                           self.nk, _p(diag), None, 0, self.stream),
                    "class_hessian_diagonal")
        return diag

    def pairs_quarter_one(self):
        """True when `oo_class_transform_sym_f64` sends two evaluations of a batch through one quarter-1 GEMM (the
        same conditions as in csrc/classes.cu: 8-fold packed integrals shared by the batch, triangular quarter 2, a
        tile configuration for the 2 nIp columns)."""
        w = 2 * self.nIp
        off = _lib.OO_FLAG_CLASS_Q1_UNPAIRED | _lib.OO_FLAG_CLASS_UNFUSED_PACK | _lib.OO_FLAG_CLASS_Q2_RECTANGULAR
        return (self.eri_packing == "8fold" and self.pair_shard is None and self.n_geom == 0 and not (self.flags & off)
                and 16 < self.nIp <= 48 and (w <= 48 or 80 < w <= 96) and self.eri_is_symmetric())

    def class_chunk(self, B):
        """How many evaluations the class path processes per batched launch: as many as keep the
        transform + Hessian workspaces under ~8 GB (always at least one) -- and two where quarter 1 runs on pairs
        of evaluations and the device has the room (N=256: 2 x 16 GB)."""
        which = _lib.OO_WS_CLASS_TRANSFORM_SYM if self.eri_is_symmetric() else _lib.OO_WS_CLASS_TRANSFORM
        per = (self.lib.oo_workspace_bytes(which, self.N, self.ld, self.nI, 1)
               + self.lib.oo_workspace_bytes(_lib.OO_WS_CLASS_HESSIAN, self.na, self.ld, self.nI, 1)
               + self.lib.oo_workspace_bytes(_lib.OO_WS_CLASS_BUFFER, self.N, self.ld, self.nI, 1))
        n = int(max(1, min(B, (8 << 30) // max(per, 1))))
        if n < 2 <= B and self.pairs_quarter_one():
            room = self._ws.get("pair_room")                 # asked once (cudaMemGetInfo is not free); forgotten with
            if room is None:                                 # the workspaces (release_workspaces)
                free, _ = torch.cuda.mem_get_info(self.device)
                free += torch.cuda.memory_reserved(self.device) - torch.cuda.memory_allocated(self.device)
                held = sum(self._ws[k].numel() for k in ("cls", "chess") if torch.is_tensor(self._ws.get(k)))
                room = self._ws["pair_room"] = bool(2 * per <= 0.6 * (free + held))
            if room:
                n = 2
        return n

    # ------------------------------------------------------------------ K3
    def active_hamiltonian(self, h, g):
        B, na = h.shape[0], self.na
        c0 = torch.empty(B, dtype=F64, device=self.device)
        c1 = torch.empty(B, na, na, dtype=F64, device=self.device)
        c2 = torch.empty(B, na, na, na, na, dtype=F64, device=self.device)
        self._check(self.lib.oo_active_hamiltonian_f64(_p(h), _p(g), self.no, na, self.N, self.ld, B,
                                                       self.nuc, None, _p(c0), _p(c1), _p(c2), self.stream),
                    "active_hamiltonian")
        return c0, c1, c2

    def _rdm_strides(self, d1, d2, B):
        na = self.na
        s1 = na * na if (d1.dim() == 3 and d1.shape[0] > 1) else 0
        s2 = na ** 4 if (d2.dim() == 5 and d2.shape[0] > 1) else 0
        assert s1 == 0 or d1.shape[0] == B
        assert s2 == 0 or d2.shape[0] == B
        return s1, s2

    def energy(self, c0, c1, c2, d1, d2):
        B = c0.shape[0]
        s1, s2 = self._rdm_strides(d1, d2, B)
        E = torch.empty(B, dtype=F64, device=self.device)
        self._check(self.lib.oo_energy_f64(_p(c0), _p(c1), _p(c2), _p(d1), s1, _p(d2), s2, self.na, B,
                                           _p(E), self.stream), "energy")
        return E

    # ------------------------------------------------------------------ K4
    def fock_gradient(self, h, g, d1, d2, want_matrix=True, want_vector=True):
        B, ld = h.shape[0], self.ld
        s1, s2 = self._rdm_strides(d1, d2, B)
        FI = torch.empty(B, ld, ld, dtype=F64, device=self.device)
        FA = torch.empty_like(FI)
        F = torch.empty_like(FI)
        G = torch.empty_like(FI) if want_matrix else None
        gv = torch.empty(B, self.nk, dtype=F64, device=self.device) if want_vector else None
        self._check(self.lib.oo_fock_gradient_f64(_p(h), _p(g), _p(d1), s1, _p(d2), s2, self.no, self.na,
                                                  self.N, ld, B, _p(self.pair_l), _p(self.pair_r), self.nk,
                                                  _p(FI), _p(FA), _p(F), _p(G), _p(gv), self.stream),
                    "fock_gradient")
        return FI, FA, F, G, gv

    def fock_gradient_vjp(self, g, FI, Gbar):
        na = self.na
        g1 = torch.empty(na, na, dtype=F64, device=self.device)
        g2 = torch.empty(na, na, na, na, dtype=F64, device=self.device)
        self._check(self.lib.oo_fock_gradient_vjp_f64(_p(g), _p(FI), _p(Gbar), self.no, na, self.N, self.ld,
                                                      _p(g1), _p(g2), self.stream), "fock_gradient_vjp")
        return g1, g2

    def hessian(self, h, g, F, d1, d2, out=None, pair_l=None, pair_r=None):
        """(nk, nk) Hessian for ONE evaluation (h, g, F are single padded tensors); the rotation
        pairs default to the engine's non-redundant ones."""
        pl = self.pair_l if pair_l is None else pair_l
        pr = self.pair_r if pair_r is None else pair_r
        nk = int(pl.numel())
        H = out if out is not None else torch.empty(nk, nk, dtype=F64, device=self.device)
        if nk == 0:
            return H
        nbytes = self.lib.oo_workspace_bytes(_lib.OO_WS_HESSIAN, self.N, self.ld, self.nI, 1)
        ws = self.workspace("hess", nbytes)
        self._check(self.lib.oo_hessian_f64(_p(h), _p(g), _p(F), _p(d1), _p(d2), self.no, self.na, self.N,
                                            self.ld, _p(pl), _p(pr), nk, _p(H), _p(ws),
                                            nbytes, self.flags, self.stream), "hessian")
        return H

    def hessian_vector(self, h, g, F, d1, d2, V, out=None):
        """H V (nk, nv) of ONE evaluation from the complete transformed integrals (single padded h, g, F)."""
        nk, nv = V.shape
        HV = out if out is not None else torch.empty(nk, nv, dtype=F64, device=self.device)
        if nk == 0 or nv == 0:
            return HV
        nbytes = self.lib.oo_workspace_bytes(_lib.OO_WS_HESSIAN_VECTOR, self.na, self.ld, self.nI, nv)
        ws = self.workspace("hvp_full", nbytes)
        self._check(self.lib.oo_hessian_vector_f64(_p(h), _p(g), _p(F), _p(d1), _p(d2), self.no, self.na, self.N,
                                                   self.ld, _p(self.pair_l), _p(self.pair_r), nk, _p(V), nv, _p(HV),
                                                   _p(ws), nbytes, self.stream), "hessian_vector")
        return HV

    def hessian_diagonal(self, h, g, F, d1, d2):
        """diag(H) (nk,) of ONE evaluation from the complete transformed integrals."""
        diag = torch.empty(self.nk, dtype=F64, device=self.device)
        if self.nk == 0:
            return diag
        nbytes = self.lib.oo_workspace_bytes(_lib.OO_WS_HESSIAN_DIAGONAL, self.N, self.ld, self.nI, 1)
        ws = self.workspace("hdiag_full", nbytes)
        self._check(self.lib.oo_hessian_diagonal_f64(_p(h), _p(g), _p(F), _p(d1), _p(d2), self.no, self.na, self.N,
                                                     self.ld, _p(self.pair_l), _p(self.pair_r), self.nk, _p(diag),
                                                     _p(ws), nbytes, self.stream), "hessian_diagonal")
        return diag

    # ------------------------------------------------------------------ Krylov arithmetic between products (krylov.cu)
    def krylov_workspace(self, n, kmax):
        nbytes = self.lib.oo_workspace_bytes(_lib.OO_WS_KRYLOV, int(n), 1, int(kmax), 1)
        return self.workspace("krylov", nbytes), nbytes

    def subspace_eigh(self, S, k, w, Y):
        """Ascending eigenvalues ``w[:k]`` and eigenvectors (columns of ``Y[:k, :k]``) of the leading k x k block of
        the symmetric ``S`` (lower triangle read); ``S (m, m)`` or a batch ``(B, m, m)`` with ``w (B, m)``,
        ``Y (B, m, m)``."""
        B = S.shape[0] if S.dim() == 3 else 1
        self._check(self.lib.oo_subspace_eigh_f64(_p(S), int(k), S.shape[-1], S.shape[-1] * S.shape[-2], B, _p(w),
                                                  w.shape[-1], _p(Y), Y.shape[-1], Y.shape[-1] * Y.shape[-2],
                                                  self.stream), "subspace_eigh")

    def davidson_project(self, Vt, k, u, out, inc, out2=None, inc2=0):
        """``out[j*inc] = Vt[j] . u`` (and ``out2[j*inc2]``) for j < k."""
        self._check(self.lib.oo_davidson_project_f64(_p(Vt), Vt.shape[1], u.numel(), int(k), _p(u), _p(out), int(inc),
                                                     _p(out2), int(inc2), self.stream), "davidson_project")

    def davidson_expand(self, Vt, HVt, k, Y, theta, D, S, x, hx, yprev, rnorm, floor):
        """Ritz pair of column 0 of Y, residual norm, and the next basis row (restart when k = rows of Vt)."""
        n, kmax = D.numel(), Vt.shape[0]
        ws, nbytes = self.krylov_workspace(n, kmax)
        self._check(self.lib.oo_davidson_expand_f64(_p(Vt), _p(HVt), n, Vt.shape[1], int(k), kmax, _p(Y), Y.shape[1],
                                                    _p(theta), _p(D), float(floor), _p(S), S.shape[1], _p(x), _p(hx),
                                                    _p(yprev), _p(rnorm), _p(ws), nbytes, self.stream),
                    "davidson_expand")

    def pcg_step(self, Ap, shift, D, x, r, p, state, rnorm, w=None, aw=None, init=False):
        """One deflated PCG step on (H + shift) x = b (``init``: the start from r = b); ``Ap = H p``."""
        n = D.numel()
        ws, nbytes = self.krylov_workspace(n, 1)
        self._check(self.lib.oo_pcg_step_f64(n, _p(Ap), float(shift), _p(D), _p(w), _p(aw), _p(x), _p(r), _p(p),
                                             _p(state), _p(rnorm), int(bool(init)), _p(ws), nbytes, self.stream),
                    "pcg_step")

    def full_rdms(self, d1, d2):
        """Dense full-space RDMs (reference full_rdms, oo_energy.py:342-379): (N,N), (N,N,N,N)."""
        N = self.N
        one = torch.empty(N, N, dtype=F64, device=self.device)
        two = torch.empty(N, N, N, N, dtype=F64, device=self.device)
        self._check(self.lib.oo_full_rdms_f64(_p(d1), _p(d2), self.no, self.na, N, _p(one), _p(two),
                                              self.stream), "full_rdms")
        return one, two

    def y_matrix_dense(self, int2e_mo, two_full):
        """Reference y_matrix (oo_energy.py:381-393) for an arbitrary dense two_full."""
        N = self.N
        g = self.to_padded(int2e_mo, 4)
        G = self.dev(two_full)
        Y = torch.empty(N, N, N, N, dtype=F64, device=self.device)
        nbytes = self.lib.oo_workspace_bytes(_lib.OO_WS_YMATRIX, N, self.ld, 0, 1)
        ws = self.workspace("ymat", nbytes)
        self._check(self.lib.oo_y_matrix_f64(_p(g), _p(G), N, self.ld, _p(Y), _p(ws), nbytes, self.stream),
                    "y_matrix")
        return Y

    def matmul(self, A, B, transA=False, transB=False, alpha=1.0):
        """alpha op(A) @ op(B) for padded (ld, ld) device matrices on the small DMMA GEMM."""
        ld = self.ld
        out = torch.empty(ld, ld, dtype=F64, device=self.device)
        self._check(self.lib.oo_dgemm_small_f64(int(transA), int(transB), ld, ld, ld, float(alpha), _p(A), ld, 0,
                                                _p(B), ld, 0, 0.0, 0, ld, 0, 0.0, _p(out), ld, 0, 1, self.stream),
                    "dgemm_small")
        return out

    # ------------------------------------------------------------------ whole evaluations
    def evaluate(self, oao_mo_coeff, d1, d2, kappa=None, want_hessian=True, squarings=None,
                 H_out=None, stage_events=None, path="class", on_result=None, on_integrals=None):
        """E (B,), packed gradient (B, nk) and Hessian (B, nk, nk) at C' = X C_oao expm(-K(kappa_b)).

        ``oao_mo_coeff``: padded (ld, ld) or (B, ld, ld) device tensor; ``kappa``: (B, nk) or None.
        One 4-index transform per evaluation serves E, G and H (the reference repeats it
        three times: oo_energy.py:207-208, :410-411, :421-422).  ``path="class"`` computes only the
        J/K integral classes E, G and H read (partial transform); ``path="full"`` the complete
        four-index transform.  Evaluations are processed
        one at a time through the N^4 stages (one g' buffer + one workspace in HBM).
        ``stage_events``: optional dict that receives, per stage name ("rotation", "transform", "energy",
        "fock_gradient", "hessian"), a list of (start, end) CUDA-event pairs recorded on the launching stream
        around the kernels of that stage (bench.py's roofline figures).
        ``on_result(b)`` is called after the kernels of evaluation ``b`` are enqueued (used to start
        the device->host copy of its Hessian while evaluation ``b+1`` computes).
        ``on_integrals(b, ints, F, g)`` is called with the :class:`MOIntegrals` of evaluation ``b``, its generalized
        Fock matrix ``F (1, ld, ld)`` and its gradient ``g (nk,)`` while they are valid: the next evaluation of the
        call reuses their buffer."""
        def staged(name, fn):
            if stage_events is None:
                return fn()
            ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
            ev[0].record()
            out = fn()
            ev[1].record()
            stage_events.setdefault(name, []).append(ev)
            return out

        Coao = oao_mo_coeff if oao_mo_coeff.dim() == 3 else oao_mo_coeff[None]
        if kappa is not None:
            kappa = self.dev(kappa).reshape(-1, self.nk)
            C = staged("rotation", lambda: self.mo_coeff(Coao, self.rotation(kappa, squarings)))
        else:
            C = self.mo_coeff(Coao)
        B = C.shape[0]
        d1 = self.dev(d1)
        d2 = self.dev(d2)
        E = torch.empty(B, dtype=F64, device=self.device)
        G = torch.empty(B, self.nk, dtype=F64, device=self.device)
        H = None
        if want_hessian:
            H = H_out if H_out is not None else torch.empty(B, self.nk, self.nk, dtype=F64, device=self.device)
        assert path == "class" or self.n_geom == 0, "geometry batches use the class path"
        if path == "class":
            chunk = self.class_chunk(B)
            cbuf = self._recycle("class")
            for lo in range(0, B, chunk):
                hi = min(B, lo + chunk)
                cbuf = staged("transform", lambda: self.class_integrals(C[lo:hi], out=cbuf, geo_lo=lo))
                d1b = d1[lo:hi] if d1.dim() == 3 else d1
                d2b = d2[lo:hi] if d2.dim() == 5 else d2

                def energy():
                    c0, c1, c2 = self.class_active_hamiltonian(cbuf, geo_lo=lo)
                    E[lo:hi] = self.energy(c0, c1, c2, d1b, d2b)
                staged("energy", energy)
                FI, FA, F, _, gv = staged("fock_gradient",
                                          lambda: self.class_fock_gradient(cbuf, d1b, d2b, want_matrix=False))
                G[lo:hi] = gv
                if want_hessian:
                    staged("hessian", lambda: self.class_hessian(cbuf, F, d1b, d2b, out=H[lo:hi]))
                if on_integrals is not None:
                    for b in range(lo, hi):
                        on_integrals(b, MOIntegrals(self, "class", cls=cbuf[b - lo:b - lo + 1]), F[b - lo:b - lo + 1],
                                     gv[b - lo])
                if on_result is not None:
                    for b in range(lo, hi):
                        on_result(b)
            self._park("class", cbuf)                        # a single-evaluation buffer is kept for reuse
            return E, G, H
        hs = self.int1e_transform(C)
        gbuf = self._recycle("full")
        for b in range(B):
            gbuf = staged("transform", lambda: self.int2e_transform(C[b:b + 1], out=gbuf))
            h1 = hs[b:b + 1]
            d1b = d1[b] if d1.dim() == 3 else d1
            d2b = d2[b] if d2.dim() == 5 else d2
            c0, c1, c2 = self.active_hamiltonian(h1, gbuf)
            E[b:b + 1] = self.energy(c0, c1, c2, d1b, d2b)
            FI, FA, F, _, gv = self.fock_gradient(h1, gbuf, d1b, d2b, want_matrix=False)
            G[b] = gv[0]
            if want_hessian:
                self.hessian(h1[0], gbuf[0], F[0], d1b, d2b, out=H[b])
            if on_integrals is not None:
                on_integrals(b, MOIntegrals(self, "full", h=h1, g=gbuf), F, gv[0])
            if on_result is not None:
                on_result(b)
        self._park("full", gbuf)
        return E, G, H

    # ------------------------------------------------------------------ CUDA-graph replay of whole evaluations
    GRAPH_CACHE = 8
    GRAPH_MAX_OUTPUT_BYTES = 256 << 20

    def evaluate_graphed(self, oao_mo_coeff, d1, d2, kappa=None, want_hessian=True, path="class", clone=True):
        """:meth:`evaluate` captured once per argument shape into a CUDA graph and replayed: one graph launch per
        call instead of ~40 kernel launches, for the launch-bound small bases (an evaluation at 7-43 orbitals is
        a few microseconds of kernels behind ~0.4 ms of launch overhead).  Inputs (device tensors, or host tensors
        copied asynchronously) are copied into the graph's static buffers; the returned E, G, H are fresh
        copies (``clone=False``: the graph's own output buffers, overwritten by the next call).  For N above the fused-expm limit the squaring count is decided on the host (one synchronisation)
        and is part of the graph key."""
        Coao = oao_mo_coeff if oao_mo_coeff.dim() == 3 else oao_mo_coeff[None]
        nb = max(Coao.shape[0], 1 if kappa is None else kappa.reshape(-1, self.nk).shape[0])
        if want_hessian and nb * self.nk * self.nk * 8 > self.GRAPH_MAX_OUTPUT_BYTES:
            # a graph pins its output buffers for its lifetime; work of this size is not launch-bound anyway
            return self.evaluate(Coao, self.dev(d1), self.dev(d2), kappa=None if kappa is None else self.dev(kappa),
                                 want_hessian=want_hessian, path=path)
        squarings = None
        if kappa is not None:
            kappa = kappa.reshape(-1, self.nk)
            if self.N > self.lib.oo_expm_device_squarings_max_n():
                squarings = self.squarings_for(kappa)
        key = ("graph", tuple(Coao.shape), None if kappa is None else kappa.shape[0], tuple(d1.shape),
               tuple(d2.shape), bool(want_hessian), path, squarings)
        graphs = self._ws.setdefault("graphs", {})
        entry = graphs.pop(key, None)
        if entry is None and key not in self._ws.setdefault("graph_seen", set()):
            # capturing costs ~40 ms (private memory pool): a shape is captured the second time it shows up
            self._ws["graph_seen"].add(key)
            return self.evaluate(Coao, self.dev(d1), self.dev(d2), kappa=None if kappa is None else self.dev(kappa),
                                 want_hessian=want_hessian, squarings=squarings, path=path)
        if entry is None:
            entry = self._capture_evaluation(Coao, d1, d2, kappa, want_hessian, path, squarings)
            while len(graphs) >= self.GRAPH_CACHE:
                graphs.pop(next(iter(graphs)))
        graphs[key] = entry                                   # most recently used last
        graph, static, out, _keep = entry
        for dst, src in zip(static, (Coao, d1, d2, kappa)):
            if dst is not None:
                dst.copy_(src, non_blocking=True)
        graph.replay()
        E, G, H = out
        if not clone:
            return E, G, H
        return E.clone(), G.clone(), (H.clone() if H is not None else None)

    def _capture_evaluation(self, Coao, d1, d2, kappa, want_hessian, path, squarings):
        mk = lambda t: None if t is None else torch.empty(tuple(t.shape), dtype=F64, device=self.device)
        static = [mk(Coao), mk(d1), mk(d2), mk(kappa)]
        for dst, src in zip(static, (Coao, d1, d2, kappa)):
            if dst is not None:
                dst.copy_(src)
        run = lambda: self.evaluate(static[0], static[1], static[2], kappa=static[3], want_hessian=want_hessian,
                                    squarings=squarings, path=path)
        self.eri_is_symmetric()                               # host-synchronising one-off decisions happen here,
        cur = torch.cuda.current_stream(self.device)          # not inside the capture
        # the graph gets a class / g' buffer of its own: it rewrites that buffer at every replay, so it must never
        # be one that the eager cache hands out to a lazy consumer (OrbitalHessian, a gradient's backward)
        eager = {k: self._icache.pop(k) for k in list(self._icache)}
        side = torch.cuda.Stream(self.device)
        side.wait_stream(cur)
        self._ws["capturing"] = True
        try:
            with torch.cuda.stream(side):
                for _ in range(2):                            # sizes every workspace outside the capture
                    run()
            cur.wait_stream(side)
            torch.cuda.synchronize(self.device)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                out = run()
        finally:
            self._ws["capturing"] = False
            self._ws.pop("chess_key", None)
        # the graph has the addresses of every workspace it touched baked in: keep those tensors alive even if
        # a later, larger call replaces them in the workspace table
        keep = ([v for v in self._ws.values() if torch.is_tensor(v)] + [self.g_packed, self.g_pairT]
                + [ent[1] for ent in self._icache.values()])
        self._icache = eager
        return graph, static, out, keep
