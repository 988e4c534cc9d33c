/*
 * oo_b200.h -- C ABI of the B200-native orbital-optimization hot path.
 *
 * The reference (Emieeel/auto_oo) has no FFI boundary: the path lives behind
 * Python methods of `OO_energy` (src/auto_oo/oo_energy.py:121-474) and the free
 * functions in oo_energy.py:21-118 / utils/active_space.py:111-212, whose
 * arithmetic is dispatched to torch CPU ops.  Each entry point below replaces
 * one group of those call sites; the citation says which.  INTEGRATION.md shows
 * the ctypes stub a maintainer of the reference would add.
 *
 * Conventions (all entry points)
 *  - plain pointers and sizes only; every pointer is a DEVICE pointer unless
 *    the name ends in `_host`; all data are float64, row-major.
 *  - N  = number of orbitals (logical), ld = padded leading dimension used for
 *    EVERY axis of every N-sized tensor (ld even, ld >= N; rows/cols N..ld-1
 *    must be zero on input and are zero on output).  A 4-index tensor is
 *    ld*ld*ld*ld doubles.
 *  - orbital classes are the contiguous ranges occ [0,no), act [no,no+na),
 *    virt [no+na,N)  (reference moldata_pyscf.py:42-56).
 *  - the caller owns every buffer, including workspaces (size from
 *    oo_workspace_bytes); the library never allocates, frees or retains them.
 *  - all work is enqueued on `stream` (a cudaStream_t); no host sync, so calls
 *    may be captured into a CUDA graph.
 *  - return 0 on success, a negative OO_ERR_* code otherwise (oo_error_string).
 */
#ifndef OO_B200_H
#define OO_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OO_ABI_VERSION 2

enum {
    OO_OK = 0,
    OO_ERR_INVALID_ARG = -1,   /* null pointer, negative size, odd ld, ...        */
    OO_ERR_UNSUPPORTED = -2,   /* size outside what the kernels were built for     */
    OO_ERR_WORKSPACE   = -3,   /* workspace too small                              */
    OO_ERR_CUDA        = -4,   /* a CUDA runtime/driver call failed (see oo_last_cuda_error) */
    OO_ERR_NO_DEVICE   = -5    /* no sm_100 device / driver entry point missing    */
};

/* workspace selectors for oo_workspace_bytes */
enum {
    OO_WS_ROTATION   = 1,      /* oo_kappa_rotation_f64                            */
    OO_WS_INT2E      = 2,      /* oo_int2e_transform_f64                           */
    OO_WS_HESSIAN    = 3,      /* oo_hessian_f64                                   */
    OO_WS_INT1E      = 4,      /* oo_int1e_transform_f64 / oo_mo_coeff_f64         */
    OO_WS_YMATRIX    = 5,      /* oo_y_matrix_f64                                  */
    OO_WS_CLASS_TRANSFORM = 6, /* oo_class_transform_f64 (nI = no+na)              */
    OO_WS_CLASS_BUFFER    = 7, /* size of the class buffer `cls` (x batch)         */
    OO_WS_CLASS_HESSIAN   = 8, /* oo_class_hessian_f64: pass N = na (!), nI = no+na, batch */
    OO_WS_CLASS_TRANSFORM_SYM = 9, /* oo_class_transform_sym_f64 (nI = no+na)      */
    OO_WS_CLASS_HESSIAN_VECTOR = 10, /* oo_class_hessian_vector_f64: pass N = na (!), nI = no+na, batch = nv */
    OO_WS_HESSIAN_VECTOR  = 11, /* oo_hessian_vector_f64: pass N = na (!), nI = no+na, batch = nv   */
    OO_WS_HESSIAN_DIAGONAL = 12, /* oo_hessian_diagonal_f64 (nI = no+na); oo_class_hessian_diagonal_f64
                                   needs no workspace                                              */
    OO_WS_KRYLOV = 13          /* oo_davidson_expand_f64 / oo_pcg_step_f64: pass N = n (vector length), nI = k
                                  (largest basis, <= 64), ld = batch = 1                                        */
};

int         oo_abi_version(void);
const char *oo_error_string(int code);
int         oo_last_cuda_error(void);                 /* cudaError_t of the last OO_ERR_CUDA */
unsigned long long oo_launch_count(void);             /* kernels launched by this library so far */

/* per-call variant switches (A/B timing and tests), OR-ed into the `flags` argument of the entry points that
 * have more than one implementation; every setting gives the same numbers to round-off.  There is no
 * process-wide mutable state: two threads driving different streams can use different flags.             */
enum {
    OO_FLAG_HESSIAN_DENSE = 1,                 /* oo_class_hessian_f64 / oo_hessian_f64: ONE dense GEMM over all of At
                                                  instead of the block form (C-block GEMM + G blocks + ELL remainder) */
    OO_FLAG_HESSIAN_ASSEMBLE_PER_ELEMENT = 2,  /* Hessian assembly: always one thread per element (default: that form
                                                  for N <= 64, row-tiled + bulk-async streamed above)                 */
    OO_FLAG_HESSIAN_ASSEMBLE_TILED = 4,        /* Hessian assembly: always the row-tiled form                         */
    OO_FLAG_CLASS_UNFUSED_PACK = 8,            /* oo_class_transform_sym_f64: separate pack / expand passes instead of
                                                  the fused epilogues of its quarter-2 / last-quarter GEMMs           */
    OO_FLAG_HESSIAN_GROUP_UNSTREAMED = 16,     /* G blocks of the Hessian T-matrix with per-thread loads instead of the
                                                  cp.async.bulk + mbarrier streamed DMMA kernel                       */
    OO_FLAG_HESSIAN_ASSEMBLE_UNSTREAMED = 32,  /* Hessian assembly without the bulk-async streamed kernel for the rows
                                                  outside occ+act                                                     */
    OO_FLAG_CLASS_Q2_RECTANGULAR = 64,         /* oo_class_transform_sym_f64: quarter 2 as the rectangular TN-GEMM that
                                                  computes every class pair (m, n) and keeps n <= m in its epilogue,
                                                  instead of the triangular kernel that only computes n <= m          */
    OO_FLAG_HESSIAN_REUSE_OPERANDS = 256,      /* oo_class_hessian_f64: same RDMs, pair list, batch and workspace as the
                                                  previous call -- the sparse table, the C-block coefficients and the
                                                  pair runs it left in the workspace are used again (a kappa sweep at
                                                  fixed RDMs rebuilds nothing that does not depend on the integrals)  */
    OO_FLAG_CLASS_DIRECT_STORES = 512,         /* oo_class_transform_sym_f64: the consumer warps of its GEMMs store their
                                                  accumulators themselves instead of staging the tile in shared memory
                                                  for the warps that ship it with bulk asynchronous copies            */
    OO_FLAG_HESSIAN_SPMM_UNPAIRED = 1024,      /* oo_class_hessian_f64: the occ-occ off-diagonal columns of the T-matrix one
                                                  by one (generic ELL SpMM) instead of in pairs that share their rows   */
    OO_FLAG_CLASS_Q1_UNPAIRED = 2048,          /* oo_class_transform_sym_f64: every evaluation of a batch through its
                                                  own quarter-1 GEMM, also when two narrow class ranges (2 nIp <= 48
                                                  columns) would share one                                              */
    OO_FLAG_CLASS_ERI_8FOLD = 128              /* oo_class_transform_sym_f64: `g_packed` is the 8-FOLD packed tensor of
                                                  oo_pack_eri_8fold_f64 (an eighth of N^4) instead of the pair-packed
                                                  one (half of N^4); quarter 1 unpacks it in its producer               */
};
/* oo_class_transform_sym_f64 only: run just the selected GEMM stages (k = 0: quarter 1 over packed pairs; 1, 2, 3:
 * quarters 2-4 of the Coulomb class; 4, 5, 6: of the exchange class) on the intermediates a complete call left in
 * the workspace.  Lets a caller time one kernel with events on both sides (bench.py); no stage bit = all stages. */
#define OO_FLAG_CLASS_STAGE(k) (1u << (16 + (k)))
int         oo_device_info(int *sm_count, int *cc_major, int *cc_minor);
size_t      oo_workspace_bytes(int which, int N, int ld, int nI, int batch);

/* ---- dense building block -------------------------------------------------
 * C[b][m][n] = sum_k At[b][k][m] * B[b][k][n]     (both operands K-major)
 * TMA (cp.async.bulk.tensor, 128B swizzle) -> smem ring -> FP64 DMMA.
 * lda/ldb/ldc in elements (even); stride* = per-batch element strides, 0 = shared.
 * Exposed because the 4-index transform and the Hessian Y-matrix are this GEMM. */
int oo_dgemm_tn_f64(const double *At, const double *B, double *C,
                    int64_t M, int64_t N, int64_t K,
                    int64_t lda, int64_t ldb, int64_t ldc,
                    int batch, int64_t strideA, int64_t strideB, int64_t strideC,
                    void *stream);

/* same product with M = d0*d1*d2 rows (a b c), additionally storing the rows in the order
 * (c b a) into C2 (same ldc): the first quarter of the class transform needs both layouts.   */
int oo_dgemm_tn_swap02_f64(const double *At, const double *B, double *C, double *C2,
                           int d0, int d1, int d2, int64_t N, int64_t K,
                           int64_t lda, int64_t ldb, int64_t ldc, void *stream);

/* general small batched product with fused epilogue (expm, C^T h C, X C U):
 * D[b] = alpha * op(A[b]) op(B[b]) + beta * E[b] + gamma * I ; op = transpose if trans* != 0;
 * E may be NULL (beta ignored) and may alias D.                                 */
int oo_dgemm_small_f64(int transA, int transB, int M, int N, int K,
                       double alpha, const double *A, int lda, int64_t strideA,
                       const double *B, int ldb, int64_t strideB,
                       double beta, const double *E, int lde, int64_t strideE,
                       double gamma, double *D, int ldd, int64_t strideD,
                       int batch, void *stream);

/* ---- K1: kappa -> U = expm(-K(kappa)) --------------------------------------
 * replaces oo_energy.py:213-219 (kappa_vector_to_matrix), :63-87
 * (vector_to_skew_symmetric) and :226-230 (math.expm(-kappa_matrix)).
 * kappa[b][nk]; pair_l/pair_r[nk] = (row, col) of each non-redundant parameter
 * (row > col): K[l,r] = +kappa, K[r,l] = -kappa.  `squarings` >= ceil(log2(||K||_1/0.95))
 * (host-chosen; degree-18 Taylor polynomial of -K/2^s by Paterson-Stockmeyer, s squarings).
 * N <= oo_expm_device_squarings_max_n(): the whole chain is ONE launch (N <= 64: one CTA per matrix out of
 * shared memory; N <= 256: one cooperative grid, a grid barrier between the products), and `squarings` = -1
 * lets the kernel apply the same rule on the device (per matrix for N <= 64, the maximum over the batch
 * above; no host round trip).
 * U[b] is ld x ld.  ws: oo_workspace_bytes(OO_WS_ROTATION, N, ld, 0, batch).      */
int oo_kappa_rotation_f64(const double *kappa, const int32_t *pair_l, const int32_t *pair_r,
                          int nk, int N, int ld, int batch, int squarings,
                          double *U, void *ws, size_t ws_bytes, void *stream);

/* largest N for which `squarings` = -1 is accepted: 256 (64 with the environment variable
 * OO_OPT_EXPM_MULTI_LAUNCH, 0 with OO_OPT_EXPM_UNFUSED; both kept for A/B tests)       */
int oo_expm_device_squarings_max_n(void);

/* expm(sign * A) of arbitrary (not nec. skew) ld x ld matrices with ||A||_1 <= 0.95 * 2^squarings */
int oo_expm_f64(const double *A, double sign, int N, int ld, int batch, int squarings,
                double *U, void *ws, size_t ws_bytes, void *stream);

/* ---- K1 epilogue / K2a ------------------------------------------------------
 * C'[b] = X * Coao[b] * U[b]          (oo_energy.py:173-176 mo_coeff, :201/:235)
 * strideX / strideCoao / strideU = 0 shares the matrix across the batch (strideX != 0:
 * one orthogonaliser per geometry); U may be NULL.                               */
int oo_mo_coeff_f64(const double *X, int64_t strideX, const double *Coao, int64_t strideCoao,
                    const double *U, int64_t strideU, int N, int ld, int batch,
                    double *Cout, void *ws, size_t ws_bytes, void *stream);

/* h'[b] = C[b]^T h C[b]               (oo_energy.py:44-46 int1e_transform)      */
int oo_int1e_transform_f64(const double *h_ao, int64_t stride_h, const double *C, int64_t strideC,
                           int N, int ld, int batch, double *h_mo,
                           void *ws, size_t ws_bytes, void *stream);   /* stride_h != 0: h per geometry */

/* ---- K2b: four-index transform ---------------------------------------------
 * g'[i,j,k,l] = sum_pqrs C0[p,i] C1[q,j] C2[r,k] C3[s,l] g[p,q,r,s]
 * replaces oo_energy.py:21-30 (general_4index_transform), :33-41, :49-51.
 * Four quarter transforms, each one TN-DGEMM [ld^3 x ld] = [ld x ld^3]^T [ld x ld]
 * that rotates the transformed index to the back, so after four quarters the
 * layout is [i,j,k,l] again.  strideG = 0 shares g_ao over the batch
 * (kappa sweep); strideC = per-batch stride of each C matrix.
 * ws: oo_workspace_bytes(OO_WS_INT2E, N, ld, 0, batch) = batch * ld^4 doubles.  */
int oo_int2e_transform_f64(const double *g_ao, int64_t strideG,
                           const double *C0, const double *C1, const double *C2,
                           const double *C3, int64_t strideC,
                           int N, int ld, int batch, double *g_mo,
                           void *ws, size_t ws_bytes, void *stream);

/* ---- K3: active-space Hamiltonian and energy -------------------------------
 * c0 = e_nuc + 2 sum_i h_ii + 2 sum_ij g_iijj - sum_ij g_ijji
 * c1_tu = h_tu + sum_i (2 g_tuii - g_tiiu) ; c2_tuvw = g_tuvw / 2
 * replaces utils/active_space.py:111-174 and :177-212.
 * c0[b], c1[b][na*na], c2[b][na^4] (dense, no padding).                          */
int oo_active_hamiltonian_f64(const double *h_mo, const double *g_mo, int no, int na,
                              int N, int ld, int batch, double e_nuc, const double *e_nuc_batch,
                              double *c0, double *c1, double *c2, void *stream);
                              /* e_nuc_batch (device, batch doubles) overrides e_nuc when not NULL */

/* E[b] = c0[b] + <c1[b],gamma[b]> + <c2[b],Gamma[b]>   (oo_energy.py:194-197)
 * stride_rdm1/2 = 0 shares the RDMs across the batch.                            */
int oo_energy_f64(const double *c0, const double *c1, const double *c2,
                  const double *gamma, int64_t stride_rdm1,
                  const double *Gamma, int64_t stride_rdm2,
                  int na, int batch, double *E, void *stream);

/* ---- K3/K4: Fock matrices and orbital gradient ------------------------------
 * FI (oo_energy.py:272-284), FA (:286-298), generalized F (:238-270),
 * Gmat = 2 (F - F^T) (:300-309), gvec[j] = Gmat[pair_l[j], pair_r[j]] (:221-224, :90-94).
 * FI, FA, F, Gmat are ld x ld per batch; any of FA, Gmat, gvec may be NULL.      */
int oo_fock_gradient_f64(const double *h_mo, const double *g_mo,
                         const double *gamma, int64_t stride_rdm1,
                         const double *Gamma, int64_t stride_rdm2,
                         int no, int na, int N, int ld, int batch,
                         const int32_t *pair_l, const int32_t *pair_r, int nk,
                         double *FI, double *FA, double *F, double *Gmat, double *gvec,
                         void *stream);

/* adjoint of (gamma, Gamma) -> Gmat, needed by jacobian(orbital_gradient, theta)
 * (oo_pqc.py:113-123): given Gbar (ld x ld), with Fbar = 2 (Gbar - Gbar^T):
 * gbar1_vw = sum_{i,n} Fbar_in 2 (g_nivw - g_nwvi / 2) + sum_n Fbar_vn FI_nw
 * gbar2_vwxy = sum_n Fbar_vn g_nwxy                                             */
int oo_fock_gradient_vjp_f64(const double *g_mo, const double *FI, const double *Gbar,
                             int no, int na, int N, int ld,
                             double *gbar1, double *gbar2, void *stream);

/* ---- K4: orbital Hessian -----------------------------------------------------
 * H[j][k] = Hfull[l_j, r_j, l_k, r_k], Hfull = (1-P_pq)(1-P_rs)(2 gf_pr h_qs
 * - (F_pr + F_rp) d_qs + 2 Y_pqrs)  -- oo_energy.py:311-340 (analytic_hessian_from_integrals),
 * :342-379 (full_rdms), :381-393 (y_matrix), :395-402 (full_hessian_to_matrix).
 * Evaluated in the I = occ+act index space (the full-space RDMs vanish outside
 * it): T[(p r),(q s)] = sum_(m n) A[(m n),(p r)] B[(m n),(q s)] is one TN-DGEMM of
 * size nI^2 x ld^2 x (2 nI^2 + 1), followed by a fused 4-term assembly.
 * F is the generalized Fock matrix from oo_fock_gradient_f64.  H is nk x nk.
 * ws: oo_workspace_bytes(OO_WS_HESSIAN, N, ld, no+na, 1).                         */
int oo_hessian_f64(const double *h_mo, const double *g_mo, const double *F,
                   const double *gamma, const double *Gamma,
                   int no, int na, int N, int ld,
                   const int32_t *pair_l, const int32_t *pair_r, int nk,
                   double *H, void *ws, size_t ws_bytes, unsigned flags, void *stream);

/* ---- partial ("class") transform path -------------------------------------------
 * Energy, gradient and the I-space Hessian read g' only through two classes with two
 * indices in I = occ+act:  J[m,n,a,b] = g'[a,b,m,n]  and  K[n,m,a,b] = g'[a,m,n,b]
 * (m,n < nIp = nI rounded up to even; a,b general).  oo_class_transform_f64 computes just
 * these (2 N^4 nI + 12 N^3 nI^2 flop instead of 8 N^5) with the same TN-DGEMM kernel, from
 * the PAIR-TRANSPOSED AO tensor g_pairT[r,s,p,q] = g[p,q,r,s] (oo_transpose_f64 on the
 * ld^2 x ld^2 matrix, once per problem; no symmetry of g is assumed).  Replaces, for the
 * callers of oo_energy.py:204-211, :404-424, the int2e_transform of oo_energy.py:49-51.
 * `cls` = [K rows (nIp^2) ; J rows (nIp^2) ; h' row], rows of ld^2 doubles
 * (oo_workspace_bytes(OO_WS_CLASS_BUFFER, N, ld, nI, batch)); the caller writes h' = C^T h C
 * into the last row with oo_int1e_transform_f64.  The oo_class_* entry points below are the
 * class-buffer forms of oo_active_hamiltonian_f64 / oo_fock_gradient_f64 /
 * oo_fock_gradient_vjp_f64 / oo_hessian_f64 (same outputs, same reference lines).      */
int oo_transpose_f64(const double *src, double *dst, int64_t rows, int64_t cols, void *stream);
int oo_class_transform_f64(const double *g_pairT, int64_t strideG, const double *C, int64_t strideC,
                           int N, int ld, int nIp, int batch, double *cls, void *ws, size_t ws_bytes,
                           void *stream);   /* stride 0 = shared over the batch; cls[b] contiguous */

/* Symmetric variant of the class transform, for AO integrals with the 8-fold symmetry
 * (pq|rs) = (qp|rs) = (rs|pq) that every real-orbital ERI tensor has (PySCF int2e,
 * moldata_pyscf.py:31).  oo_eri_symmetry_defect_f64 writes defect3 = { max |g_pqrs - g_qprs|,
 * max |g_pqrs - g_rspq|, max |g| } (device) so the caller can decide; oo_pack_eri_pairs_f64 builds
 * g_packed[r,s,pq] = g[r,s,p,q], p >= q, pq = p(p+1)/2 + q over the ld PADDED orbitals, row length
 * oo_pair_ld(ld) = ld(ld+1)/2 rounded up to even, padding zero (half the HBM of the full tensor).
 * oo_class_transform_sym_f64 fills the same class buffer as oo_class_transform_f64 with
 * N^4 nI + ~7 N^3 nI^2 flop: quarter 1 runs over packed pairs only (its epilogue unpacks the pair
 * for the exchange class), and only class pairs m >= n go through the last two quarters
 * (J[m,n,a,b] = J[n,m,a,b], K[n,m,a,b] = K[m,n,b,a]).  ws: OO_WS_CLASS_TRANSFORM_SYM.            */
int     oo_eri_symmetry_defect_f64(const double *g_ao, int ld, double *defect3, void *stream);
int64_t oo_pair_ld(int ld);
int     oo_pack_eri_pairs_f64(const double *g_ao, double *g_packed, int ld, void *stream);
/* g_packed8[RS][PQ] = g[r,s,p,q], r >= s, p >= q, RS = r(r+1)/2 + s, PQ = p(p+1)/2 + q over the ld padded orbitals:
 * ld(ld+1)/2 rows of oo_pair_ld(ld) doubles, an eighth of the full tensor (8.7 GB instead of 34.4 GB at N = 256).
 * With OO_FLAG_CLASS_ERI_8FOLD the quarter-1 GEMM of oo_class_transform_sym_f64 reads this layout directly: the
 * k-row r of the tile (s, PQ-range) is row RS(max(r,s), min(r,s)), fetched by one bulk copy; tiles that share a
 * PQ panel run together so the second use of every row (as (r,s) and as (s,r)) comes from L2.   (SURVEY 8f row 4) */
int     oo_pack_eri_8fold_f64(const double *g_ao, double *g_packed8, int ld, void *stream);
int     oo_class_transform_sym_f64(const double *g_packed, int64_t strideG, const double *C, int64_t strideC,
                                   int N, int ld, int nIp, int batch, double *cls, void *ws, size_t ws_bytes,
                                   unsigned flags, void *stream);
/* Sharded evaluation (SURVEY 8e, second decomposition): every rank holds a SLAB of the pair columns of the 8-fold
 * packed tensor, g_packed8_slab[RS][j] = g8[RS][pq_lo + j], j < pq_cnt, row pitch slab_ld (pq_lo, pq_cnt, slab_ld
 * even).  Quarter 1 and the Coulomb quarter 2 run over the slab only; all later steps are linear in the quarter-1
 * result, so `cls` receives this slab's ADDITIVE share of the K and J rows of the class buffer: the caller sums the
 * shares over the ranks (one NCCL all-reduce over NVLink) and then writes the h' row.  Same workspace as
 * oo_class_transform_sym_f64.                                                                                */
int oo_class_transform_sym_slab_f64(const double *g_packed8_slab, int64_t slab_ld, int64_t pq_lo, int64_t pq_cnt,
                                    const double *C, int64_t strideC, int N, int ld, int nIp, int batch, double *cls,
                                    void *ws, size_t ws_bytes, unsigned flags, void *stream);
int oo_class_active_hamiltonian_f64(const double *cls, int no, int na, int N, int ld, int nIp,
                                    int batch, double e_nuc, const double *e_nuc_batch, double *c0,
                                    double *c1, double *c2, void *stream);
int oo_class_fock_gradient_f64(const double *cls, const double *gamma, int64_t stride_rdm1,
                               const double *Gamma, int64_t stride_rdm2, int no, int na, int N,
                               int ld, int nIp, int batch, const int32_t *pair_l,
                               const int32_t *pair_r, int nk, double *FI, double *FA, double *F,
                               double *Gmat, double *gvec, void *stream);
int oo_class_fock_gradient_vjp_f64(const double *cls, const double *FI, const double *Gbar, int no,
                                   int na, int N, int ld, int nIp, double *gbar1, double *gbar2,
                                   void *stream);
int oo_class_hessian_f64(const double *cls, const double *F, const double *gamma, int64_t stride_rdm1,
                         const double *Gamma, int64_t stride_rdm2, int no, int na, int N, int ld,
                         int nIp, int batch, const int32_t *pair_l, const int32_t *pair_r, int nk,
                         double *H, void *ws, size_t ws_bytes, unsigned flags, void *stream);
                         /* batched: cls[b], F[b] (ld^2), H[b] (nk^2) contiguous per evaluation */

/* ---- K4, matrix free: Hessian-vector products and the Hessian diagonal ------------------------------------
 * The same H as oo_class_hessian_f64 / oo_hessian_f64 (oo_energy.py:311-340, :342-379, :381-393, :395-402) for
 * ONE evaluation, without forming it or the T-matrix.  V and HV are nk x nv, row-major: HV = H V.  With V the
 * skew matrix of a vector (V[l_j, r_j] = v_j = -V[r_j, l_j]),
 *   W[p,q] = -((F + F^T) V)[p,q] + [p in I] sum_{r in I, s} T[(p r),(q s)] V[r,s],   (H v)_j = W[l_j,r_j] - W[r_j,l_j],
 * and the T part is one streamed pass over the class planes per block of up to 8 vectors (DMMA on each plane times
 * the rows of At V it meets); larger nv is processed in blocks.  diag[j] = H[j][j] is a dot product of four
 * columns of At with the class planes.  Every reduction runs in a fixed order: identical calls give identical
 * bits.  Every unordered pair (pair_l[j], pair_r[j]) must occur at most once, pair_l[j] != pair_r[j].
 * ws: oo_workspace_bytes(OO_WS_CLASS_HESSIAN_VECTOR, na, ld, no+na, nv) (pass N = na); the class diagonal needs
 * no workspace (ws may be NULL).  The (h_mo, g_mo) forms first gather the class layout out of the complete g'
 * into their workspace (OO_WS_HESSIAN_VECTOR with N = na and batch = nv, OO_WS_HESSIAN_DIAGONAL).             */
int oo_class_hessian_vector_f64(const double *cls, const double *F, const double *gamma, const double *Gamma,
                                int no, int na, int N, int ld, int nIp, const int32_t *pair_l,
                                const int32_t *pair_r, int nk, const double *V, int nv, double *HV,
                                void *ws, size_t ws_bytes, void *stream);
int oo_class_hessian_diagonal_f64(const double *cls, const double *F, const double *gamma, const double *Gamma,
                                  int no, int na, int N, int ld, int nIp, const int32_t *pair_l,
                                  const int32_t *pair_r, int nk, double *diag, void *ws, size_t ws_bytes,
                                  void *stream);
int oo_hessian_vector_f64(const double *h_mo, const double *g_mo, const double *F, const double *gamma,
                          const double *Gamma, int no, int na, int N, int ld, const int32_t *pair_l,
                          const int32_t *pair_r, int nk, const double *V, int nv, double *HV,
                          void *ws, size_t ws_bytes, void *stream);
int oo_hessian_diagonal_f64(const double *h_mo, const double *g_mo, const double *F, const double *gamma,
                            const double *Gamma, int no, int na, int N, int ld, const int32_t *pair_l,
                            const int32_t *pair_r, int nk, double *diag, void *ws, size_t ws_bytes,
                            void *stream);

/* ---- Krylov arithmetic between products: lowest Hessian eigenpair (Davidson-Liu) and shifted Newton solve (PCG) ----
 * The products themselves are oo_class_hessian_vector_f64 / oo_hessian_vector_f64; these entry points are the solver
 * arithmetic between them (auto_oo_b200/krylov.py drives them).  Vectors have length n; a Davidson basis is stored
 * as ROWS Vt[j][0..n) (row pitch ldv), with its products HVt[j] = H Vt[j].  Every reduction runs in a fixed order
 * (per-CTA block sums, then the CTA partials in CTA order): identical calls give identical bits; no host sync.
 *
 *  oo_subspace_eigh_f64     eigenvalues (ascending) w[b][0..k) and eigenvectors Y[b] (column j of the k x k
 *                           row-major Y, pitch ldy, belongs to w[j]) of `batch` symmetric k x k matrices S[b] (pitch
 *                           lds; the lower triangle is read), k <= 64: one CTA per matrix, cyclic Jacobi in shared
 *                           memory.
 *  oo_davidson_project_f64  out[j*inc] = Vt[j] . u for j < k (and out2[j*inc2] when out2 != NULL): the new row and
 *                           column of S = V^T H V after the product u = H Vt[m].
 *  oo_davidson_expand_f64   with y = column 0 of Y and theta = *theta (device): x = V^T y, hx = HV^T y,
 *                           r = hx - theta x, *rnorm = ||r||, t = r / (D - theta) with |D - theta| floored at `floor_`,
 *                           two-pass classical Gram-Schmidt of t against the basis, t / ||t|| -> Vt[k].  When k == kmax
 *                           the basis restarts first: Vt[0] = x, Vt[1] = the previous Ritz vector (yprev, kept by the
 *                           previous call) made orthonormal to x, HVt[0..1] and S[0..1][0..1] to match, t -> Vt[2].
 *                           Vt, HVt need kmax rows, S is kmax x kmax (pitch lds), yprev kmax doubles (zero at first).
 *                           rnorm[0] = ||r||; rnorm[1] = 1 when the orthogonalised correction vanished against the
 *                           basis (breakdown: the new row is written as zeros), else 0.
 *  oo_pcg_step_f64          deflated preconditioned CG on (H + shift) x = b with preconditioner D + shift (> 0) and the
 *                           deflation vector w, aw = (H + shift) w (both NULL: plain PCG).  init != 0: r holds b on
 *                           entry; x = w (w.b)/(w.aw), r = b - aw (w.b)/(w.aw), p = z - w (aw.z)/(w.aw), Ap unused.
 *                           init == 0: Ap = H p (no shift): alpha = (r.z)/(p.(Ap + shift p)), x += alpha p,
 *                           r -= alpha (Ap + shift p), z = r / (D + shift), p = z + beta p - w (aw.z)/(w.aw).
 *                           state[0..1] carries r.z and w.aw between calls; *rnorm = ||r||.
 * ws: oo_workspace_bytes(OO_WS_KRYLOV, n, 1, kmax, 1).  k > 64, null pointers and pitches below the length give
 * OO_ERR_INVALID_ARG, a short workspace OO_ERR_WORKSPACE, both before any launch.                                 */
int oo_subspace_eigh_f64(const double *S, int k, int lds, int64_t strideS, int batch, double *w, int64_t stridew,
                         double *Y, int ldy, int64_t strideY, void *stream);
int oo_davidson_project_f64(const double *Vt, int64_t ldv, int64_t n, int k, const double *u, double *out, int inc,
                            double *out2, int inc2, void *stream);
int oo_davidson_expand_f64(double *Vt, double *HVt, int64_t n, int64_t ldv, int k, int kmax, const double *Y, int ldy,
                           const double *theta, const double *D, double floor_, double *S, int lds, double *x,
                           double *hx, double *yprev, double *rnorm, void *ws, size_t ws_bytes, void *stream);
int oo_pcg_step_f64(int64_t n, const double *Ap, double shift, const double *D, const double *w, const double *aw,
                    double *x, double *r, double *p, double *state, double *rnorm, int init, void *ws, size_t ws_bytes,
                    void *stream);

/* Lower triangle (diagonal included) of `batch` symmetric n x n matrices, rows back to back in np.tril_indices(n)
 * order: packed[b][i(i+1)/2 + j] = H[b][i][j], j <= i.  The orbital Hessian of full_hessian_to_matrix
 * (oo_energy.py:395-402) is symmetric; shipping the triangle halves the device->host bytes per evaluation.   */
int oo_pack_lower_f64(const double *H, int n, int batch, double *packed, void *stream);

/* dst[i] = src[i], i < n, by a kernel.  `src` may be pinned host memory (cudaHostAlloc; read over PCIe through the
 * unified address space): the small per-call inputs of an evaluation (kappa, gamma, Gamma) reach the device
 * without a DMA-engine copy, which would otherwise queue behind the device->host copy of the previous Hessian. */
int oo_copy_f64(const double *src, double *dst, int64_t n, void *stream);

/* ---- RDMs from a state vector (SURVEY 8f row 3; the producer of the hot path's gamma, Gamma) -----
 * replaces Parameterized_circuit.get_rdms_from_state (pqc.py:192-218) with the operators of
 * utils/active_space.py:29-83 (restricted = spin-summed): gamma_pq = Re<psi|E_pq|psi>,
 * Gamma_pqrs = Re<psi|E_pq E_rs - delta_qr E_ps|psi>, Jordan-Wigner with qubit 0 the most significant
 * bit of the state index, spin orbitals 2p/2p+1 (up_then_down: p/p+ncas).
 * psi: 2^(2 ncas) amplitudes, float64 or interleaved complex128 (is_complex).
 *  oo_rdm_excitations_f64  Phi[k][c] (transposed=0, row length oo_rdm_columns(ncas)) or Phi[c][k]
 *                          (transposed=1) for the basis states x0 <= x < x0+nx: c = r*ncas+s -> (E_rs psi)[x],
 *                          c = ncas^2 -> psi[x], then zero padding; rows k = [Re x-chunk ; Im x-chunk].
 *  then  C = PhiL^T PhiR  with oo_dgemm_tn_f64 (k split over the batch argument),
 *  oo_rdm_accumulate_f64   acc += sum_b parts[b]      (fixed order),
 *  oo_rdm_assemble_f64     gamma_pq = C[ncas^2,(p q)], Gamma_pqrs = C[(q p),(r s)] - delta_qr gamma_ps.
 * With PhiL from u and PhiR from v the same calls give the transition form Re<u|O|v>; its adjoint
 *  (g1, g2, v) -> sum g1_pq E_pq v + sum g2_pqrs e_pqrs v  is
 *  oo_rdm_operator_matrix_f64  Mext[c][(p q)]  ((ncolp) x (ncas^2 rounded up to even)),
 *  Wt = Mext^T Phi_v^T (oo_dgemm_tn_f64 on the transposed Phi), and
 *  oo_rdm_apply_gather_f64     w[x] = sum_pq (E_pq Wt[pq])[x]   (Wt_im NULL for a real state).        */
int64_t oo_rdm_columns(int ncas);
int oo_rdm_excitations_f64(const double *psi, int is_complex, int ncas, int up_then_down,
                           int64_t x0, int64_t nx, int transposed, double *Phi,
                           const int32_t *xlist, int64_t nlist, void *stream);
int oo_rdm_accumulate_f64(const double *parts, int nparts, int64_t n, double *acc, void *stream);
int oo_rdm_assemble_f64(const double *C, int ncas, double *one_rdm, double *two_rdm, void *stream);
int oo_rdm_operator_matrix_f64(const double *g1, const double *g2, int ncas, double *Mext, void *stream);
int oo_rdm_apply_gather_f64(const double *Wt_re, const double *Wt_im, int ncas, int up_then_down,
                            int64_t R, int64_t ldW, const int32_t *xlist, const int32_t *pos,
                            double *w, void *stream);
/* Particle-number sectors (n_up, n_down) -> id n_up*(ncas+1)+n_down.  Every E_rs conserves both counts, so
 * all of the above can run on the COMPACT list of basis states of the sectors psi occupies (one sector for the
 * reference's number-conserving ansaetze: 5 % of the 4^ncas states at CAS(12,12)):
 *  oo_rdm_sector_flags_f64  flags[id] = 1 where psi has a non-zero amplitude (flags zeroed by the caller),
 *  oo_rdm_sector_mask       mask[x] = flags[id(x)]  (the caller turns it into xlist = nonzero(mask) and
 *                           pos = exclusive scan);  xlist/nlist above: rows are x = xlist[x0 + k] (zero rows past
 *                           nlist); apply_gather: R compact states, Wt row length ldW, column of x at pos[x],
 *                           w full length and zero-initialised.  xlist = pos = NULL: all 4^ncas states.          */
int oo_rdm_sector_flags_f64(const double *psi, int is_complex, int ncas, int up_then_down,
                            int32_t *flags, void *stream);
int oo_rdm_sector_mask(const int32_t *flags, int ncas, int up_then_down, int32_t *mask, void *stream);

/* ---- API-parity helpers (not on the hot path) ------------------------------
 * Dense full-space RDMs exactly as full_rdms defines them (oo_energy.py:342-379):
 * one_full N x N, two_full N^4 (dense, no padding).                               */
int oo_full_rdms_f64(const double *gamma, const double *Gamma, int no, int na, int N,
                     double *one_full, double *two_full, void *stream);

/* Y_pqrs = sum_mn [(G_pmrn + G_pmnr) g_qmns + G_prmn g_qsmn] for an ARBITRARY dense
 * two_full G (N^4, no padding) -- y_matrix, oo_energy.py:381-393.  g_mo is padded
 * (ld^4); Y is dense N^4.  ws: oo_workspace_bytes(OO_WS_YMATRIX, N, ld, 0, 1).       */
int oo_y_matrix_f64(const double *g_mo, const double *two_full, int N, int ld, double *Y,
                    void *ws, size_t ws_bytes, void *stream);

/* ---- layout helpers ----------------------------------------------------------
 * zero-padded copy between a dense N^rank tensor and its ld^rank padded image
 * (rank 2 or 4).  to_padded != 0: src dense -> dst padded (padding zeroed).     */
int oo_pad_copy_f64(const double *src, double *dst, int N, int ld, int rank,
                    int batch, int to_padded, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* OO_B200_H */
