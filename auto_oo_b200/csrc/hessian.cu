// K4-Hessian: analytic orbital Hessian reduced to the non-redundant kappa block.
//
// Reference: analytic_hessian_from_integrals (oo_energy.py:311-340) builds
//   X_pqrs = 2 gf_pr h_qs - (F_pr + F_rp) d_qs + 2 Y_pqrs,
//   Y_pqrs = sum_mn [(Gf_pmrn + Gf_pmnr) g_qmns + Gf_prmn g_qsmn]   (y_matrix, :381-393)
//   H_pqrs = X_pqrs - X_pqsr - X_qprs + X_qpsr,
// from full-space RDMs gf, Gf (full_rdms, :342-379) as dense N^4 tensors and three
// N^6 einsums, then gathers H[l_j, r_j, l_k, r_k] (full_hessian_to_matrix, :395-402).
//
// Here: Gf and gf vanish unless all their indices are in I = occ+act (nI = no+na),
// so Y and the gf (x) h term only exist for p, r in I.  With k = (m,n) in I x I:
//   T[(p r),(q s)] = sum_k At[k,(p r)] B[k,(q s)]
//     At[(m n),      (p r)] = 2 (Gf_pmrn + Gf_pmnr)     B[(m n),      (q s)] = g_qmns
//     At[nI^2+(m n), (p r)] = 2  Gf_prmn                B[nI^2+(m n), (q s)] = g_qsmn
//     At[2 nI^2,     (p r)] = 2  gf_pr                  B[2 nI^2,     (q s)] = h_qs
// is a product of size nI^2 x ld^2 x (2 nI^2 + 1), and
//   X(p,q,r,s) = -(F_pr + F_rp) d_qs + [p,r in I] T[(p r),(q s)]
// is combined four ways directly into the (nk x nk) output.
// B is the class buffer of classes.cu (or is gathered into that layout from the complete g').  At is not dense:
// it splits into the C block (one TN-DGEMM), one G block per occupied orbital (bulk-async streamed DMMA kernel)
// and an ELL remainder -- see "block structure of At" below; OO_FLAG_HESSIAN_DENSE keeps the single dense GEMM
// over all of At for A/B tests.  The assembly is row-tiled and, for the rows outside I, streamed with bulk copies.
#include <stdlib.h>

#include "common.cuh"

namespace oo {


int dgemm_tn(const double *At, const double *B, double *C, int64_t M, int64_t N, int64_t K,
             int64_t lda, int64_t ldb, int64_t ldc, int batch, int64_t strideA, int64_t strideB,
             int64_t strideC, cudaStream_t stream);

namespace {

struct RdmView {
    const double *d1, *d2;
    int no, na;
};

// full-space 1-RDM on I x I  (oo_energy.py:359-361)
__device__ __forceinline__ double gf1(const RdmView &r, int p, int q) {
    if (p >= r.no + r.na || q >= r.no + r.na) return 0.0;
    if (p < r.no || q < r.no) return (p == q) ? 2.0 : 0.0;
    return r.d1[(p - r.no) * r.na + (q - r.no)];
}

// full-space 2-RDM on I^4  (oo_energy.py:363-378)
__device__ __forceinline__ double gf2(const RdmView &r, int p, int q, int s, int t) {
    const int no = r.no, na = r.na;
    const int nI = no + na;
    if (p >= nI || q >= nI || s >= nI || t >= nI) return 0.0;
    const bool op = p < no, oq = q < no, os = s < no, ot = t < no;
    const int code = (op ? 8 : 0) | (oq ? 4 : 0) | (os ? 2 : 0) | (ot ? 1 : 0);
    switch (code) {
        case 15:  // occ occ occ occ : 4 d_pq d_st - 2 d_pt d_qs
            return (p == q && s == t ? 4.0 : 0.0) - (p == t && q == s ? 2.0 : 0.0);
        case 12:  // occ occ act act : 2 gamma_st d_pq
            return p == q ? 2.0 * r.d1[(s - no) * na + (t - no)] : 0.0;
        case 3:   // act act occ occ : 2 gamma_pq d_st
            return s == t ? 2.0 * r.d1[(p - no) * na + (q - no)] : 0.0;
        case 9:   // occ act act occ : -gamma_qs d_pt
            return p == t ? -r.d1[(q - no) * na + (s - no)] : 0.0;
        case 6:   // act occ occ act : -gamma_tp d_qs
            return q == s ? -r.d1[(t - no) * na + (p - no)] : 0.0;
        case 0:   // act act act act
            return r.d2[(((int64_t)(p - no) * na + (q - no)) * na + (s - no)) * na + (t - no)];
        default:
            return 0.0;
    }
}

// At rows: [0,nI^2) exchange-type, [nI^2, 2nI^2) Coulomb-type, 2nI^2: one-body.  lda >= nI^2 (even).
// nI here is the ROW STRIDE of the I-space (nI for the full-tensor path, nIp for the class path;
// gf1/gf2 return 0 for indices beyond occ+act).  swap_exch: exchange rows are ordered (n,m)
// instead of (m,n) -- the order in which classes.cu stores K[n,m,a,b].
// At[k, (p r)]: k < nI^2 exchange row (m,n) -- or (n,m) when swap_exch --, k < 2 nI^2 Coulomb row (m,n),
// k = 2 nI^2 the one-body row.  `mn` receives the (m, n) the row stands for (-1 for the one-body row).
__device__ __forceinline__ double at_value(const RdmView &rdm, int nI, int swap_exch, int64_t k, int p, int r,
                                           int &m, int &n) {
    const int nI2 = nI * nI;
    if (k < nI2) {
        const int k1 = (int)(k / nI), k2 = (int)(k % nI);
        m = swap_exch ? k2 : k1;
        n = swap_exch ? k1 : k2;
        return 2.0 * (gf2(rdm, p, m, r, n) + gf2(rdm, p, m, n, r));
    }
    if (k < 2 * nI2) {
        const int kk = (int)(k - nI2);
        m = kk / nI;
        n = kk % nI;
        return 2.0 * gf2(rdm, p, r, m, n);
    }
    m = n = -1;
    return 2.0 * gf1(rdm, p, r);
}

__global__ void hess_build_at_kernel(RdmView rdm, int nI, int swap_exch, int64_t lda, double *__restrict__ At) {
    const int nI2 = nI * nI;
    const int64_t total = (int64_t)(2 * nI2 + 1) * lda;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        const int64_t k = i / lda;
        const int col = (int)(i % lda);
        double v = 0.0;
        int m, n;
        if (col < nI2) v = at_value(rdm, nI, swap_exch, k, col / nI, col % nI, m, n);
        At[i] = v;
    }
}

// ---- block structure of At (class path) -------------------------------------------------------
// The full-space 2-RDM is a dense na^4 block plus Kronecker-delta core blocks (full_rdms,
// oo_energy.py:356-379), so At = [dense blocks] + [O(1) entries per column]:
//   C block  columns: the na^2 act-act pairs (t u) and the no occupied diagonal pairs (i i);
//            rows:    exchange / Coulomb rows of the act-act pairs and of the occupied diagonal pairs, one-body row
//            (Gamma_tuvw, and the delta_ij gamma / delta_ij delta_kl terms summed over a whole class)
//            -> ONE TN-DGEMM  Tc = Atc^T Bc  on the tensor pipe                    (~4 (na^2+no)^2 N^2 flop)
//   G block of every occupied i   columns: (i t) and (t i), t active;
//            rows: exchange / Coulomb rows at the positions (i u) and (u i), u active (the gamma_tu delta_ij terms)
//            -> hess_group_kernel: the 4 na rows are read once per column chunk, 2 na x 4 na coefficients in smem
//   rest     (occ-occ pairs i != j: three entries per column) -> ELL SpMM (hess_spmm_kernel), which also adds
//            whatever a column of the two blocks has outside its block (nothing for the reference's RDM layout).
// Every coefficient comes from the same at_value() as the all-dense route; a row k is identified by its
// position pair (a, b) = ((k mod nIs^2) / nIs, (k mod nIs^2) mod nIs), which makes the row sets independent of
// the storage order of the exchange rows.
struct Blocks {
    int no, na, nIs;
    __device__ __host__ int ncol_c() const { return na * na + no; }
    __device__ __host__ int nrow_c() const { return 2 * (na * na + no) + 1; }
    __device__ __host__ int ncol_g() const { return 2 * na; }
    __device__ __host__ int nrow_g() const { return 4 * na; }
    // column cc of the C block -> (p, r)
    __device__ void col_c(int cc, int &p, int &r) const {
        if (cc < na * na) { p = no + cc / na; r = no + cc % na; } else { p = r = cc - na * na; }
    }
    // row kc of the C block -> row of At / B
    __device__ int64_t row_c(int kc) const {
        const int nC = na * na + no;
        const int64_t nI2 = (int64_t)nIs * nIs;
        if (kc >= 2 * nC) return 2 * nI2;
        const int j = kc % nC;
        const int a = j < na * na ? no + j / na : j - na * na, b = j < na * na ? no + j % na : j - na * na;
        return (kc >= nC ? nI2 : 0) + (int64_t)a * nIs + b;
    }
    // column e of the G block of occupied i -> (p, r);  row kg -> row of At / B
    __device__ void col_g(int i, int e, int &p, int &r) const {
        if (e < na) { p = i; r = no + e; } else { p = no + e - na; r = i; }
    }
    __device__ int64_t row_g(int i, int kg) const {
        const int u = no + kg % na, part = kg / na;              // 0: exch (i u), 1: exch (u i), 2: coul (i u), 3: coul (u i)
        const int a = (part & 1) ? u : i, b = (part & 1) ? i : u;
        return (part >= 2 ? (int64_t)nIs * nIs : 0) + (int64_t)a * nIs + b;
    }
    // home of column (p, r): 1 = C block, 2 = G block, 0 = none (ELL only)
    __device__ int home(int p, int r) const {
        const int nI = no + na;
        if (p >= nI || r >= nI) return 0;
        const bool po = p < no, ro = r < no;
        if (!po && !ro) return 1;
        if (po && ro) return p == r ? 1 : 0;
        return 2;
    }
    // is entry (row k, column (p r)) part of the column's dense block?
    __device__ bool covered(int p, int r, int64_t k) const {
        const int h = home(p, r);
        if (h == 0) return false;
        const int64_t nI2 = (int64_t)nIs * nIs;
        const int nI = no + na;
        if (k == 2 * nI2) return h == 1;
        const int kk = (int)(k % nI2), a = kk / nIs, b = kk % nIs;
        if (a >= nI || b >= nI) return false;
        if (h == 1) return (a >= no && b >= no) || (a == b && a < no);
        const int i = p < no ? p : r;
        return (a == i && b >= no) || (b == i && a >= no);
    }
    // offset (in rows of ld^2 doubles) of column (p, r) inside its block's result buffer
    __device__ int64_t slot_c(int p, int r) const { return p < no ? na * na + p : (p - no) * na + (r - no); }
    __device__ int64_t slot_g(int p, int r) const {
        return p < no ? (int64_t)p * 2 * na + (r - no) : (int64_t)r * 2 * na + na + (p - no);
    }
};

// one warp per column (p r) of At: ELL list (k, val) of its non-zeros outside the dense block
__global__ void __launch_bounds__(256)
hess_sparse_build_kernel(RdmView rdm0, int64_t sd1, int64_t sd2, int nIs, int swap_exch, int width,
                         int *__restrict__ cnt, int *__restrict__ idx, double *__restrict__ val,
                         int *__restrict__ overflow) {
    const int lane = threadIdx.x & 31;
    const int col = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (col >= nIs * nIs) return;
    // blockIdx.y = which set of RDMs (one ELL table per set)
    const RdmView rdm{rdm0.d1 + blockIdx.y * sd1, rdm0.d2 + blockIdx.y * sd2, rdm0.no, rdm0.na};
    cnt += (int64_t)blockIdx.y * nIs * nIs;
    idx += (int64_t)blockIdx.y * nIs * nIs * width;
    val += (int64_t)blockIdx.y * nIs * nIs * width;
    const int p = col / nIs, r = col % nIs;
    const int nI = rdm.no + rdm.na;
    int base = 0;
    if (p < nI && r < nI) {
        const int64_t krows = 2 * (int64_t)nIs * nIs + 1;
        for (int64_t k0 = 0; k0 < krows; k0 += 32) {
            const int64_t k = k0 + lane;
            double v = 0.0;
            if (k < krows) {
                int m, n;                                  // (block entries are not even evaluated: no Gamma loads here)
                if (!Blocks{rdm.no, rdm.na, nIs}.covered(p, r, k)) v = at_value(rdm, nIs, swap_exch, k, p, r, m, n);
            }
            const unsigned mask = __ballot_sync(0xffffffffu, v != 0.0);
            if (v != 0.0) {
                const int pos = base + __popc(mask & ((1u << lane) - 1u));
                if (pos < width) {
                    idx[(int64_t)col * width + pos] = (int)k;
                    val[(int64_t)col * width + pos] = v;
                } else {
                    *overflow = 1;
                }
            }
            base += __popc(mask);
        }
    }
    if (lane == 0) cnt[col] = base < width ? base : width;
}

// C block operands: Atc[kc, cc] and Bc[kc, :] = the matching row of the class buffer
__global__ void hess_dense_at_kernel(RdmView rdm0, int64_t sd1, int64_t sd2, int nIs, int swap_exch, int64_t lda,
                                     double *__restrict__ Atc) {
    const RdmView rdm{rdm0.d1 + blockIdx.y * sd1, rdm0.d2 + blockIdx.y * sd2, rdm0.no, rdm0.na};
    const Blocks bl{rdm.no, rdm.na, nIs};
    const int64_t total = (int64_t)bl.nrow_c() * lda;
    Atc += (int64_t)blockIdx.y * total;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
         i += (int64_t)gridDim.x * blockDim.x) {
        const int kc = (int)(i / lda), cc = (int)(i % lda);
        double v = 0.0;
        if (cc < bl.ncol_c()) {
            int p, r, m, n;
            bl.col_c(cc, p, r);
            v = at_value(rdm, nIs, swap_exch, bl.row_c(kc), p, r, m, n);
        }
        Atc[i] = v;
    }
}

__global__ void hess_dense_b_kernel(const double *__restrict__ cls, int64_t cls_stride, int no, int na, int nIs,
                                    int64_t mat, double *__restrict__ Bc) {
    const Blocks bl{no, na, nIs};
    const int kc = blockIdx.y;
    cls += (int64_t)blockIdx.z * cls_stride;
    Bc += (int64_t)blockIdx.z * bl.nrow_c() * mat;
    const double2 *src = reinterpret_cast<const double2 *>(cls + bl.row_c(kc) * mat);
    double2 *dst = reinterpret_cast<double2 *>(Bc + (int64_t)kc * mat);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < mat / 2;
         i += (int64_t)gridDim.x * blockDim.x)
        dst[i] = src[i];
}

// G blocks: Tg[i][e][c] = sum_kg coef[kg][e] B[row_g(i, kg)][c].  grid (no, column tiles of 256, batch), 128 threads,
// two columns c per thread; CH result columns at a time with the accumulators in registers (CH >= 2 na for the usual
// active spaces: every B row is read exactly once), two B rows in flight per thread, coefficients and row offsets in
// shared memory.
template <int CH>
__global__ void __launch_bounds__(128)
hess_group_kernel(const double *__restrict__ B, int64_t b_stride, RdmView rdm0, int64_t sd1, int64_t sd2,
                  int rdm_batched, int nIs, int swap_exch, int64_t mat, double *__restrict__ Tg) {
    extern __shared__ __align__(16) double coef[];                 // [4 na][2 na] then int64 row offsets [4 na]
    const int bz = blockIdx.z;
    const RdmView rdm{rdm0.d1 + (rdm_batched ? bz * sd1 : 0), rdm0.d2 + (rdm_batched ? bz * sd2 : 0), rdm0.no,
                      rdm0.na};
    const Blocks bl{rdm.no, rdm.na, nIs};
    const int i = blockIdx.x, nr = bl.nrow_g(), nc = bl.ncol_g();
    int64_t *rowoff = reinterpret_cast<int64_t *>(coef + nr * nc);
    for (int x = threadIdx.x; x < nr * nc; x += blockDim.x) {
        int p, r, m, n;
        bl.col_g(i, x % nc, p, r);
        coef[x] = at_value(rdm, nIs, swap_exch, bl.row_g(i, x / nc), p, r, m, n);
    }
    for (int x = threadIdx.x; x < nr; x += blockDim.x) rowoff[x] = bl.row_g(i, x) * mat;
    __syncthreads();
    const int64_t c = ((int64_t)blockIdx.y * blockDim.x + threadIdx.x) * 2;
    if (c >= mat) return;
    B += bz * b_stride + c;
    Tg += ((int64_t)bz * rdm.no + i) * nc * mat + c;
    for (int e0 = 0; e0 < nc; e0 += CH) {
        double2 acc[CH];
#pragma unroll
        for (int j = 0; j < CH; ++j) acc[j] = make_double2(0.0, 0.0);
        for (int kg = 0; kg < nr; kg += 2) {                      // nr = 4 na is even: two B rows in flight
            const double2 b0 = __ldg(reinterpret_cast<const double2 *>(B + rowoff[kg]));
            const double2 b1 = __ldg(reinterpret_cast<const double2 *>(B + rowoff[kg + 1]));
            const double *cf0 = coef + kg * nc + e0, *cf1 = cf0 + nc;
#pragma unroll
            for (int j = 0; j < CH; ++j) {
                const bool in = e0 + j < nc;
                const double v0 = in ? cf0[j] : 0.0, v1 = in ? cf1[j] : 0.0;
                acc[j].x = fma(v0, b0.x, acc[j].x);
                acc[j].y = fma(v0, b0.y, acc[j].y);
                acc[j].x = fma(v1, b1.x, acc[j].x);
                acc[j].y = fma(v1, b1.y, acc[j].y);
            }
        }
#pragma unroll
        for (int j = 0; j < CH; ++j)
            if (e0 + j < nc) *reinterpret_cast<double2 *>(Tg + (int64_t)(e0 + j) * mat) = acc[j];
    }
}

// Streamed tensor-core form of the same product for large ld^2.  The kernel above issues one shared-memory
// coefficient load per two FMAs and ends up issue-bound at 2.4 TB/s (N = 256), however many loads are in flight.
// A G block is a small GEMM, Tg_i[e, c] = sum_kg coef[kg, e] B[row(kg), c] with K = 4 na, so:
//   * a CTA owns a contiguous range of (occupied i, 256-column tile) work items; per item ONE thread issues a
//     bulk asynchronous copy (cp.async.bulk, completion on an mbarrier) per B row into a shared-memory stage
//     (4 na segments of 2 KB, two stages => 100-200 KB in flight per SM);
//   * eight warps run FP64 DMMA.8x8x4 on the stage: M = 32 columns c per warp, N = 2 na result rows, K = 4 na;
//     stage rows are 260 doubles apart and coefficient rows NCP + 4 (both = 4 mod 8): conflict-free fragments;
//   * the accumulators go straight to Tg (64-byte runs).
// Same coefficients (at_value) as hess_group_kernel; the summation order inside a DMMA differs, so the two agree
// to round-off, not bit for bit.
constexpr int kGrpTile = 256;                       // columns per tile
constexpr int kGrpRow = kGrpTile + 4;               // stage row stride (doubles)
constexpr int kGrpStages = 2;

__device__ __forceinline__ void bulk_load(void *smem_dst, const void *gsrc, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(smem_dst)),
                 "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

size_t group_stream_smem_bytes(int na) {
    const int ncp = (2 * na + 7) / 8 * 8;
    return (size_t)kGrpStages * 4 * na * kGrpRow * sizeof(double) + (size_t)4 * na * (ncp + 4) * sizeof(double) +
           kGrpStages * sizeof(uint64_t) + 16;
}

constexpr int kGrpWarps = 8;                        // 32 columns (4 DMMA row tiles) per warp
constexpr int kGrpMT = kGrpTile / kGrpWarps / 8;

template <int NT>                                   // result rows padded to 8 NT >= 2 na
__global__ void __launch_bounds__(32 * kGrpWarps, 1)
hess_group_stream_kernel(const double *__restrict__ B, int64_t b_stride, RdmView rdm0, int64_t sd1, int64_t sd2,
                         int rdm_batched, int nIs, int swap_exch, int64_t mat, double *__restrict__ Tg,
                         int tiles_per_i, int items_per_cta) {
    extern __shared__ __align__(128) unsigned char gs_smem[];
    const int bz = blockIdx.y;
    const RdmView rdm{rdm0.d1 + (rdm_batched ? bz * sd1 : 0), rdm0.d2 + (rdm_batched ? bz * sd2 : 0), rdm0.no,
                      rdm0.na};
    const Blocks bl{rdm.no, rdm.na, nIs};
    const int nr = bl.nrow_g(), nc = bl.ncol_g();
    constexpr int CS = 8 * NT + 4;                  // coefficient row stride
    double *stage_buf = reinterpret_cast<double *>(gs_smem);
    double *coef = stage_buf + (size_t)kGrpStages * nr * kGrpRow;
    uint64_t *full = reinterpret_cast<uint64_t *>(coef + nr * CS);
    const int total = rdm.no * tiles_per_i;
    const int w0 = blockIdx.x * items_per_cta, w1 = min(w0 + items_per_cta, total);
    if (w0 >= w1) return;
    if (threadIdx.x == 0) {
        for (int s = 0; s < kGrpStages; ++s) mbar_init(&full[s], 1);
        fence_barrier_init();
    }
    __syncthreads();
    B += bz * b_stride;
    Tg += (int64_t)bz * rdm.no * nc * mat;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
    auto issue = [&](int w, int s) {                       // warp 0: all row segments of work item w into stage s
        const int i = w / tiles_per_i;
        const int64_t c0 = (int64_t)(w % tiles_per_i) * kGrpTile;
        const uint32_t seg = (uint32_t)((mat - c0 < kGrpTile ? mat - c0 : kGrpTile) * sizeof(double));
        if (lane == 0) mbar_arrive_expect_tx(&full[s], seg * nr);
        __syncwarp();
        double *dst = stage_buf + (size_t)s * nr * kGrpRow;
        for (int kg = lane; kg < nr; kg += 32)             // one or two bulk copies per lane
            bulk_load(dst + kg * kGrpRow, B + bl.row_g(i, kg) * mat + c0, seg, &full[s]);
    };
    if (warp == 0)
        for (int k = 0; k < kGrpStages && w0 + k < w1; ++k) issue(w0 + k, k);

    int cur_i = -1;
    for (int w = w0; w < w1; ++w) {
        const int k = w - w0, s = k % kGrpStages;
        const int i = w / tiles_per_i;
        if (i != cur_i) {                                  // (at most twice per CTA) coefficients of occupied i
            __syncthreads();
            for (int x = threadIdx.x; x < nr * 8 * NT; x += blockDim.x) {
                const int kg = x / (8 * NT), e = x % (8 * NT);
                double v = 0.0;
                if (e < nc) {
                    int p, r, m, n;
                    bl.col_g(i, e, p, r);
                    v = at_value(rdm, nIs, swap_exch, bl.row_g(i, kg), p, r, m, n);
                }
                coef[kg * CS + e] = v;
            }
            __syncthreads();
            cur_i = i;
        }
        mbar_wait(&full[s], (uint32_t)(k / kGrpStages) & 1u);
        const double *st = stage_buf + (size_t)s * nr * kGrpRow + 8 * kGrpMT * warp + g;
        double acc[kGrpMT][NT][2];
#pragma unroll
        for (int mt = 0; mt < kGrpMT; ++mt)
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) acc[mt][nt][0] = acc[mt][nt][1] = 0.0;
#pragma unroll 2
        for (int k0 = 0; k0 < nr; k0 += 4) {               // nr = 4 na
            double a[kGrpMT], bf[NT];
            const double *srow = st + (k0 + t) * kGrpRow;
#pragma unroll
            for (int mt = 0; mt < kGrpMT; ++mt) a[mt] = srow[8 * mt];
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) bf[nt] = coef[(k0 + t) * CS + 8 * nt + g];
#pragma unroll
            for (int mt = 0; mt < kGrpMT; ++mt)
#pragma unroll
                for (int nt = 0; nt < NT; ++nt) dmma884(acc[mt][nt][0], acc[mt][nt][1], a[mt], bf[nt]);
        }
        const int64_t c0 = (int64_t)(w % tiles_per_i) * kGrpTile + 8 * kGrpMT * warp + g;
        double *out = Tg + (int64_t)i * nc * mat;
#pragma unroll
        for (int mt = 0; mt < kGrpMT; ++mt) {
            const int64_t c = c0 + 8 * mt;
            if (c >= mat) continue;
#pragma unroll
            for (int nt = 0; nt < NT; ++nt)
#pragma unroll
                for (int cc = 0; cc < 2; ++cc) {
                    const int e = 8 * nt + 2 * t + cc;
                    if (e < nc) out[(int64_t)e * mat + c] = acc[mt][nt][cc];
                }
        }
        __syncthreads();                                   // every thread is done with stage s
        if (warp == 0 && w + kGrpStages < w1) issue(w + kGrpStages, s);
    }
}

// T[(p r), c] (= or +=) sum_e val[e] * B[idx[e], c].   grid (columns (p r), column tiles of 512);
// consecutive CTAs share a column tile of B, which therefore stays in L2.
__global__ void __launch_bounds__(256)
hess_spmm_kernel(const double *__restrict__ B, int64_t b_stride, const int *__restrict__ cnt,
                 const int *__restrict__ idx, const double *__restrict__ val, int rdm_batched, int width, int no,
                 int na, int nIs, int64_t mat, double *__restrict__ T, double *__restrict__ Tc,
                 double *__restrict__ Tg, int skip_occ_pairs) {
    const int col = blockIdx.x;
    const int p = col / nIs, r = col % nIs, nI = no + na;
    if (p >= nI || r >= nI) return;
    if (skip_occ_pairs && p < no && r < no && p != r) return;      // hess_spmm_pair_kernel does these
    const Blocks bl{no, na, nIs};
    const int home = bl.home(p, r);
    {
        const int64_t bz = blockIdx.z, nI2 = (int64_t)nIs * nIs;
        B += bz * b_stride;
        T += bz * nI2 * mat;
        Tc += bz * (int64_t)bl.ncol_c() * mat;
        Tg += bz * (int64_t)no * bl.ncol_g() * mat;
        if (rdm_batched) {
            cnt += bz * nI2;
            idx += bz * nI2 * width;
            val += bz * nI2 * width;
        }
    }
    // the column's (row, value) list goes to shared memory once: in the loop below every B load is then paired
    // with two broadcast LDS instead of two more global loads through the same L1 pipe
    extern __shared__ __align__(16) unsigned char spmm_smem[];
    double *vl = reinterpret_cast<double *>(spmm_smem);
    int *ix = reinterpret_cast<int *>(vl + width);
    const int n = cnt[col];
    if (n == 0 && home != 0) return;                      // the column's dense block holds all of it
    for (int e = threadIdx.x; e < n; e += blockDim.x) {
        ix[e] = idx[(int64_t)col * width + e];
        vl[e] = val[(int64_t)col * width + e];
    }
    __syncthreads();
    // (grid.y may be smaller than the number of 512-column tiles: with the pair kernel taking the occ-occ columns, a
    //  reference-shaped RDM leaves this kernel nothing to do, and 250 000 CTAs that only find that out cost 0.15 ms)
    for (int64_t c = ((int64_t)blockIdx.y * blockDim.x + threadIdx.x) * 2; c < mat; c += (int64_t)gridDim.y * blockDim.x * 2) {
    double2 acc = make_double2(0.0, 0.0);
    int e = 0;
    for (; e + 4 <= n; e += 4) {
        double2 b0 = __ldg(reinterpret_cast<const double2 *>(B + (int64_t)ix[e] * mat + c));
        double2 b1 = __ldg(reinterpret_cast<const double2 *>(B + (int64_t)ix[e + 1] * mat + c));
        double2 b2 = __ldg(reinterpret_cast<const double2 *>(B + (int64_t)ix[e + 2] * mat + c));
        double2 b3 = __ldg(reinterpret_cast<const double2 *>(B + (int64_t)ix[e + 3] * mat + c));
        const double v0 = vl[e], v1 = vl[e + 1], v2 = vl[e + 2], v3 = vl[e + 3];
        acc.x = fma(v0, b0.x, acc.x); acc.y = fma(v0, b0.y, acc.y);
        acc.x = fma(v1, b1.x, acc.x); acc.y = fma(v1, b1.y, acc.y);
        acc.x = fma(v2, b2.x, acc.x); acc.y = fma(v2, b2.y, acc.y);
        acc.x = fma(v3, b3.x, acc.x); acc.y = fma(v3, b3.y, acc.y);
    }
    for (; e < n; ++e) {
        const double2 b0 = __ldg(reinterpret_cast<const double2 *>(B + (int64_t)ix[e] * mat + c));
        const double v0 = vl[e];
        acc.x = fma(v0, b0.x, acc.x); acc.y = fma(v0, b0.y, acc.y);
    }
    if (home != 0) {                                      // add to what the dense block produced
        double2 *o = reinterpret_cast<double2 *>((home == 1 ? Tc + bl.slot_c(p, r) * mat : Tg + bl.slot_g(p, r) * mat) + c);
        double2 t = *o;
        t.x += acc.x; t.y += acc.y;
        *o = t;
    } else {
        *reinterpret_cast<double2 *>(T + (int64_t)col * mat + c) = acc;
    }
    }
}

// The occ-occ off-diagonal columns in PAIRS: T[(i j), c] and T[(j i), c], i > j, from one pass over the rows either
// of them needs.  Their two ELL lists name the same few rows of B -- the exchange rows (i j), (j i) and the Coulomb
// rows (i j), (j i), which hold identical numbers (J[m,n] = J[n,m]) and are read through ONE index -- so a pair costs
// 3 row reads + 2 row writes instead of 6 + 2, and every thread has 4 x 3 independent 16-byte loads in flight.
// grid (pairs, column chunks of kPairChunk, batch); `skip` tells hess_spmm_kernel to leave these columns alone.
constexpr int kPairUnroll = 4, kPairChunk = 256 * 2 * kPairUnroll, kPairMaxRows = 16;

__global__ void __launch_bounds__(256)
hess_spmm_pair_kernel(const double *__restrict__ B, int64_t b_stride, const int *__restrict__ cnt,
                      const int *__restrict__ idx, const double *__restrict__ val, int rdm_batched, int width, int no,
                      int nIs, int64_t mat, double *__restrict__ T) {
    __shared__ int urow[kPairMaxRows];
    __shared__ double uv0[kPairMaxRows], uv1[kPairMaxRows];
    __shared__ int un;
    int i = (int)((sqrtf(8.0f * (float)blockIdx.x + 1.0f) + 1.0f) * 0.5f);          // pair index -> i > j >= 0
    while (i * (i - 1) / 2 > (int)blockIdx.x) --i;
    while ((i + 1) * i / 2 <= (int)blockIdx.x) ++i;
    const int j = (int)blockIdx.x - i * (i - 1) / 2;
    const int64_t bz = blockIdx.z, nI2 = (int64_t)nIs * nIs;
    B += bz * b_stride;
    T += bz * nI2 * mat;
    if (rdm_batched) {
        cnt += bz * nI2;
        idx += bz * nI2 * width;
        val += bz * nI2 * width;
    }
    const int col0 = i * nIs + j, col1 = j * nIs + i;
    if (threadIdx.x == 0) {
        int n = 0;
        for (int which = 0; which < 2; ++which) {
            const int col = which ? col1 : col0;
            for (int e = 0; e < cnt[col]; ++e) {
                int k = idx[(int64_t)col * width + e];
                if (k >= nI2 && k < 2 * nI2) {                        // Coulomb row (m n): read it as (max, min)
                    const int kk = k - (int)nI2, m = kk / nIs, nn = kk % nIs;
                    if (m < nn) k = (int)nI2 + nn * nIs + m;
                }
                int u = 0;
                while (u < n && urow[u] != k) ++u;
                if (u == n && n < kPairMaxRows) {
                    urow[n] = k;
                    uv0[n] = uv1[n] = 0.0;
                    ++n;
                }
                if (u < kPairMaxRows) (which ? uv1 : uv0)[u] += val[(int64_t)col * width + e];
            }
        }
        un = n;
    }
    __syncthreads();
    const int n = un;
    const int64_t c0 = (int64_t)blockIdx.y * kPairChunk + threadIdx.x * 2;
    double2 a0[kPairUnroll], a1[kPairUnroll];
#pragma unroll
    for (int u = 0; u < kPairUnroll; ++u) a0[u] = a1[u] = make_double2(0.0, 0.0);
    for (int e = 0; e < n; ++e) {
        const double *row = B + (int64_t)urow[e] * mat;
        const double v0 = uv0[e], v1 = uv1[e];
        double2 b[kPairUnroll];
#pragma unroll
        for (int u = 0; u < kPairUnroll; ++u) {
            const int64_t c = c0 + (int64_t)u * 512;
            b[u] = c < mat ? __ldg(reinterpret_cast<const double2 *>(row + c)) : make_double2(0.0, 0.0);
        }
#pragma unroll
        for (int u = 0; u < kPairUnroll; ++u) {
            a0[u].x = fma(v0, b[u].x, a0[u].x); a0[u].y = fma(v0, b[u].y, a0[u].y);
            a1[u].x = fma(v1, b[u].x, a1[u].x); a1[u].y = fma(v1, b[u].y, a1[u].y);
        }
    }
#pragma unroll
    for (int u = 0; u < kPairUnroll; ++u) {
        const int64_t c = c0 + (int64_t)u * 512;
        if (c < mat) {
            *reinterpret_cast<double2 *>(T + (int64_t)col0 * mat + c) = a0[u];
            *reinterpret_cast<double2 *>(T + (int64_t)col1 * mat + c) = a1[u];
        }
    }
}

// B rows as above; columns (q s) over ld x ld (padding columns come out as the zero padding of g, h).
__global__ void hess_gather_b_kernel(const double *__restrict__ h, const double *__restrict__ g, int nI,
                                     int ld, double *__restrict__ B) {
    const int nI2 = nI * nI;
    const int64_t mat = (int64_t)ld * ld;
    const int64_t total = (int64_t)(2 * nI2 + (h ? 1 : 0)) * mat;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        const int64_t k = i / mat;
        const int64_t c = i % mat;
        const int q = (int)(c / ld), s = (int)(c % ld);
        double v;
        if (k < nI2) {
            const int m = (int)(k / nI), n = (int)(k % nI);
            v = g[(((int64_t)q * ld + m) * ld + n) * ld + s];
        } else if (k < 2 * nI2) {
            const int kk = (int)(k - nI2);
            const int m = kk / nI, n = kk % nI;
            v = g[(((int64_t)q * ld + s) * ld + m) * ld + n];
        } else {
            v = h[c];
        }
        B[i] = v;
    }
}

struct TView {
    const double *T;     // rows (a c) -> a * nIs + c
    const double *Taa;   // optional (class path): results of the C block (Blocks::slot_c); null = everything in T
    const double *Tg;    // with Taa: results of the G blocks (Blocks::slot_g)
    int nI, nIs, no, na;
    int64_t t_stride, taa_stride, tg_stride, f_stride, h_stride;   // per-evaluation strides (blockIdx.z)
    // row (a c) of T, a, c < nI  (ld2 = ld * ld)
    __device__ __forceinline__ const double *row(int a, int c, int64_t ld2) const {
        if (Taa) {
            const Blocks bl{no, na, nIs};
            const int h = bl.home(a, c);
            if (h == 1) return Taa + bl.slot_c(a, c) * ld2;
            if (h == 2) return Tg + bl.slot_g(a, c) * ld2;
        }
        return T + ((int64_t)a * nIs + c) * ld2;
    }
    __device__ __forceinline__ void at_batch(int b) {
        T += b * t_stride;
        if (Taa) { Taa += b * taa_stride; Tg += b * tg_stride; }
    }
};

__device__ __forceinline__ double hess_x(const TView &tv, const double *__restrict__ F, int ld, int a, int b,
                                         int c, int d) {
    // X(a,b,c,d) = -(F_ac + F_ca) delta_bd + [a,c in I] T[(a c),(b d)]
    double v = 0.0;
    if (b == d) v = -(F[(int64_t)a * ld + c] + F[(int64_t)c * ld + a]);
    if (a < tv.nI && c < tv.nI) v += tv.row(a, c, (int64_t)ld * ld)[(int64_t)b * ld + d];
    return v;
}

__global__ void __launch_bounds__(256)
hess_assemble_kernel(TView tv, const double *__restrict__ F,
                     const int32_t *__restrict__ pl, const int32_t *__restrict__ pr, int nk, int ld,
                     double *__restrict__ H) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    const int j = blockIdx.y;
    if (k >= nk) return;
    tv.at_batch(blockIdx.z);
    F += blockIdx.z * tv.f_stride;
    H += blockIdx.z * tv.h_stride;
    const int p = pl[j], q = pr[j];
    const int r = pl[k], s = pr[k];
    const double v = hess_x(tv, F, ld, p, q, r, s) - hess_x(tv, F, ld, p, q, s, r)
                   - hess_x(tv, F, ld, q, p, r, s) + hess_x(tv, F, ld, q, p, s, r);
    H[(int64_t)j * nk + k] = v;
}

// ---- row-tiled assembly -----------------------------------------------------------------------
// The kernel above reads T[(q s),(p r)] with consecutive threads on consecutive s: a different row of T per
// thread, 32 cache lines per warp load.  Two of the four terms are contiguous in s (natural k order), the
// other two in r.  With the pairs sorted by their row index (np.tril_indices order, what the engine passes)
// a CTA takes one row j and RT consecutive orbital rows r, i.e. one contiguous k range, evaluates the
// s-contiguous terms in k order, the r-contiguous terms in (s, r) order (warp = 32 consecutive r of one s:
// two cache lines per load) into a shared-memory strip, and writes the strip out coalesced.
// hess_pair_runs_kernel finds the k range of every orbital row (binary search) and verifies the structure
// (rows non-decreasing, columns consecutive within a row); when it does not hold the same kernel falls
// back to the per-thread form over k tiles -- decided on the device, no host round trip.
constexpr int kAsmRows = 32;                       // orbital rows per CTA
constexpr int kAsmStrip = kAsmRows * (64 + 1);     // shared-memory strip (doubles): runs of up to 64 columns

// runs[l] = first k of orbital row l (l <= N); runs[N+1] = 1 when the pair list is row-sorted with consecutive
// columns inside a row; runs[N+2] = S > 0 when, in addition, every row l >= rows_in (rows_in = nI rounded up to
// even) holds exactly the columns 0 .. S-1 with S <= min(nI, 64): the layout the streamed assembly needs.
__global__ void hess_pair_runs_kernel(const int32_t *__restrict__ pl, const int32_t *__restrict__ pr, int nk, int N,
                                      int nI, int *__restrict__ runs) {
    __shared__ int bad, nonuniform;
    if (threadIdx.x == 0) bad = nonuniform = 0;
    __syncthreads();
    for (int l = threadIdx.x; l <= N; l += blockDim.x) {      // lower_bound(pl, l)
        int lo = 0, hi = nk;
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (pl[mid] < l) lo = mid + 1; else hi = mid;
        }
        runs[l] = lo;
    }
    int mybad = 0;
    for (int k = threadIdx.x + 1; k < nk; k += blockDim.x) {
        if (pl[k] < pl[k - 1]) mybad = 1;
        if (pl[k] == pl[k - 1] && pr[k] != pr[k - 1] + 1) mybad = 1;
    }
    for (int k = threadIdx.x; k < nk; k += blockDim.x)
        if (pl[k] < 0 || pl[k] >= N || pr[k] < 0 || pr[k] >= N) mybad = 1;
    if (mybad) bad = 1;
    __syncthreads();
    const int rows_in = min((nI + 1) & ~1, N);
    const int S = rows_in < N ? runs[rows_in + 1] - runs[rows_in] : 0;
    if (!bad)
        for (int l = rows_in + threadIdx.x; l < N; l += blockDim.x)
            if (runs[l + 1] - runs[l] != S || S <= 0 || pr[runs[l]] != 0) nonuniform = 1;
    __syncthreads();
    if (threadIdx.x == 0) {
        runs[N + 1] = bad ? 0 : 1;
        runs[N + 2] = (!bad && !nonuniform && S > 0 && S <= nI && S <= 64) ? S : 0;
    }
}

__device__ __forceinline__ double hess_t(const TView &tv, int ld, int a, int c, int b, int d) {
    // [a, c in I] T[(a c),(b d)]
    if (a >= tv.nI || c >= tv.nI) return 0.0;
    return __ldg(tv.row(a, c, (int64_t)ld * ld) + (int64_t)b * ld + d);
}

__device__ __forceinline__ double fock_sym(const double *__restrict__ F, int ld, int a, int c) {
    return __ldg(F + (int64_t)a * ld + c) + __ldg(F + (int64_t)c * ld + a);
}

constexpr int kAsmJ = 4;              // Hessian rows j per CTA (measured 2 / 4 / 8: 0.53 / 0.44 / 0.75 ms at N = 256) (the row-tile bookkeeping is shared by all of them)

__global__ void __launch_bounds__(256, 4)
hess_assemble_rows_kernel(TView tv, const double *__restrict__ F, const int32_t *__restrict__ pl,
                          const int32_t *__restrict__ pr, const int *__restrict__ runs, int nk, int N, int ld,
                          double *__restrict__ H, int stream_partner) {
    __shared__ double strip[kAsmStrip];
    __shared__ unsigned char rowof[kAsmStrip];
    __shared__ int rstart[kAsmRows], rlen[kAsmRows], rs0[kAsmRows];
    __shared__ int s_lo, s_hi;
    tv.at_batch(blockIdx.z);
    F += blockIdx.z * tv.f_stride;
    H += blockIdx.z * tv.h_stride;
    const int j0 = blockIdx.y * kAsmJ, j1 = min(j0 + kAsmJ, nk);
    const bool structured = runs[N + 1] != 0;
    // row tiles: tile 0 = the orbital rows inside I (short runs, all four terms: per-thread form), tile t >= 1 =
    // kAsmRows rows outside I
    const int rows_in = min((tv.nI + 1) & ~1, N);
    if (blockIdx.x > 0 && stream_partner && runs[N + 2] > 0) return;      // hess_assemble_stream_kernel has these tiles
    const int l0 = blockIdx.x == 0 ? 0 : rows_in + ((int)blockIdx.x - 1) * kAsmRows;
    const int l1 = blockIdx.x == 0 ? rows_in : min(l0 + kAsmRows, N);
    int kb = 0, ke = 0;
    if (structured) {
        if (l0 >= N) return;
        kb = runs[l0];
        ke = runs[l1];
        if (kb == ke) return;
    }
    // Rows r outside I kill the two s-contiguous terms ([p,r in I] and [q,r in I]); what is left is contiguous in
    // r.  Tiles with a row inside I (a few short runs) and unstructured pair lists take the per-thread form.
    if (!structured || blockIdx.x == 0 || ke - kb + kAsmRows > kAsmStrip) {
        // work items (j, k), k fastest: all 256 threads busy even when the tile holds a handful of pairs
        const int nj = j1 - j0;
        if (structured) {
            const int cnt = ke - kb;
            for (int idx = threadIdx.x; idx < cnt * nj; idx += blockDim.x) {
                const int k = kb + idx % cnt, j = j0 + idx / cnt;
                const int r = pl[k], s = pr[k], p = pl[j], q = pr[j];
                H[(int64_t)j * nk + k] = hess_x(tv, F, ld, p, q, r, s) - hess_x(tv, F, ld, p, q, s, r)
                                       - hess_x(tv, F, ld, q, p, r, s) + hess_x(tv, F, ld, q, p, s, r);
            }
        } else {
            for (int k0 = blockIdx.x * 256; k0 < nk; k0 += gridDim.x * 256) {
                const int k = k0 + threadIdx.x;
                if (k >= nk) continue;
                const int r = pl[k], s = pr[k];
                for (int j = j0; j < j1; ++j) {
                    const int p = pl[j], q = pr[j];
                    H[(int64_t)j * nk + k] = hess_x(tv, F, ld, p, q, r, s) - hess_x(tv, F, ld, p, q, s, r)
                                           - hess_x(tv, F, ld, q, p, r, s) + hess_x(tv, F, ld, q, p, s, r);
                }
            }
        }
        return;
    }
    if (threadIdx.x < kAsmRows) {
        const int l = l0 + threadIdx.x;
        const int a = l < N ? runs[l] : ke, b = l < N ? runs[l + 1] : ke;
        rstart[threadIdx.x] = a - kb + threadIdx.x;        // one pad slot per orbital row: conflict-free strip writes
        rlen[threadIdx.x] = b - a;
        const int first = b > a ? pr[a] : N, last = b > a ? first + (b - a) - 1 : -1;
        rs0[threadIdx.x] = b > a ? first : 0;
        int lo = first, hi = last;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            lo = min(lo, __shfl_xor_sync(0xffffffffu, lo, o));
            hi = max(hi, __shfl_xor_sync(0xffffffffu, hi, o));
        }
        if (threadIdx.x == 0) {
            s_lo = lo;
            s_hi = hi;
        }
    }
    for (int i = threadIdx.x; i < ke - kb; i += blockDim.x) rowof[i] = (unsigned char)(pl[kb + i] - l0);
    __syncthreads();
    // (s, r) order, r fastest: a warp reads 32 consecutive r of one row of T
    const int ns = s_hi - s_lo + 1;
    const int ri = threadIdx.x % kAsmRows, r = l0 + ri;
    const int my_s0 = rs0[ri], my_len = rlen[ri], my_start = rstart[ri];
    for (int j = j0; j < j1; ++j) {
        const int p = pl[j], q = pr[j];
        const bool p_in = p < tv.nI;
#pragma unroll 6
        for (int si = threadIdx.x / kAsmRows; si < ns; si += 256 / kAsmRows) {
            const int s = s_lo + si;
            const int pos = s - my_s0;
            if (pos < 0 || pos >= my_len) continue;
            double v = hess_t(tv, ld, q, s, p, r);
            if (p_in) v -= hess_t(tv, ld, p, s, q, r);
            if (q == s) v -= fock_sym(F, ld, p, r);
            if (q == r) v += fock_sym(F, ld, p, s);
            if (p == s) v += fock_sym(F, ld, q, r);
            if (p == r) v -= fock_sym(F, ld, q, s);
            strip[my_start + pos] = v;
        }
        __syncthreads();
        double *Hj = H + (int64_t)j * nk + kb;
        for (int i = threadIdx.x; i < ke - kb; i += blockDim.x) Hj[i] = strip[i + rowof[i]];
        __syncthreads();
    }
}

// Streamed assembly of the rows outside I (the bulk: (N - nI) / N of the orbital rows).  For a Hessian row
// j = (p, q) and 32 orbital rows r, the surviving term T[(q s),(p r)] is, for each column s, one 256-byte piece of
// a row of T: warp jj issues those S pieces of "its" j as bulk asynchronous copies (cp.async.bulk -> shared memory,
// one mbarrier per j), so all 8 x S pieces of the CTA (90 KB at N = 256) are in flight at once instead of one
// 8-byte load per thread; the pieces are then transposed through a padded strip and written out coalesced.
// Needs the uniform pair layout hess_pair_runs_kernel certifies (runs[N+2] = S); otherwise this kernel returns at
// once and hess_assemble_rows_kernel does the tiles.
__global__ void __launch_bounds__(256)
hess_assemble_stream_kernel(TView tv, const double *__restrict__ F, const int32_t *__restrict__ pl,
                            const int32_t *__restrict__ pr, const int *__restrict__ runs, int nk, int N, int ld,
                            double *__restrict__ H) {
    extern __shared__ __align__(128) unsigned char as_smem[];
    const int S = runs[N + 2];
    if (S == 0) return;
    const int rows_in = min((tv.nI + 1) & ~1, N);
    const int l0 = rows_in + (int)blockIdx.x * kAsmRows;
    if (l0 >= N) return;
    const int nrows = min(kAsmRows, N - l0);
    const uint32_t seg = (uint32_t)(min(kAsmRows, ld - l0) * sizeof(double));     // even count: 16-byte multiple
    const int kb = runs[l0];
    double *stage = reinterpret_cast<double *>(as_smem);                          // [kAsmJ][S][kAsmRows]
    double *strip = stage + (size_t)kAsmJ * S * kAsmRows;                         // [kAsmRows][S + 1]
    uint64_t *bar = reinterpret_cast<uint64_t *>(strip + kAsmRows * (S + 1) + ((kAsmRows * (S + 1)) & 1));
    tv.at_batch(blockIdx.z);
    F += blockIdx.z * tv.f_stride;
    H += blockIdx.z * tv.h_stride;
    const int j0 = blockIdx.y * kAsmJ, j1 = min(j0 + kAsmJ, nk);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t ld2 = (int64_t)ld * ld;
    if (threadIdx.x == 0) {
        for (int jj = 0; jj < kAsmJ; ++jj) mbar_init(&bar[jj], 1);
        fence_barrier_init();
    }
    __syncthreads();
    {                                                     // warp jj fetches the pieces of Hessian row j0 + jj
        const int j = j0 + warp;
        if (j < j1) {
            const int p = pl[j], q = pr[j];
            if (q < tv.nI) {
                if (lane == 0) mbar_arrive_expect_tx(&bar[warp], seg * S);
                __syncwarp();
                for (int sx = lane; sx < S; sx += 32)
                    bulk_load(stage + ((size_t)warp * S + sx) * kAsmRows, tv.row(q, sx, ld2) + (int64_t)p * ld + l0, seg,
                              &bar[warp]);
            }
        }
    }
    // strip positions of this thread's elements in the coalesced write-out (the same for every Hessian row)
    constexpr int kFlush = 6;
    int sidx[kFlush];
#pragma unroll
    for (int m = 0; m < kFlush; ++m) {
        const int i = threadIdx.x + m * 256;
        sidx[m] = (i / S) * (S + 1) + i % S;
    }
    for (int jj = 0; jj < j1 - j0; ++jj) {
        const int j = j0 + jj;
        const int p = pl[j], q = pr[j];
        const bool q_in = q < tv.nI, p_in = p < tv.nI;
        if (q_in) mbar_wait(&bar[jj], 0);
        const int r = l0 + lane;
        if (lane < nrows) {
            for (int sx = warp; sx < S; sx += 8) {
                double v = q_in ? stage[((size_t)jj * S + sx) * kAsmRows + lane] : 0.0;
                if (p_in) v -= __ldg(tv.row(p, sx, ld2) + (int64_t)q * ld + r);
                if (q == sx) v -= fock_sym(F, ld, p, r);
                if (q == r) v += fock_sym(F, ld, p, sx);      // (q >= rows_in: a pair (p, q) in a row inside I)
                if (p == sx) v += fock_sym(F, ld, q, r);
                if (p == r) v -= fock_sym(F, ld, q, sx);
                strip[lane * (S + 1) + sx] = v;
            }
        }
        __syncthreads();
        double *Hj = H + (int64_t)j * nk + kb;
#pragma unroll
        for (int m = 0; m < kFlush; ++m) {
            const int i = threadIdx.x + m * 256;
            if (i < nrows * S) Hj[i] = strip[sidx[m]];
        }
        for (int i = threadIdx.x + kFlush * 256; i < nrows * S; i += blockDim.x)
            Hj[i] = strip[(i / S) * (S + 1) + i % S];
        __syncthreads();
    }
}

// ---- API-parity helpers: dense full-space RDMs and the dense Y-matrix -----------------
// (reference full_rdms oo_energy.py:342-379 and y_matrix :381-393 for an arbitrary dense
// two_full; the Hessian path above never materialises either)
__global__ void full_rdms_kernel(RdmView rdm, int N, double *__restrict__ d1, double *__restrict__ d2) {
    const int64_t n2 = (int64_t)N * N, n4 = n2 * n2;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
        const int t = (int)(i % N), s = (int)((i / N) % N), q = (int)((i / n2) % N), p = (int)(i / (n2 * N));
        d2[i] = gf2(rdm, p, q, s, t);
        if (i < n2) d1[i] = gf1(rdm, (int)(i / N), (int)(i % N));
    }
}

// At rows [0,N^2): G[p,m,r,n] + G[p,m,n,r]; rows [N^2, 2N^2): G[p,r,m,n]; column (p r); dense G (N^4)
__global__ void y_build_at_kernel(const double *__restrict__ G, int N, int64_t lda, double *__restrict__ At) {
    const int N2 = N * N;
    const int64_t total = (int64_t)2 * N2 * lda;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    auto at = [&](int a, int b, int c, int d) { return G[(((int64_t)a * N + b) * N + c) * N + d]; };
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        const int64_t k = i / lda;
        const int col = (int)(i % lda);
        double v = 0.0;
        if (col < N2) {
            const int p = col / N, r = col % N;
            const int kk = (int)(k % N2);
            const int m = kk / N, n = kk % N;
            v = (k < N2) ? at(p, m, r, n) + at(p, m, n, r) : at(p, r, m, n);
        }
        At[i] = v;
    }
}

// Y[p,q,r,s] (dense N^4) = T[(p r),(q s)] (row pitch ld*ld)
__global__ void y_permute_kernel(const double *__restrict__ T, int N, int ld, double *__restrict__ Y) {
    const int64_t n2 = (int64_t)N * N, n4 = n2 * n2;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
        const int s = (int)(i % N), r = (int)((i / N) % N), q = (int)((i / n2) % N), p = (int)(i / (n2 * N));
        Y[i] = T[((int64_t)p * N + r) * ld * ld + (int64_t)q * ld + s];
    }
}

size_t assemble_scratch_bytes(int ld) { return align_up((size_t)(ld + 3) * sizeof(int), 1024); }

int launch_assemble(const TView &tv, const double *F, const int32_t *pl, const int32_t *pr, int nk, int N, int ld,
                    int batch, double *H, void *scratch, unsigned flags, cudaStream_t stream) {
    const bool per_element = (flags & OO_FLAG_HESSIAN_ASSEMBLE_PER_ELEMENT) != 0;
    const bool tiled = (flags & OO_FLAG_HESSIAN_ASSEMBLE_TILED) != 0;
    const bool g_hessian_assemble_unstreamed = (flags & OO_FLAG_HESSIAN_ASSEMBLE_UNSTREAMED) != 0;
    // small bases: a handful of CTAs either way, and the per-thread kernel needs no pair-structure pass
    if (per_element || (!tiled && N <= 64)) {
        dim3 grid((unsigned)ceil_div(nk, 256), (unsigned)nk, (unsigned)batch);
        hess_assemble_kernel<<<grid, 256, 0, stream>>>(tv, F, pl, pr, nk, ld, H);
        OO_LAUNCH_CHECK();
        return OO_OK;
    }
    int *runs = reinterpret_cast<int *>(scratch);
    if (!(flags & OO_FLAG_HESSIAN_REUSE_OPERANDS)) {         // (same pair list as the previous call: runs are there)
        hess_pair_runs_kernel<<<1, 1024, 0, stream>>>(pl, pr, nk, N, tv.nI, runs);
        OO_LAUNCH_CHECK();
    }
    const int rows_in = (tv.nI + 1) & ~1;
    const int rows_out = N > rows_in ? N - rows_in : 0;
    const int smax = tv.nI < 64 ? tv.nI : 64;
    const size_t smem = ((size_t)kAsmJ * smax * kAsmRows + (size_t)kAsmRows * (smax + 1) + 2 + kAsmJ) * sizeof(double);
    const int streamed = !g_hessian_assemble_unstreamed && rows_out > 0 &&
                         smem <= 110 * 1024;
    dim3 grid((unsigned)(1 + ceil_div(rows_out, kAsmRows)), (unsigned)ceil_div(nk, kAsmJ), (unsigned)batch);
    hess_assemble_rows_kernel<<<grid, 256, 0, stream>>>(tv, F, pl, pr, runs, nk, N, ld, H, streamed);
    OO_LAUNCH_CHECK();
    if (streamed) {
        static unsigned long long cfgd = 0;
        if (once_per_device(cfgd))
            OO_CUDA_CHECK(cudaFuncSetAttribute(hess_assemble_stream_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                               110 * 1024));
        dim3 sgrid((unsigned)ceil_div(rows_out, kAsmRows), (unsigned)ceil_div(nk, kAsmJ), (unsigned)batch);
        hess_assemble_stream_kernel<<<sgrid, 256, smem, stream>>>(tv, F, pl, pr, runs, nk, N, ld, H);
        OO_LAUNCH_CHECK();
    }
    return OO_OK;
}

struct HessLayout {
    int64_t lda, krows;
    size_t off_b, off_t, off_runs, total;
};

HessLayout hess_layout(int ld, int nI) {
    HessLayout L;
    const int64_t nI2 = (int64_t)nI * nI;
    L.lda = (nI2 + 1) & ~1ll;
    L.krows = 2 * nI2 + 1;
    const size_t at_bytes = align_up((size_t)L.krows * L.lda * sizeof(double), 1024);
    const size_t b_bytes = align_up((size_t)L.krows * ld * ld * sizeof(double), 1024);
    const size_t t_bytes = align_up((size_t)nI2 * ld * ld * sizeof(double), 1024);
    L.off_b = at_bytes;
    L.off_t = at_bytes + b_bytes;
    L.off_runs = at_bytes + b_bytes + t_bytes;
    L.total = L.off_runs + assemble_scratch_bytes(ld);
    return L;
}

}  // namespace

int class_hessian(const double *cls, const double *F, const double *d1, int64_t sd1, const double *d2,
                  int64_t sd2, int no, int na, int N, int ld, int nIp, int batch, const int32_t *pl,
                  const int32_t *pr, int nk, double *H, void *ws, size_t ws_bytes, unsigned flags,
                  cudaStream_t stream);
size_t class_hessian_ws_bytes(int ld, int nIp, int no, int na, int batch);

namespace {
// class-layout B operand from the complete tensor: rows [K(n,m) | J(m,n) | h], m, n < nIp (zero rows beyond nI)
//   K[n,m,a,b] = g'[a,m,n,b],  J[m,n,a,b] = g'[a,b,m,n]   (the layout classes.cu produces)
__global__ void hess_gather_class_kernel(const double *__restrict__ h, const double *__restrict__ g, int nI, int nIp,
                                         int ld, double *__restrict__ B) {
    const int64_t nI2 = (int64_t)nIp * nIp, mat = (int64_t)ld * ld;
    const int64_t total = (2 * nI2 + 1) * mat;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        const int64_t k = i / mat, c = i % mat;
        const int a = (int)(c / ld), b = (int)(c % ld);
        double v = 0.0;
        if (k < nI2) {
            const int n = (int)(k / nIp), m = (int)(k % nIp);
            if (m < nI && n < nI) v = g[(((int64_t)a * ld + m) * ld + n) * ld + b];
        } else if (k < 2 * nI2) {
            const int kk = (int)(k - nI2), m = kk / nIp, n = kk % nIp;
            if (m < nI && n < nI) v = g[(((int64_t)a * ld + b) * ld + m) * ld + n];
        } else {
            v = h[c];
        }
        B[i] = v;
    }
}

size_t full_hessian_b_bytes(int ld, int nIp) {
    return align_up((size_t)(2 * (size_t)nIp * nIp + 1) * ld * ld * sizeof(double), 1024);
}
}  // namespace

// workspace of oo_hessian_f64: the gathered class-layout operand + the class Hessian's own workspace (largest over
// the occ / act splits of nI, which this query does not know)
size_t hessian_ws_bytes(int ld, int nI) {
    const int nIp = nI + (nI & 1);
    size_t worst = 0;
    for (int na = 1; na <= nI; ++na) {
        const size_t w = class_hessian_ws_bytes(ld, nIp, nI - na, na, 1);
        worst = w > worst ? w : worst;
    }
    return full_hessian_b_bytes(ld, nIp) + worst;
}

// Hessian from the COMPLETE transformed tensor g' (oo_hessian_f64): the J / K classes are gathered out of g' into the
// class layout (one HBM-bound pass) and the block-structured class Hessian below does the rest -- the same kernels
// for both integral representations.
int hessian(const double *h, const double *g, const double *F, const double *d1, const double *d2,
            int no, int na, int N, int ld, const int32_t *pl, const int32_t *pr, int nk, double *H,
            void *ws, size_t ws_bytes, unsigned flags, cudaStream_t stream) {
    OO_REQUIRE(h && g && F && d1 && d2 && H && ws && pl && pr);
    OO_REQUIRE(no >= 0 && na > 0 && no + na <= N && ld >= N && (ld % 2) == 0 && nk > 0);
    const int nI = no + na, nIp = nI + (nI & 1);
    const size_t b_bytes = full_hessian_b_bytes(ld, nIp);
    const size_t c_bytes = class_hessian_ws_bytes(ld, nIp, no, na, 1);
    if (ws_bytes < b_bytes + c_bytes) return OO_ERR_WORKSPACE;
    if (nk > 65535) return OO_ERR_UNSUPPORTED;
    uint8_t *w = reinterpret_cast<uint8_t *>(ws);
    double *B = reinterpret_cast<double *>(w);
    const int64_t mat = (int64_t)ld * ld;
    int64_t blocks = ceil_div((2 * (int64_t)nIp * nIp + 1) * mat, 256);
    if (blocks > 16 * sm_count()) blocks = 16 * sm_count();
    hess_gather_class_kernel<<<(unsigned)blocks, 256, 0, stream>>>(h, g, nI, nIp, ld, B);
    OO_LAUNCH_CHECK();
    return class_hessian(B, F, d1, 0, d2, 0, no, na, N, ld, nIp, 1, pl, pr, nk, H, w + b_bytes, c_bytes, flags,
                         stream);
}

// Hessian from the class buffer of classes.cu: cls = [K rows; J rows; h' row] IS the B operand.
struct ClassHessLayout {
    int width;                       // ELL width of the sparse part
    int64_t lda_c, krows_c, ncol_c;  // C block
    size_t off_cnt, off_idx, off_val, off_flag, off_atc, off_bc, off_taa, off_tg, off_t, off_runs, total;
};

static ClassHessLayout class_hess_layout(int ld, int nIp, int no, int na, int batch) {
    ClassHessLayout L;
    const int64_t nI2 = (int64_t)nIp * nIp, mat = (int64_t)ld * ld, na2 = (int64_t)na * na;
    L.width = 2 * na * na + 2 * (no + na) + 8;
    L.ncol_c = na2 + no;
    L.lda_c = (L.ncol_c + 1) & ~1ll;
    L.krows_c = 2 * L.ncol_c + 1;
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off += align_up(bytes, 1024); return o; };
    L.off_cnt = take((size_t)batch * nI2 * sizeof(int));
    L.off_idx = take((size_t)batch * nI2 * L.width * sizeof(int));
    L.off_val = take((size_t)batch * nI2 * L.width * sizeof(double));
    L.off_flag = take(sizeof(int));
    L.off_atc = take((size_t)batch * L.krows_c * L.lda_c * sizeof(double));
    L.off_bc = take((size_t)batch * L.krows_c * mat * sizeof(double));
    L.off_taa = take((size_t)batch * L.ncol_c * mat * sizeof(double));
    L.off_tg = take((size_t)batch * no * 2 * na * mat * sizeof(double) + 1024);
    L.off_t = take((size_t)batch * nI2 * mat * sizeof(double));
    L.off_runs = take(assemble_scratch_bytes(ld));
    L.total = off;
    return L;
}

size_t class_hessian_ws_bytes(int ld, int nIp, int no, int na, int batch) {
    const HessLayout D = hess_layout(ld, nIp);
    const size_t dense = D.off_b + (D.total - D.off_t);          // At + T + pair runs (no gathered B); batch 1 only
    const size_t sparse = class_hess_layout(ld, nIp, no, na, batch).total;
    return dense > sparse ? dense : sparse;
}

static int class_hessian_dense(const double *cls, const double *F, const RdmView &rdm, int N, int ld, int nIp,
                               const int32_t *pl, const int32_t *pr, int nk, double *H, void *ws,
                               unsigned flags, cudaStream_t stream) {
    const HessLayout L = hess_layout(ld, nIp);
    uint8_t *w = reinterpret_cast<uint8_t *>(ws);
    double *At = reinterpret_cast<double *>(w);
    double *T = reinterpret_cast<double *>(w + L.off_b);
    const int64_t nI2 = (int64_t)nIp * nIp, mat = (int64_t)ld * ld;
    int64_t blocks = ceil_div(L.krows * L.lda, 256);
    if (blocks > 8 * sm_count()) blocks = 8 * sm_count();
    hess_build_at_kernel<<<(unsigned)blocks, 256, 0, stream>>>(rdm, nIp, 1, L.lda, At);
    OO_LAUNCH_CHECK();
    int rc = dgemm_tn(At, cls, T, nI2, mat, L.krows, L.lda, mat, mat, 1, 0, 0, 0, stream);
    if (rc) return rc;
    return launch_assemble(TView{T, nullptr, nullptr, rdm.no + rdm.na, nIp, rdm.no, rdm.na, 0, 0, 0, 0, 0}, F, pl, pr, nk, N, ld, 1,
                           H, w + L.off_b + (L.off_runs - L.off_t), flags, stream);
}

// batch evaluations: cls[b] (class buffers, contiguous), F[b] (ld^2), H[b] (nk^2); RDMs shared
// (stride 0) or per evaluation.
int class_hessian(const double *cls, const double *F, const double *d1, int64_t sd1, const double *d2,
                  int64_t sd2, int no, int na, int N, int ld, int nIp, int batch, const int32_t *pl,
                  const int32_t *pr, int nk, double *H, void *ws, size_t ws_bytes, unsigned flags,
                  cudaStream_t stream) {
    OO_REQUIRE(cls && F && d1 && d2 && H && ws && pl && pr);
    OO_REQUIRE(no >= 0 && na > 0 && no + na <= N && ld >= N && (ld % 2) == 0 && nk > 0 && batch > 0);
    const bool g_hessian_dense = (flags & OO_FLAG_HESSIAN_DENSE) != 0;
    const bool g_hessian_group_unstreamed = (flags & OO_FLAG_HESSIAN_GROUP_UNSTREAMED) != 0;
    OO_REQUIRE(nIp >= no + na && (nIp % 2) == 0 && nIp <= ld);
    const int rdm_batched = (batch > 1 && (sd1 != 0 || sd2 != 0)) ? 1 : 0;
    const int nsets = rdm_batched ? batch : 1;
    if (ws_bytes < class_hessian_ws_bytes(ld, nIp, no, na, batch)) return OO_ERR_WORKSPACE;
    if (nk > 65535 || batch > 65535) return OO_ERR_UNSUPPORTED;
    RdmView rdm{d1, d2, no, na};
    const int64_t nI2 = (int64_t)nIp * nIp, mat = (int64_t)ld * ld, na2 = (int64_t)na * na;
    const int64_t cls_stride = (2 * nI2 + 1) * mat;
    if (g_hessian_dense) {
        for (int b = 0; b < batch; ++b) {
            RdmView rb{d1 + b * sd1, d2 + b * sd2, no, na};
            int rc = class_hessian_dense(cls + b * cls_stride, F + b * mat, rb, N, ld, nIp, pl, pr, nk,
                                         H + (int64_t)b * nk * nk, ws, flags, stream);
            if (rc) return rc;
        }
        return OO_OK;
    }

    const ClassHessLayout L = class_hess_layout(ld, nIp, no, na, batch);
    uint8_t *w = reinterpret_cast<uint8_t *>(ws);
    int *cnt = reinterpret_cast<int *>(w + L.off_cnt);
    int *idx = reinterpret_cast<int *>(w + L.off_idx);
    double *val = reinterpret_cast<double *>(w + L.off_val);
    int *flag = reinterpret_cast<int *>(w + L.off_flag);
    double *Atc = reinterpret_cast<double *>(w + L.off_atc);
    double *Bc = reinterpret_cast<double *>(w + L.off_bc);
    double *Taa = reinterpret_cast<double *>(w + L.off_taa);
    double *Tg = reinterpret_cast<double *>(w + L.off_tg);
    double *T = reinterpret_cast<double *>(w + L.off_t);

    // What depends on the RDMs alone -- the ELL lists and the C-block coefficients -- is still in the workspace when
    // the caller says nothing changed since the previous call (a kappa sweep at fixed RDMs)
    const bool reuse = (flags & OO_FLAG_HESSIAN_REUSE_OPERANDS) != 0;
    // ELL lists of what lies outside the dense blocks (one table per set of RDMs)
    if (!reuse) {
        hess_sparse_build_kernel<<<dim3((unsigned)ceil_div(nI2, 8), (unsigned)nsets), 256, 0, stream>>>(
            rdm, sd1, sd2, nIp, 1, L.width, cnt, idx, val, flag);
        OO_LAUNCH_CHECK();
    }
    // C block: Tc[b] = Atc^T Bc[b]
    {
        int64_t blocks = ceil_div(L.krows_c * L.lda_c, 256);
        if (!reuse) {
            hess_dense_at_kernel<<<dim3((unsigned)blocks, (unsigned)nsets), 256, 0, stream>>>(rdm, sd1, sd2, nIp, 1,
                                                                                             L.lda_c, Atc);
            OO_LAUNCH_CHECK();
        }
        int64_t bx = ceil_div(mat / 2, 256);
        if (bx > 64) bx = 64;
        hess_dense_b_kernel<<<dim3((unsigned)bx, (unsigned)L.krows_c, (unsigned)batch), 256, 0, stream>>>(
            cls, cls_stride, no, na, nIp, mat, Bc);
        OO_LAUNCH_CHECK();
        int rc = dgemm_tn(Atc, Bc, Taa, L.ncol_c, mat, L.krows_c, L.lda_c, mat, mat, batch,
                          rdm_batched ? L.krows_c * L.lda_c : 0, L.krows_c * mat, L.ncol_c * mat, stream);
        if (rc) return rc;
    }
    // G blocks, one per occupied orbital
    if (no > 0) {
        const size_t smem = (size_t)4 * na * (2 * na + 1) * sizeof(double);
        if (smem > 48 * 1024) return OO_ERR_UNSUPPORTED;
        const size_t smem_stream = group_stream_smem_bytes(na);
        if (!g_hessian_group_unstreamed && mat >= 16 * kGrpTile && 2 * na <= 24 && smem_stream <= 220 * 1024 &&
            batch <= 65535) {
            // large ld^2: bulk-async streamed kernel, one CTA per SM, contiguous ranges of (i, tile) work items
            const int tiles_per_i = (int)ceil_div(mat, kGrpTile);
            const int total = no * tiles_per_i;
            const int ctas = total < sm_count() ? total : sm_count();
            const int items = (int)ceil_div(total, ctas);
            dim3 sgrid((unsigned)ceil_div(total, items), (unsigned)batch);
#define OO_GROUP_STREAM(CH)                                                                                        \
    do {                                                                                                           \
        static unsigned long long cfgd = 0;                                                                        \
        if (once_per_device(cfgd))                                                                                 \
            OO_CUDA_CHECK(cudaFuncSetAttribute(hess_group_stream_kernel<CH>,                                       \
                                               cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));          \
        hess_group_stream_kernel<CH><<<sgrid, 32 * kGrpWarps, smem_stream, stream>>>(cls, cls_stride, rdm, sd1, sd2,          \
                                                                         rdm_batched, nIp, 1, mat, Tg,             \
                                                                         tiles_per_i, items);                     \
    } while (0)
            if (2 * na <= 8) OO_GROUP_STREAM(1);
            else if (2 * na <= 16) OO_GROUP_STREAM(2);
            else OO_GROUP_STREAM(3);
#undef OO_GROUP_STREAM
        } else {
        dim3 grid((unsigned)no, (unsigned)ceil_div(mat / 2, 128), (unsigned)batch);
#define OO_GROUP(CH) hess_group_kernel<CH><<<grid, 128, smem, stream>>>(cls, cls_stride, rdm, sd1, sd2, rdm_batched, \
                                                                       nIp, 1, mat, Tg)
        // (measured at N = 256, na = 12: 8 / 12 / 24 columns per pass all take 0.48-0.51 ms -- DRAM latency bound)
        if (2 * na <= 8) OO_GROUP(8);
        else if (2 * na <= 16) OO_GROUP(16);
        else OO_GROUP(24);
#undef OO_GROUP
        }
        OO_LAUNCH_CHECK();
    }
    // the rest (occ-occ pairs i != j), plus anything a block column has outside its block
    {
        // occ-occ off-diagonal columns two at a time (they share their rows), everything else column by column
        const bool pairs = no >= 2 && !(flags & OO_FLAG_HESSIAN_SPMM_UNPAIRED) && (mat % 2) == 0;
        if (pairs) {
            dim3 pgrid((unsigned)(no * (no - 1) / 2), (unsigned)ceil_div(mat, kPairChunk), (unsigned)batch);
            hess_spmm_pair_kernel<<<pgrid, 256, 0, stream>>>(cls, cls_stride, cnt, idx, val, rdm_batched, L.width, no,
                                                             nIp, mat, T);
            OO_LAUNCH_CHECK();
        }
        int64_t ytiles = ceil_div(mat / 2, 256);
        if (pairs && ytiles > 8) ytiles = 8;              // what is left is (almost always) nothing: few CTAs per column
        dim3 grid((unsigned)nI2, (unsigned)ytiles, (unsigned)batch);
        const size_t smem = (size_t)L.width * (sizeof(double) + sizeof(int));
        if (smem > 48 * 1024) return OO_ERR_UNSUPPORTED;
        hess_spmm_kernel<<<grid, 256, smem, stream>>>(cls, cls_stride, cnt, idx, val, rdm_batched, L.width, no, na,
                                                   nIp, mat, T, Taa, Tg, pairs ? 1 : 0);
        OO_LAUNCH_CHECK();
    }
    return launch_assemble(TView{T, Taa, Tg, no + na, nIp, no, na, nI2 * mat, L.ncol_c * mat,
                                 (int64_t)no * 2 * na * mat, mat, (int64_t)nk * nk},
                           F, pl, pr, nk, N, ld, batch, H, w + L.off_runs, flags, stream);
}

namespace {
// P[b][i(i+1)/2 + j] = H[b][i][j], j <= i: the lower triangle of the symmetric Hessian, rows back to back
// (np.tril_indices(n) order).  Four rows per CTA; reads and writes are contiguous runs of i+1 doubles.
__global__ void __launch_bounds__(256) pack_lower_kernel(const double *__restrict__ H, int n, int64_t npk,
                                                         double *__restrict__ P) {
    const double *Hb = H + (int64_t)blockIdx.y * n * n;
    double *Pb = P + (int64_t)blockIdx.y * npk;
    const int i0 = blockIdx.x * 4;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const int i = i0 + r;
        if (i >= n) return;
        const double *src = Hb + (int64_t)i * n;
        double *dst = Pb + (int64_t)i * (i + 1) / 2;
        for (int j = threadIdx.x; j <= i; j += 256) dst[j] = src[j];
    }
}
}  // namespace

namespace {
__global__ void __launch_bounds__(256) copy_kernel(const double *__restrict__ src, double *__restrict__ dst, int64_t n) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) dst[i] = src[i];
}
}  // namespace

// dst[i] = src[i] by a kernel: src may be PINNED HOST memory (read over PCIe through the unified address space).
// Small inputs (kappa, RDMs) enter the device this way so that no DMA-engine copy of the compute stream can queue
// behind the multi-millisecond device->host copy of a Hessian that a copy stream has in flight.
int copy_f64(const double *src, double *dst, int64_t n, cudaStream_t stream) {
    OO_REQUIRE(src && dst && n >= 0);
    if (n == 0) return OO_OK;
    int64_t blocks = ceil_div(n, 256);
    if (blocks > 4 * sm_count()) blocks = 4 * sm_count();
    copy_kernel<<<(unsigned)blocks, 256, 0, stream>>>(src, dst, n);
    OO_LAUNCH_CHECK();
    return OO_OK;
}

int pack_lower(const double *H, int n, int batch, double *P, cudaStream_t stream) {
    OO_REQUIRE(H && P && n > 0 && batch > 0);
    if (batch > 65535) return OO_ERR_UNSUPPORTED;
    pack_lower_kernel<<<dim3((unsigned)ceil_div(n, 4), (unsigned)batch), 256, 0, stream>>>(
        H, n, (int64_t)n * (n + 1) / 2, P);
    OO_LAUNCH_CHECK();
    return OO_OK;
}

int full_rdms(const double *d1, const double *d2, int no, int na, int N, double *one_full,
              double *two_full, cudaStream_t stream) {
    OO_REQUIRE(d1 && d2 && one_full && two_full);
    OO_REQUIRE(no >= 0 && na > 0 && no + na <= N);
    RdmView rdm{d1, d2, no, na};
    int64_t blocks = ceil_div((int64_t)N * N * N * N, 256);
    if (blocks > 16 * sm_count()) blocks = 16 * sm_count();
    full_rdms_kernel<<<(unsigned)blocks, 256, 0, stream>>>(rdm, N, one_full, two_full);
    OO_LAUNCH_CHECK();
    return OO_OK;
}

size_t y_matrix_ws_bytes(int ld, int N) { return hess_layout(ld, N).total; }

int y_matrix(const double *g, const double *two_full, int N, int ld, double *Y, void *ws,
             size_t ws_bytes, cudaStream_t stream) {
    OO_REQUIRE(g && two_full && Y && ws);
    OO_REQUIRE(N > 0 && ld >= N && (ld % 2) == 0);
    const HessLayout L = hess_layout(ld, N);
    if (ws_bytes < L.total) return OO_ERR_WORKSPACE;
    uint8_t *w = reinterpret_cast<uint8_t *>(ws);
    double *At = reinterpret_cast<double *>(w);
    double *B = reinterpret_cast<double *>(w + L.off_b);
    double *T = reinterpret_cast<double *>(w + L.off_t);
    const int64_t N2 = (int64_t)N * N, mat = (int64_t)ld * ld;
    int64_t blocks = ceil_div(2 * N2 * L.lda, 256);
    if (blocks > 16 * sm_count()) blocks = 16 * sm_count();
    y_build_at_kernel<<<(unsigned)blocks, 256, 0, stream>>>(two_full, N, L.lda, At);
    OO_LAUNCH_CHECK();
    blocks = ceil_div(2 * N2 * mat, 256);
    if (blocks > 16 * sm_count()) blocks = 16 * sm_count();
    hess_gather_b_kernel<<<(unsigned)blocks, 256, 0, stream>>>(nullptr, g, N, ld, B);
    OO_LAUNCH_CHECK();
    int rc = dgemm_tn(At, B, T, N2, mat, 2 * N2, L.lda, mat, mat, 1, 0, 0, 0, stream);
    if (rc) return rc;
    blocks = ceil_div(N2 * N2, 256);
    if (blocks > 16 * sm_count()) blocks = 16 * sm_count();
    y_permute_kernel<<<(unsigned)blocks, 256, 0, stream>>>(T, N, ld, Y);
    OO_LAUNCH_CHECK();
    return OO_OK;
}

// ---- matrix-free Hessian: H v and diag(H) straight from the class buffer ----------------------------------------------
// For a block of vectors v (nk) let V be the skew matrix of each, V[l_j, r_j] = v_j = -V[r_j, l_j].  Then
//   W[p,q]  = -((F + F^T) V)[p,q] + [p in I] sum_{r in I, s} T[(p r),(q s)] V[r,s],      (H v)_j = W[l_j,r_j] - W[r_j,l_j]
// and with A_k[p,r] = At[k,(p r)] (at_value) the T part is
//   sum_k sum_s B[k][q,s] M_k[p,s],   M_k[p,s] = sum_r A_k[p,r] V[r,s]:
// every class plane B[k] is read once per block of vectors and multiplied (DMMA) by the few rows M_k has; neither T
// nor the nk x nk matrix is formed.  The diagonal needs four T elements per parameter, each a dot product of a column
// of At with one element of every plane.
namespace {

constexpr int kHvpQT = 32;                          // q rows per CTA tile (4 DMMA row tiles)
constexpr int kHvpSC = 32;                          // s columns per CTA tile (8 DMMA k-steps)
constexpr int kHvpSR = kHvpSC + 4;                  // shared-memory row stride (= 4 mod 32: conflict-free fragments)
constexpr int kHvpStages = 4;                       // class-plane tiles in flight per CTA
constexpr int kHvpMaxVec = 8;                       // vectors per pass at most
constexpr int kHvpCtas = 592;                       // target grid (a fixed number: the summation order, and with it every
                                                    // bit of the result, does not depend on the device)
constexpr size_t kHvpSmemMax = 200 * 1024;

// Non-zeros of one class row of At.  From the Kronecker structure of the full-space RDMs (gf1 / gf2) a row has at
// most na^2 + no + 4 of them (the act-act block, the occupied diagonal and a few occ-occ terms), below the width
// of the ELL table the T-matrix build uses; that width is kept here.
int hvp_width(int no, int na) { return 2 * na * na + 2 * (no + na) + 8; }

struct HvpLayout {
    int nvc, width, kc, rows_per, nsc, nqt;
    size_t smem, off_np, off_plist, off_pstart, off_er, off_ev, off_part, off_v, off_w, total;
};

size_t hvp_smem_bytes(int nI, int nvc) {
    const size_t ncol = (size_t)nI * nvc;
    return ((size_t)kHvpStages * kHvpQT * kHvpSR + ncol * kHvpSR + (ncol + 7) / 8 * 8 * kHvpSR +
            (size_t)nI * kHvpQT * nvc) * sizeof(double);
}

HvpLayout hvp_layout(int ld, int nIp, int no, int na, int nv) {
    HvpLayout L;
    const int nI = no + na;
    const int64_t krows = 2 * (int64_t)nIp * nIp + 1, mat = (int64_t)ld * ld;
    L.nvc = 0;
    for (int c = 1; c <= kHvpMaxVec && c <= nv; ++c)
        if (hvp_smem_bytes(nI, c) <= kHvpSmemMax) L.nvc = c;
    L.smem = hvp_smem_bytes(nI, L.nvc > 0 ? L.nvc : 1);
    L.width = hvp_width(no, na);
    L.nqt = (int)ceil_div(ld, kHvpQT);
    L.nsc = (int)ceil_div(ld, kHvpSC);
    const int64_t tiles = (int64_t)L.nqt * L.nsc;
    int64_t kc = ceil_div(kHvpCtas, tiles);
    if (kc > krows) kc = krows;
    L.rows_per = (int)ceil_div(krows, kc);
    L.kc = (int)ceil_div(krows, L.rows_per);
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off += align_up(bytes, 1024); return o; };
    L.off_np = take((size_t)krows * sizeof(int));
    L.off_plist = take((size_t)krows * nI * sizeof(int));
    L.off_pstart = take((size_t)krows * (nI + 1) * sizeof(int));
    L.off_er = take((size_t)krows * L.width * sizeof(int));
    L.off_ev = take((size_t)krows * L.width * sizeof(double));
    const int nvc = L.nvc > 0 ? L.nvc : 1;
    L.off_part = take((size_t)L.kc * L.nsc * nvc * nI * ld * sizeof(double));
    L.off_v = take((size_t)nvc * mat * sizeof(double));
    L.off_w = take((size_t)nvc * mat * sizeof(double));
    L.total = off;
    return L;
}

// One warp per class row k: its non-zero coefficients A_k[p,r] (p, r < nI) grouped by p -- the distinct p in
// plist[k][0, np), the entries of the i-th in [pstart[k][i], pstart[k][i+1]) with column r and value.
__global__ void __launch_bounds__(256)
hvp_table_kernel(RdmView rdm, int nIp, int64_t krows, int width, int *__restrict__ npk, int *__restrict__ plist,
                 int *__restrict__ pstart, int *__restrict__ er, double *__restrict__ ev) {
    const int lane = threadIdx.x & 31;
    const int64_t k = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (k >= krows) return;
    const int nI = rdm.no + rdm.na;
    int base = 0, np = 0;
    for (int p = 0; p < nI; ++p) {
        const int start = base;
        for (int r0 = 0; r0 < nI; r0 += 32) {
            const int r = r0 + lane;
            double v = 0.0;
            int m, n;
            if (r < nI) v = at_value(rdm, nIp, 1, k, p, r, m, n);
            const unsigned mask = __ballot_sync(0xffffffffu, v != 0.0);
            const int pos = base + __popc(mask & ((1u << lane) - 1u));
            if (v != 0.0 && pos < width) {
                er[k * width + pos] = r;
                ev[k * width + pos] = v;
            }
            base += __popc(mask);
        }
        if (base > start) {
            if (lane == 0) {
                plist[k * nI + np] = p;
                pstart[k * (nI + 1) + np] = min(start, width);
            }
            ++np;
        }
    }
    if (lane == 0) {
        pstart[k * (nI + 1) + np] = min(base, width);
        npk[k] = np;
    }
}

// Vm[v][l_j][r_j] = V[j][v0 + v] = -Vm[v][r_j][l_j]  (Vm zeroed before)
__global__ void hvp_scatter_kernel(const double *__restrict__ V, int nv, int v0, int nvc, const int32_t *__restrict__ pl,
                                   const int32_t *__restrict__ pr, int nk, int ld, double *__restrict__ Vm) {
    const int64_t total = (int64_t)nk * nvc, mat = (int64_t)ld * ld;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int j = (int)(i / nvc), v = (int)(i % nvc);
        const double x = V[(int64_t)j * nv + v0 + v];
        Vm[v * mat + (int64_t)pl[j] * ld + pr[j]] = x;
        Vm[v * mat + (int64_t)pr[j] * ld + pl[j]] = -x;
    }
}

__device__ __forceinline__ void cp_async16(void *smem_dst, const void *gsrc, uint32_t src_bytes) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_u32(smem_dst)), "l"(gsrc), "r"(src_bytes)
                 : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// The streamed pass.  CTA (q tile, s tile; range of class rows): for every row k of its range, the 32 x 32 tile
// B[k][q0.., s0..] arrives by cp.async in a four-stage ring, M_k[(p v), s] = sum_r A_k[p,r] V_v[r,s] is formed in
// shared memory from the CTA's slice of V (rows r in I), U[q, (p v)] = sum_s B[k][q,s] M_k[(p v), s] runs on DMMA,
// and U is added to the CTA's W[p][q][v] (each element by exactly one thread per row k: a fixed order).  The CTA
// writes its W to its own slice of `part`; hvp_reduce_kernel sums the slices in a fixed order.
__global__ void __launch_bounds__(256)
hvp_plane_kernel(const double *__restrict__ cls, int ld, int nI, int64_t krows, int rows_per, int nsc, int nvc,
                 const int *__restrict__ npk, const int *__restrict__ plist, const int *__restrict__ pstart,
                 const int *__restrict__ er, const double *__restrict__ ev, int width, const double *__restrict__ Vm,
                 double *__restrict__ part) {
    extern __shared__ __align__(16) double hv_smem[];
    const int ncol_max = nI * nvc;
    double *stage = hv_smem;                                          // [stages][QT][SR]
    double *Vs = stage + kHvpStages * kHvpQT * kHvpSR;                // [(r v)][SR]
    double *Ms = Vs + (size_t)ncol_max * kHvpSR;                      // [(i v)][SR], rows padded to 8
    double *Ws = Ms + (size_t)(ncol_max + 7) / 8 * 8 * kHvpSR;        // [p][QT][v]
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
    const int qt = blockIdx.x / nsc, sc = blockIdx.x % nsc;
    const int q0 = qt * kHvpQT, s0 = sc * kHvpSC;
    const int64_t mat = (int64_t)ld * ld;
    const int64_t k0 = (int64_t)blockIdx.y * rows_per, k1 = min(k0 + rows_per, krows);

    for (int x = tid; x < ncol_max * kHvpSC; x += blockDim.x) {
        const int row = x / kHvpSC, s = x % kHvpSC, r = row / nvc, v = row % nvc;
        Vs[row * kHvpSR + s] = s0 + s < ld ? Vm[v * mat + (int64_t)r * ld + s0 + s] : 0.0;
    }
    for (int x = tid; x < nI * kHvpQT * nvc; x += blockDim.x) Ws[x] = 0.0;

    auto issue = [&](int64_t k, int slot) {                           // 32 rows x 16 granules of 16 bytes
        for (int x = tid; x < kHvpQT * kHvpSC / 2; x += blockDim.x) {
            const int row = x / (kHvpSC / 2), c2 = 2 * (x % (kHvpSC / 2));
            const int q = q0 + row, s = s0 + c2;
            const bool ok = q < ld && s < ld;
            cp_async16(stage + (slot * kHvpQT + row) * kHvpSR + c2, ok ? cls + k * mat + (int64_t)q * ld + s : cls,
                       ok ? 16u : 0u);
        }
    };
    for (int i = 0; i < kHvpStages - 1; ++i) {
        if (k0 + i < k1) issue(k0 + i, i);
        cp_async_commit();
    }
    for (int64_t k = k0; k < k1; ++k) {
        const int it = (int)(k - k0), slot = it % kHvpStages;
        if (k + kHvpStages - 1 < k1) issue(k + kHvpStages - 1, (it + kHvpStages - 1) % kHvpStages);
        cp_async_commit();
        cp_async_wait<kHvpStages - 1>();
        const int np = npk[k], ncol = np * nvc, ncolp = (ncol + 7) & ~7;
        __syncthreads();                                              // tile k visible; Vs / Ws initialised
        for (int x = tid; x < ncolp * kHvpSC; x += blockDim.x) {
            const int col = x / kHvpSC, s = x % kHvpSC;
            double m = 0.0;
            if (col < ncol) {
                const int i = col / nvc, v = col % nvc;
                const int e1 = pstart[k * (nI + 1) + i + 1];
                for (int e = pstart[k * (nI + 1) + i]; e < e1; ++e)
                    m = fma(ev[k * width + e], Vs[(er[k * width + e] * nvc + v) * kHvpSR + s], m);
            }
            Ms[col * kHvpSR + s] = m;
        }
        __syncthreads();
        const double *st = stage + slot * kHvpQT * kHvpSR;
        for (int w = warp; w < 4 * (ncolp / 8); w += 8) {
            const int mt = w & 3, nt = w >> 2;
            double c0 = 0.0, c1 = 0.0;
#pragma unroll
            for (int ks = 0; ks < kHvpSC / 4; ++ks)
                dmma884(c0, c1, st[(8 * mt + g) * kHvpSR + 4 * ks + t], Ms[(8 * nt + g) * kHvpSR + 4 * ks + t]);
#pragma unroll
            for (int cc = 0; cc < 2; ++cc) {
                const int col = 8 * nt + 2 * t + cc;
                if (col < ncol) {
                    const int p = plist[k * nI + col / nvc], v = col % nvc;
                    Ws[(p * kHvpQT + 8 * mt + g) * nvc + v] += cc ? c1 : c0;
                }
            }
        }
        __syncthreads();                                              // stage slot and Ms free for reuse
    }
    cp_async_wait<0>();
    __syncthreads();
    double *out = part + (int64_t)(blockIdx.y * nsc + sc) * nvc * nI * ld;
    for (int x = tid; x < nI * kHvpQT * nvc; x += blockDim.x) {
        const int v = x % nvc, ql = (x / nvc) % kHvpQT, p = x / (nvc * kHvpQT);
        if (q0 + ql < ld) out[((int64_t)v * nI + p) * ld + q0 + ql] = Ws[x];
    }
}

// Wy[v][p][q] = sum over the slices of `part` (fixed order) for p in I, 0 elsewhere
__global__ void hvp_reduce_kernel(const double *__restrict__ part, int nslices, int nvc, int nI, int ld,
                                  double *__restrict__ Wy) {
    const int64_t mat = (int64_t)ld * ld, total = nvc * mat, slice = (int64_t)nvc * nI * ld;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int v = (int)(i / mat), p = (int)((i % mat) / ld), q = (int)(i % ld);
        double w = 0.0;
        if (p < nI) {
            const double *src = part + ((int64_t)v * nI + p) * ld + q;
            for (int j = 0; j < nslices; ++j) w += src[j * slice];
        }
        Wy[i] = w;
    }
}

// HV[j][v0 + v] = W[v][l_j][r_j] - W[v][r_j][l_j]
__global__ void hvp_gather_kernel(const double *__restrict__ W, int nvc, const int32_t *__restrict__ pl,
                                  const int32_t *__restrict__ pr, int nk, int ld, int nv, int v0,
                                  double *__restrict__ HV) {
    const int64_t total = (int64_t)nk * nvc, mat = (int64_t)ld * ld;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int j = (int)(i / nvc), v = (int)(i % nvc);
        const double *Wv = W + v * mat;
        HV[(int64_t)j * nv + v0 + v] = Wv[(int64_t)pl[j] * ld + pr[j]] - Wv[(int64_t)pr[j] * ld + pl[j]];
    }
}

// One warp per parameter j = (l, r):
//   H_jj = X(l,r,l,r) - X(l,r,r,l) - X(r,l,l,r) + X(r,l,r,l),  X(a,b,c,d) = -(F_ac + F_ca) d_bd + [a,c in I] T[(a c),(b d)]
// with the four T elements summed over the class rows in lane order and reduced by warp_sum (a fixed order).
__global__ void __launch_bounds__(256)
hess_diag_kernel(const double *__restrict__ cls, const double *__restrict__ F, RdmView rdm, int nIp, int ld,
                 const int32_t *__restrict__ pl, const int32_t *__restrict__ pr, int nk, double *__restrict__ diag) {
    const int lane = threadIdx.x & 31;
    const int j = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (j >= nk) return;
    const int l = pl[j], r = pr[j], nI = rdm.no + rdm.na;
    const bool li = l < nI, ri = r < nI;
    const int64_t krows = 2 * (int64_t)nIp * nIp + 1, mat = (int64_t)ld * ld;
    const int64_t o_llrr = (int64_t)r * ld + r, o_lrrl = (int64_t)r * ld + l, o_rllr = (int64_t)l * ld + r,
                  o_rrll = (int64_t)l * ld + l;
    double t = 0.0;                                   // T[(l l),(r r)] - T[(l r),(r l)] - T[(r l),(l r)] + T[(r r),(l l)]
    if (li || ri) {
        for (int64_t k = lane; k < krows; k += 32) {
            const double *Bk = cls + k * mat;
            int m, n;
            if (li) {
                const double a = at_value(rdm, nIp, 1, k, l, l, m, n);
                if (a != 0.0) t = fma(a, Bk[o_llrr], t);
            }
            if (li && ri) {
                const double a = at_value(rdm, nIp, 1, k, l, r, m, n);
                if (a != 0.0) t = fma(-a, Bk[o_lrrl], t);
                const double b = at_value(rdm, nIp, 1, k, r, l, m, n);
                if (b != 0.0) t = fma(-b, Bk[o_rllr], t);
            }
            if (ri) {
                const double a = at_value(rdm, nIp, 1, k, r, r, m, n);
                if (a != 0.0) t = fma(a, Bk[o_rrll], t);
            }
        }
    }
    t = warp_sum(t);
    if (lane == 0) {
        const double Fll = F[(int64_t)l * ld + l], Frr = F[(int64_t)r * ld + r];
        const double Fx = l == r ? F[(int64_t)l * ld + r] + F[(int64_t)r * ld + l] : 0.0;
        diag[j] = -2.0 * Fll + 2.0 * Fx - 2.0 * Frr + t;
    }
}

}  // namespace

size_t class_hessian_vector_ws_bytes(int ld, int nIp, int no, int na, int nv) {
    return hvp_layout(ld, nIp, no, na, nv).total;
}

size_t hessian_vector_ws_bytes(int ld, int nI, int na, int nv) {
    const int nIp = nI + (nI & 1);
    return full_hessian_b_bytes(ld, nIp) + class_hessian_vector_ws_bytes(ld, nIp, nI - na, na, nv);
}

size_t hessian_diagonal_ws_bytes(int ld, int nI) { return full_hessian_b_bytes(ld, nI + (nI & 1)); }

int dgemm_small(int transA, int transB, int M, int N, int K, double alpha, const double *A, int lda,
                int64_t strideA, const double *B, int ldb, int64_t strideB, double beta,
                const double *E, int lde, int64_t strideE, double gamma, double *D, int ldd,
                int64_t strideD, int batch, cudaStream_t stream, int eye_n);

// HV = H V for one evaluation: V, HV are nk x nv row-major.
int class_hessian_vector(const double *cls, const double *F, const double *d1, const double *d2, int no, int na,
                         int N, int ld, int nIp, const int32_t *pl, const int32_t *pr, int nk, const double *V,
                         int nv, double *HV, void *ws, size_t ws_bytes, cudaStream_t stream) {
    OO_REQUIRE(cls && F && d1 && d2 && V && HV && ws && pl && pr);
    OO_REQUIRE(no >= 0 && na > 0 && no + na <= N && ld >= N && (ld % 2) == 0 && nk > 0 && nv > 0);
    OO_REQUIRE(nIp >= no + na && (nIp % 2) == 0 && nIp <= ld);
    const HvpLayout L = hvp_layout(ld, nIp, no, na, nv);
    if (L.nvc == 0) return OO_ERR_UNSUPPORTED;
    if (ws_bytes < L.total) return OO_ERR_WORKSPACE;
    if (L.kc > 65535) return OO_ERR_UNSUPPORTED;
    const int nI = no + na;
    const int64_t krows = 2 * (int64_t)nIp * nIp + 1, mat = (int64_t)ld * ld;
    uint8_t *w = reinterpret_cast<uint8_t *>(ws);
    int *npk = reinterpret_cast<int *>(w + L.off_np);
    int *plist = reinterpret_cast<int *>(w + L.off_plist);
    int *pstart = reinterpret_cast<int *>(w + L.off_pstart);
    int *er = reinterpret_cast<int *>(w + L.off_er);
    double *ev = reinterpret_cast<double *>(w + L.off_ev);
    double *part = reinterpret_cast<double *>(w + L.off_part);
    double *Vm = reinterpret_cast<double *>(w + L.off_v);
    double *Wm = reinterpret_cast<double *>(w + L.off_w);
    const RdmView rdm{d1, d2, no, na};
    hvp_table_kernel<<<(unsigned)ceil_div(krows, 8), 256, 0, stream>>>(rdm, nIp, krows, L.width, npk, plist, pstart,
                                                                      er, ev);
    OO_LAUNCH_CHECK();
    static unsigned long long cfgd = 0;
    if (once_per_device(cfgd))
        OO_CUDA_CHECK(cudaFuncSetAttribute(hvp_plane_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           (int)kHvpSmemMax));
    const int cap = 4 * sm_count();
    for (int v0 = 0; v0 < nv; v0 += L.nvc) {
        const int nvc = nv - v0 < L.nvc ? nv - v0 : L.nvc;
        OO_CUDA_CHECK(cudaMemsetAsync(Vm, 0, (size_t)nvc * mat * sizeof(double), stream));
        int64_t blocks = ceil_div((int64_t)nk * nvc, 256);
        hvp_scatter_kernel<<<(unsigned)(blocks < cap ? blocks : cap), 256, 0, stream>>>(V, nv, v0, nvc, pl, pr, nk, ld,
                                                                                        Vm);
        OO_LAUNCH_CHECK();
        hvp_plane_kernel<<<dim3((unsigned)(L.nqt * L.nsc), (unsigned)L.kc), 256, hvp_smem_bytes(nI, nvc), stream>>>(
            cls, ld, nI, krows, L.rows_per, L.nsc, nvc, npk, plist, pstart, er, ev, L.width, Vm, part);
        OO_LAUNCH_CHECK();
        blocks = ceil_div(nvc * mat, 256);
        hvp_reduce_kernel<<<(unsigned)(blocks < cap ? blocks : cap), 256, 0, stream>>>(part, L.kc * L.nsc, nvc, nI, ld,
                                                                                       Wm);
        OO_LAUNCH_CHECK();
        // W -= F V  and  W -= F^T V   (the one-body part of X, on the small DMMA GEMM; E aliases D)
        for (int tr = 0; tr < 2; ++tr) {
            int rc = dgemm_small(tr, 0, ld, ld, ld, -1.0, F, ld, 0, Vm, ld, mat, 1.0, Wm, ld, mat, 0.0, Wm, ld, mat,
                                 nvc, stream, 0);
            if (rc) return rc;
        }
        blocks = ceil_div((int64_t)nk * nvc, 256);
        hvp_gather_kernel<<<(unsigned)(blocks < cap ? blocks : cap), 256, 0, stream>>>(Wm, nvc, pl, pr, nk, ld, nv, v0,
                                                                                       HV);
        OO_LAUNCH_CHECK();
    }
    return OO_OK;
}

int class_hessian_diagonal(const double *cls, const double *F, const double *d1, const double *d2, int no, int na,
                           int N, int ld, int nIp, const int32_t *pl, const int32_t *pr, int nk, double *diag,
                           cudaStream_t stream) {
    OO_REQUIRE(cls && F && d1 && d2 && diag && pl && pr);
    OO_REQUIRE(no >= 0 && na > 0 && no + na <= N && ld >= N && (ld % 2) == 0 && nk > 0);
    OO_REQUIRE(nIp >= no + na && (nIp % 2) == 0 && nIp <= ld);
    hess_diag_kernel<<<(unsigned)ceil_div(nk, 8), 256, 0, stream>>>(cls, F, RdmView{d1, d2, no, na}, nIp, ld, pl, pr,
                                                                    nk, diag);
    OO_LAUNCH_CHECK();
    return OO_OK;
}

// (h', g') forms: the class layout is gathered out of the complete g' into the workspace (as oo_hessian_f64 does)
static int gather_class_layout(const double *h, const double *g, int nI, int ld, double *B, cudaStream_t stream) {
    const int nIp = nI + (nI & 1);
    int64_t blocks = ceil_div((2 * (int64_t)nIp * nIp + 1) * ld * ld, 256);
    if (blocks > 16 * sm_count()) blocks = 16 * sm_count();
    hess_gather_class_kernel<<<(unsigned)blocks, 256, 0, stream>>>(h, g, nI, nIp, ld, B);
    OO_LAUNCH_CHECK();
    return OO_OK;
}

int hessian_vector(const double *h, const double *g, const double *F, const double *d1, const double *d2, int no,
                   int na, int N, int ld, const int32_t *pl, const int32_t *pr, int nk, const double *V, int nv,
                   double *HV, void *ws, size_t ws_bytes, cudaStream_t stream) {
    OO_REQUIRE(h && g && F && d1 && d2 && V && HV && ws && pl && pr);
    OO_REQUIRE(no >= 0 && na > 0 && no + na <= N && ld >= N && (ld % 2) == 0 && nk > 0 && nv > 0);
    const int nI = no + na, nIp = nI + (nI & 1);
    const size_t b_bytes = full_hessian_b_bytes(ld, nIp);
    if (ws_bytes < b_bytes) return OO_ERR_WORKSPACE;
    uint8_t *w = reinterpret_cast<uint8_t *>(ws);
    const HvpLayout L = hvp_layout(ld, nIp, no, na, nv);
    if (L.nvc == 0) return OO_ERR_UNSUPPORTED;
    if (ws_bytes < b_bytes + L.total) return OO_ERR_WORKSPACE;
    int rc = gather_class_layout(h, g, nI, ld, reinterpret_cast<double *>(w), stream);
    if (rc) return rc;
    return class_hessian_vector(reinterpret_cast<double *>(w), F, d1, d2, no, na, N, ld, nIp, pl, pr, nk, V, nv, HV,
                                w + b_bytes, ws_bytes - b_bytes, stream);
}

int hessian_diagonal(const double *h, const double *g, const double *F, const double *d1, const double *d2, int no,
                     int na, int N, int ld, const int32_t *pl, const int32_t *pr, int nk, double *diag, void *ws,
                     size_t ws_bytes, cudaStream_t stream) {
    OO_REQUIRE(h && g && F && d1 && d2 && diag && ws && pl && pr);
    OO_REQUIRE(no >= 0 && na > 0 && no + na <= N && ld >= N && (ld % 2) == 0 && nk > 0);
    const int nI = no + na, nIp = nI + (nI & 1);
    if (ws_bytes < full_hessian_b_bytes(ld, nIp)) return OO_ERR_WORKSPACE;
    int rc = gather_class_layout(h, g, nI, ld, reinterpret_cast<double *>(ws), stream);
    if (rc) return rc;
    return class_hessian_diagonal(reinterpret_cast<double *>(ws), F, d1, d2, no, na, N, ld, nIp, pl, pr, nk, diag,
                                  stream);
}

}  // namespace oo


extern "C" int oo_hessian_f64(const double *h_mo, const double *g_mo, const double *F,
                              const double *gamma, const double *Gamma, int no, int na, int N, int ld,
                              const int32_t *pair_l, const int32_t *pair_r, int nk, double *H, void *ws,
                              size_t ws_bytes, unsigned flags, void *stream) {
    return oo::hessian(h_mo, g_mo, F, gamma, Gamma, no, na, N, ld, pair_l, pair_r, nk, H, ws, ws_bytes, flags,
                       (cudaStream_t)stream);
}

extern "C" int oo_copy_f64(const double *src, double *dst, int64_t n, void *stream) {
    return oo::copy_f64(src, dst, n, (cudaStream_t)stream);
}

extern "C" int oo_pack_lower_f64(const double *H, int n, int batch, double *packed, void *stream) {
    return oo::pack_lower(H, n, batch, packed, (cudaStream_t)stream);
}

extern "C" int oo_full_rdms_f64(const double *gamma, const double *Gamma, int no, int na, int N,
                                double *one_full, double *two_full, void *stream) {
    return oo::full_rdms(gamma, Gamma, no, na, N, one_full, two_full, (cudaStream_t)stream);
}

extern "C" int oo_y_matrix_f64(const double *g_mo, const double *two_full, int N, int ld, double *Y,
                               void *ws, size_t ws_bytes, void *stream) {
    return oo::y_matrix(g_mo, two_full, N, ld, Y, ws, ws_bytes, (cudaStream_t)stream);
}

extern "C" int oo_class_hessian_f64(const double *cls, const double *F, const double *gamma,
                                    int64_t stride_rdm1, const double *Gamma, int64_t stride_rdm2, int no,
                                    int na, int N, int ld, int nIp, int batch, const int32_t *pair_l,
                                    const int32_t *pair_r, int nk, double *H, void *ws, size_t ws_bytes,
                                    unsigned flags, void *stream) {
    return oo::class_hessian(cls, F, gamma, stride_rdm1, Gamma, stride_rdm2, no, na, N, ld, nIp, batch, pair_l,
                             pair_r, nk, H, ws, ws_bytes, flags, (cudaStream_t)stream);
}

extern "C" int oo_class_hessian_vector_f64(const double *cls, const double *F, const double *gamma,
                                           const double *Gamma, int no, int na, int N, int ld, int nIp,
                                           const int32_t *pair_l, const int32_t *pair_r, int nk, const double *V,
                                           int nv, double *HV, void *ws, size_t ws_bytes, void *stream) {
    return oo::class_hessian_vector(cls, F, gamma, Gamma, no, na, N, ld, nIp, pair_l, pair_r, nk, V, nv, HV, ws,
                                    ws_bytes, (cudaStream_t)stream);
}

extern "C" int oo_class_hessian_diagonal_f64(const double *cls, const double *F, const double *gamma,
                                             const double *Gamma, int no, int na, int N, int ld, int nIp,
                                             const int32_t *pair_l, const int32_t *pair_r, int nk, double *diag,
                                             void *ws, size_t ws_bytes, void *stream) {
    (void)ws;
    (void)ws_bytes;
    return oo::class_hessian_diagonal(cls, F, gamma, Gamma, no, na, N, ld, nIp, pair_l, pair_r, nk, diag,
                                      (cudaStream_t)stream);
}

extern "C" int oo_hessian_vector_f64(const double *h_mo, const double *g_mo, const double *F, const double *gamma,
                                     const double *Gamma, int no, int na, int N, int ld, const int32_t *pair_l,
                                     const int32_t *pair_r, int nk, const double *V, int nv, double *HV, void *ws,
                                     size_t ws_bytes, void *stream) {
    return oo::hessian_vector(h_mo, g_mo, F, gamma, Gamma, no, na, N, ld, pair_l, pair_r, nk, V, nv, HV, ws, ws_bytes,
                              (cudaStream_t)stream);
}

extern "C" int oo_hessian_diagonal_f64(const double *h_mo, const double *g_mo, const double *F, const double *gamma,
                                       const double *Gamma, int no, int na, int N, int ld, const int32_t *pair_l,
                                       const int32_t *pair_r, int nk, double *diag, void *ws, size_t ws_bytes,
                                       void *stream) {
    return oo::hessian_diagonal(h_mo, g_mo, F, gamma, Gamma, no, na, N, ld, pair_l, pair_r, nk, diag, ws, ws_bytes,
                                (cudaStream_t)stream);
}
