// The coefficients At[k, (p r)] of the orbital Hessian's T-matrix, shared by the T-matrix Hessian (hessian.cu) and
// the matrix-free operator (hessian_operator.cu):
//   T[(p r),(q s)] = sum_k At[k,(p r)] B[k,(q s)],   B = the class buffer of classes.cu.
#pragma once
#include "common.cuh"

namespace oo {

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

// At rows: [0,nIp^2) exchange-type, [nIp^2, 2nIp^2) Coulomb-type, 2nIp^2: one-body, where nIp is the padded class
// index of the class buffer (gf1/gf2 return 0 for indices beyond occ+act).  Exchange row k < nIp^2 stands for
// (m, n) = (k mod nIp, k / nIp), the order in which classes.cu stores K[n,m,a,b]; Coulomb row nIp^2 + k for
// (m, n) = (k / nIp, k mod nIp).  `m`, `n` receive the pair the row stands for (-1 for the one-body row).
__device__ __forceinline__ double at_value(const RdmView &rdm, int nIp, int64_t k, int p, int r, int &m, int &n) {
    const int nI2 = nIp * nIp;
    if (k < nI2) {
        n = (int)(k / nIp);
        m = (int)(k % nIp);
        return 2.0 * (gf2(rdm, p, m, r, n) + gf2(rdm, p, m, n, r));
    }
    if (k < 2 * nI2) {
        const int kk = (int)(k - nI2);
        m = kk / nIp;
        n = kk % nIp;
        return 2.0 * gf2(rdm, p, r, m, n);
    }
    m = n = -1;
    return 2.0 * gf1(rdm, p, r);
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

// Width of the ELL tables of At: the non-zeros of a column outside its dense block (hess_sparse_build_kernel) and
// the non-zeros of one class row (hvp_table_kernel).  From the Kronecker structure of the full-space RDMs a row has
// at most na^2 + no + 4 of them (the act-act block, the occupied diagonal and a few occ-occ terms), a column
// (tests/test_oracle.py::test_hessian_sparse_row_bound) at most this width.
inline int ell_width(int no, int na) { return 2 * na * na + 2 * (no + na) + 8; }

}  // namespace oo
