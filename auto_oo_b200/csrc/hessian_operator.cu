// Matrix-free orbital Hessian: H v and diag(H) straight from the class buffer of classes.cu.
//
// For a block of vectors v (nk) let V be the skew matrix of each, V[l_j, r_j] = v_j = -V[r_j, l_j].  Then
//   W[p,q]  = -((F + F^T) V)[p,q] + [p in I] sum_{r in I, s} T[(p r),(q s)] V[r,s],      (H v)_j = W[l_j,r_j] - W[r_j,l_j]
// and with A_k[p,r] = At[k,(p r)] (at_value) the T part is
//   sum_k sum_s B[k][q,s] M_k[p,s],   M_k[p,s] = sum_r A_k[p,r] V[r,s]:
// every class plane B[k] is read once per block of vectors and multiplied (DMMA) by the few rows M_k has; neither T
// nor the nk x nk matrix is formed.  The diagonal needs four T elements per parameter, each a dot product of a column
// of At with one element of every plane.
#include "hessian_terms.cuh"

namespace oo {

namespace {

constexpr int kHvpQT = 32;                          // q rows per CTA tile (4 DMMA row tiles)
constexpr int kHvpSC = 32;                          // s columns per CTA tile (8 DMMA k-steps)
constexpr int kHvpSR = kHvpSC + 4;                  // shared-memory row stride (= 4 mod 32: conflict-free fragments)
constexpr int kHvpStages = 4;                       // class-plane tiles in flight per CTA
constexpr int kHvpMaxVec = 8;                       // vectors per pass at most
constexpr int kHvpCtas = 592;                       // target grid (a fixed number: the summation order, and with it every
                                                    // bit of the result, does not depend on the device)
constexpr size_t kHvpSmemMax = 200 * 1024;

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
    L.width = ell_width(no, na);
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
            if (r < nI) v = at_value(rdm, nIp, k, p, r, m, n);
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
                const double a = at_value(rdm, nIp, k, l, l, m, n);
                if (a != 0.0) t = fma(a, Bk[o_llrr], t);
            }
            if (li && ri) {
                const double a = at_value(rdm, nIp, k, l, r, m, n);
                if (a != 0.0) t = fma(-a, Bk[o_lrrl], t);
                const double b = at_value(rdm, nIp, k, r, l, m, n);
                if (b != 0.0) t = fma(-b, Bk[o_rllr], t);
            }
            if (ri) {
                const double a = at_value(rdm, nIp, k, r, r, m, n);
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
