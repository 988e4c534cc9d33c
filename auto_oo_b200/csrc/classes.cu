// Partial ("class") integral transformation: only the two integral classes the energy, the
// orbital gradient and the I-space Hessian read,
//   J[m,n,a,b] = g'[a,b,m,n] = (ab|mn)      K[n,m,a,b] = g'[a,m,n,b] = (am|nb)
// with m, n in I = occ + act (padded to nIp) and a, b general, instead of the complete
// g'[i,j,k,l] of general_4index_transform (reference oo_energy.py:21-30).  The numbers every
// consumer reads are the same sums in the same association as the full transform followed by
// slicing; the cost drops from 8 N^5 to 2 N^4 nI + 12 N^3 nI^2 flop.
//
// Every step is the rotating TN-GEMM of dgemm_tn.cu (the contracted LEADING index leaves, its
// image is appended at the back), starting from the pair-transposed AO tensor
// gp[r,s,p,q] = g[p,q,r,s] (built once per problem by oo_transpose_f64; no symmetry of g is assumed):
//   Q1            T1[s,p,q,m]  = sum_r gp[r,(s p q)] C[r,m]        2 N^4 nI flop   (m < nIp)
//   J:  Q2        X[p,q,m,n]   = sum_s T1[s,(p q m)] C[s,n]
//       Q3        X'[q,m,n,a]  = sum_p X[p,(q m n)]  C[p,a]
//       Q4        J[m,n,a,b]   = sum_q X'[q,(m n a)] C[q,b]
//   K:  swap      T1t[q,p,s,m] = T1[s,p,q,m]                       (second store in Q1's epilogue)
//       K2        X[p,s,n,m]   = sum_q T1t[q,(p s n)] C[q,m]
//       K3        X'[s,n,m,a]  = sum_p X[p,(s n m)]   C[p,a]
//       K4        K[n,m,a,b]   = sum_s X'[s,(n m a)]  C[s,b]
// The results land in ONE buffer  cls = [K rows (nIp^2) ; J rows (nIp^2) ; h' row], each row ld^2,
// which is exactly the B operand of the Hessian's T-matrix GEMM (hessian.cu) -- no gather pass.
#include "common.cuh"

namespace oo {

namespace {

// dst[c][r] = src[r][c]  (rows x cols doubles), 32x32 tiles through padded shared memory
__global__ void __launch_bounds__(256) transpose_kernel(const double *__restrict__ src,
                                                        double *__restrict__ dst, int64_t rows,
                                                        int64_t cols) {
    __shared__ double tile[32][33];
    const int64_t c0 = (int64_t)blockIdx.x * 32, r0 = (int64_t)blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
#pragma unroll
    for (int j = ty; j < 32; j += 8) {
        const int64_t r = r0 + j, c = c0 + tx;
        if (r < rows && c < cols) tile[j][tx] = src[r * cols + c];
    }
    __syncthreads();
#pragma unroll
    for (int j = ty; j < 32; j += 8) {
        const int64_t c = c0 + j, r = r0 + tx;
        if (r < rows && c < cols) dst[c * rows + r] = tile[tx][j];
    }
}

}  // namespace

int transpose(const double *src, double *dst, int64_t rows, int64_t cols, cudaStream_t stream) {
    OO_REQUIRE(src && dst && rows > 0 && cols > 0 && src != dst);
    const int64_t gx = ceil_div(cols, 32), gy = ceil_div(rows, 32);
    if (gx > 0x7fffffffll || gy > 65535) return OO_ERR_UNSUPPORTED;
    transpose_kernel<<<dim3((unsigned)gx, (unsigned)gy), 256, 0, stream>>>(src, dst, rows, cols);
    OO_LAUNCH_CHECK();
    return OO_OK;
}

size_t class_transform_ws_bytes(int ld, int nIp, int batch) {
    const size_t ld2 = (size_t)ld * ld;
    return (size_t)batch * (2 * ld2 * ld * nIp + 2 * ld2 * nIp * nIp) * sizeof(double);
}

size_t class_buffer_bytes(int ld, int nIp) {
    return (size_t)(2 * (size_t)nIp * nIp + 1) * ld * ld * sizeof(double);
}

// batch evaluations at once: C[b] (strideC, 0 = shared), gp[b] (strideG, 0 = shared AO integrals),
// cls[b] contiguous class buffers.  Every step is one batched TN-GEMM launch.
int class_transform(const double *gp, int64_t strideG, const double *C, int64_t strideC, int N, int ld,
                    int nIp, int batch, double *cls, void *ws, size_t ws_bytes, cudaStream_t stream) {
    OO_REQUIRE(gp && C && cls && ws);
    OO_REQUIRE(N > 0 && ld >= N && (ld % 2) == 0 && nIp > 0 && (nIp % 2) == 0 && nIp <= ld && batch > 0);
    if (ws_bytes < class_transform_ws_bytes(ld, nIp, batch)) return OO_ERR_WORKSPACE;
    if (ld > 65535) return OO_ERR_UNSUPPORTED;
    const int64_t ld2 = (int64_t)ld * ld, ld3 = ld2 * ld, nI2 = (int64_t)nIp * nIp;
    const int64_t sT1 = ld3 * nIp, sX = ld2 * nI2, sCls = (2 * nI2 + 1) * ld2;
    double *T1 = reinterpret_cast<double *>(ws);
    double *T1t = T1 + (int64_t)batch * sT1;
    double *X = T1t + (int64_t)batch * sT1;
    double *Xp = X + (int64_t)batch * sX;
    double *Kout = cls, *Jout = cls + nI2 * ld2;
    int rc;
#define Q(in, sIn, out, sOut, M, Ncols)                                                                  \
    if ((rc = dgemm_tn((in), C, (out), (M), (Ncols), ld, (M), ld, (Ncols), batch, (sIn), strideC, (sOut), \
                       stream)))                                                                         \
    return rc
    // Q1 writes T1[s,p,q,m] and its (s <-> q) swapped copy T1t[q,p,s,m] from the same accumulators
    if ((rc = dgemm_tn_swap02(gp, C, T1, T1t, ld, ld, ld, nIp, ld, ld3, ld, nIp, batch, strideG, strideC, sT1,
                              stream)))
        return rc;
    Q(T1, sT1, X, sX, ld2 * nIp, nIp);         // [p,q,m,n]
    Q(X, sX, Xp, sX, ld * nI2, ld);            // [q,m,n,a]
    Q(Xp, sX, Jout, sCls, nI2 * ld, ld);       // [m,n,a,b]
    Q(T1t, sT1, X, sX, ld2 * nIp, nIp);        // [p,s,n,m]
    Q(X, sX, Xp, sX, ld * nI2, ld);            // [s,n,m,a]
    Q(Xp, sX, Kout, sCls, nI2 * ld, ld);       // [n,m,a,b]
#undef Q
    return OO_OK;
}


// =====================================================================================
// Symmetric variant.  Real AO integrals have the 8-fold symmetry (pq|rs) = (qp|rs) = (rs|pq);
// eri_symmetry_defect measures it and the host selects this path only when the defect is
// round-off.  Then
//   * the AO tensor is kept with the LAST pair packed, gpk[r,s,pq] = g[r,s,p,q], p >= q
//     (half the HBM of g_pairT, which equals g itself), and Q1 runs over packed pairs only:
//       Q1   T1[s,pq,m] = sum_r gpk[r,(s pq)] C[r,m]              N^4 nI flop (half of the general Q1)
//     its epilogue also writes the unpacked, pair-first copy T1t[q,p,s,m] = T1t[p,q,s,m] for K;
//   * J[m,n,a,b] = J[n,m,a,b] and K[n,m,a,b] = K[m,n,b,a]: only class pairs m >= n go through
//     the last two quarters (packed pair index mn).  The "pack" and "expand" steps below are epilogue modes of
//     the GEMMs next to them (dgemm_tn_class_pack / dgemm_tn_class_expand: the quarter-2 GEMM stores only n <= m,
//     packed; the last-quarter GEMM stores (m n) and its mirror (n m), transposed for K); the separate kernels
//     remain behind OO_FLAG_CLASS_UNFUSED_PACK for A/B tests.
//       J:  Q2   X[pq,m,n]    = sum_s T1[s,(pq m)] C[s,n]
//           pack Xf[p,q,mn]   = X[tri(p,q),m,n]                     (pair index unpacked, class pair packed)
//           Q3   X'[q,mn,a]   = sum_p Xf[p,(q mn)] C[p,a]
//           Q4   Jp[mn,a,b]   = sum_q X'[q,(mn a)] C[q,b]
//       K:  K2   X2[p,s,m,n]  = sum_q T1t[q,(p s m)] C[q,n]
//           pack X2p[p,s,mn]  = X2[p,s,m,n]
//           K3   X3[s,mn,a]   = sum_p X2p[p,(s mn)] C[p,a]
//           K4   Kp[mn,a,b]   = sum_s X3[s,(mn a)] C[s,b]           = g'[a,n,m,b]
//       expand   J[m,n] = J[n,m] = Jp[mn];  K[m,n] = Kp[mn],  K[n,m] = Kp[mn]^T
// Total 2 N^4 nI / 2 + ~7 N^3 nI^2 flop: 4.2e11 at N=256, nI=44 instead of 7.7e11.
namespace {

__host__ __device__ inline int64_t tri_count(int n) { return (int64_t)n * (n + 1) / 2; }

__device__ __forceinline__ void tri_decode(int pq, int &p, int &q) {
    p = (int)((sqrt(8.0 * pq + 1.0) - 1.0) * 0.5);
    while ((p + 1) * (p + 2) / 2 <= pq) ++p;
    while (p * (p + 1) / 2 > pq) --p;
    q = pq - p * (p + 1) / 2;
}

__device__ __forceinline__ void atomic_max_nonneg(double *addr, double v) {
    // non-negative doubles order like their bit patterns
    atomicMax(reinterpret_cast<unsigned long long *>(addr), (unsigned long long)__double_as_longlong(v));
}

// defect[0] = max |g[p,q,r,s] - g[q,p,r,s]|, defect[1] = max |g[p,q,r,s] - g[r,s,p,q]|, defect[2] = max |g|
// g viewed as a (ld^2 x ld^2) matrix; 32x32 tiles, the mirrored tile read transposed through smem.
__global__ void __launch_bounds__(256) eri_defect_kernel(const double *__restrict__ g, int ld,
                                                         double *__restrict__ defect) {
    __shared__ double tile[32][33];
    __shared__ double red[32];
    const int64_t ld2 = (int64_t)ld * ld;
    const int64_t c0 = (int64_t)blockIdx.x * 32, r0 = (int64_t)blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    for (int j = ty; j < 32; j += 8) {      // mirrored tile: rows c0.., cols r0..
        const int64_t r = c0 + j, c = r0 + tx;
        tile[j][tx] = (r < ld2 && c < ld2) ? g[r * ld2 + c] : 0.0;
    }
    __syncthreads();
    double d_pq = 0.0, d_pair = 0.0, amax = 0.0;
    for (int j = ty; j < 32; j += 8) {
        const int64_t r = r0 + j, c = c0 + tx;
        if (r < ld2 && c < ld2) {
            const double v = g[r * ld2 + c];
            amax = fmax(amax, fabs(v));
            d_pair = fmax(d_pair, fabs(v - tile[tx][j]));
            const int p = (int)(r / ld), q = (int)(r % ld);
            d_pq = fmax(d_pq, fabs(v - g[((int64_t)q * ld + p) * ld2 + c]));
        }
    }
    double vals[3] = {d_pq, d_pair, amax};
    for (int k = 0; k < 3; ++k) {
        double v = vals[k];
        for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
        __syncthreads();
        if (tx == 0) red[ty] = v;
        __syncthreads();
        if (threadIdx.x == 0) {
            double m = 0.0;
            for (int w = 0; w < 8; ++w) m = fmax(m, red[w]);
            atomic_max_nonneg(&defect[k], m);
        }
    }
}

// gpk[(r s), pq] = g[(r s), p, q] for p >= q < ld; pq in [npair, ldp) zero.  One CTA per (r,s) row.
__global__ void __launch_bounds__(256) pack_pairs_kernel(const double *__restrict__ g, double *__restrict__ gpk,
                                                         int ld, int64_t ldp) {
    const int64_t row = blockIdx.x;
    const double *src = g + row * (int64_t)ld * ld;
    double *dst = gpk + row * ldp;
    const int npair = (int)tri_count(ld);
    for (int pq = threadIdx.x; pq < ldp; pq += blockDim.x) {
        double v = 0.0;
        if (pq < npair) {
            int p, q;
            tri_decode(pq, p, q);
            v = src[(int64_t)p * ld + q];
        }
        dst[pq] = v;
    }
}

// g8[RS][PQ] = g[r, s, p, q] for r >= s, p >= q (both pairs packed: the 8-fold symmetry class representatives);
// PQ in [npair, ldp) zero.  One CTA per RS row.
__global__ void __launch_bounds__(256) pack_8fold_kernel(const double *__restrict__ g, double *__restrict__ g8,
                                                         int ld, int64_t ldp) {
    int r, s;
    tri_decode((int)blockIdx.x, r, s);
    const double *src = g + ((int64_t)r * ld + s) * (int64_t)ld * ld;
    double *dst = g8 + (int64_t)blockIdx.x * ldp;
    const int npair = (int)tri_count(ld);
    for (int pq = threadIdx.x; pq < ldp; pq += blockDim.x) {
        double v = 0.0;
        if (pq < npair) {
            int p, q;
            tri_decode(pq, p, q);
            v = src[(int64_t)p * ld + q];
        }
        dst[pq] = v;
    }
}

// dst[b][row][mn] = src[b][srow][m*nIp + n], m >= n, mn = m(m+1)/2 + n (zero for mn >= npI);
// srow = row (identity) or, with tri_rows, row = (p,q) of ld x ld and srow = tri(max,min).
__global__ void __launch_bounds__(128) pack_class_pairs_kernel(const double *__restrict__ src,
                                                               double *__restrict__ dst, int ld, int nIp,
                                                               int npIp, int tri_rows, int64_t src_stride,
                                                               int64_t dst_stride) {
    const int64_t row = blockIdx.x;
    const int b = blockIdx.y;
    int64_t srow = row;
    if (tri_rows) {
        const int p = (int)(row / ld), q = (int)(row % ld);
        const int hi = p > q ? p : q, lo = p > q ? q : p;
        srow = tri_count(hi) + lo;
    }
    const double *s = src + b * src_stride + srow * (int64_t)nIp * nIp;
    double *d = dst + b * dst_stride + row * (int64_t)npIp;
    const int npI = (int)tri_count(nIp);
    for (int mn = threadIdx.x; mn < npIp; mn += blockDim.x) {
        double v = 0.0;
        if (mn < npI) {
            int m, n;
            tri_decode(mn, m, n);
            v = s[m * nIp + n];
        }
        d[mn] = v;
    }
}

// cls J rows: J[m,n,:,:] = J[n,m,:,:] = Jp[mn,:,:];  K rows: K[m,n,:,:] = Kp[mn,:,:], K[n,m,:,:] = Kp[mn,:,:]^T.
// grid (ld/32, ld/32, npI * batch); 32x32 tiles (the transposed copy goes through padded smem).
__global__ void __launch_bounds__(256) expand_class_kernel(const double *__restrict__ Jp,
                                                           const double *__restrict__ Kp, double *__restrict__ cls,
                                                           int ld, int nIp, int npI, int64_t pk_stride,
                                                           int64_t cls_stride) {
    __shared__ double tile[32][33];
    const int mn = blockIdx.z % npI, b = blockIdx.z / npI;
    int m, n;
    tri_decode(mn, m, n);
    const int64_t ld2 = (int64_t)ld * ld;
    const double *jp = Jp + b * pk_stride + (int64_t)mn * ld2;
    const double *kp = Kp + b * pk_stride + (int64_t)mn * ld2;
    double *Kc = cls + b * cls_stride;
    double *Jc = Kc + (int64_t)nIp * nIp * ld2;
    const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int64_t row_mn = (int64_t)m * nIp + n, row_nm = (int64_t)n * nIp + m;
    for (int j = ty; j < 32; j += 8) {
        const int r = r0 + j, c = c0 + tx;
        if (r < ld && c < ld) {
            const double vj = jp[(int64_t)r * ld + c], vk = kp[(int64_t)r * ld + c];
            Jc[row_mn * ld2 + (int64_t)r * ld + c] = vj;
            Kc[row_mn * ld2 + (int64_t)r * ld + c] = vk;
            if (m != n) Jc[row_nm * ld2 + (int64_t)r * ld + c] = vj;
            tile[j][tx] = vk;
        }
    }
    if (m == n) return;
    __syncthreads();
    for (int j = ty; j < 32; j += 8) {
        const int c = c0 + j, r = r0 + tx;          // element (r, c) of Kp -> (c, r) of K[n,m]
        if (r < ld && c < ld) Kc[row_nm * ld2 + (int64_t)c * ld + r] = tile[tx][j];
    }
}

// Ccat[j][k][h * nIp + n] = C[2 j + h][k][n], n < nIp: the class columns of two evaluations side by side
__global__ void concat_class_columns_kernel(const double *__restrict__ C, int64_t strideC, int ld, int nIp,
                                            double *__restrict__ Ccat) {
    const int k = blockIdx.x, j = blockIdx.y;
    for (int c = threadIdx.x; c < 2 * nIp; c += blockDim.x) {
        const int h = c / nIp, n = c - h * nIp;
        Ccat[((int64_t)j * ld + k) * (2 * nIp) + c] = C[(int64_t)(2 * j + h) * strideC + (int64_t)k * ld + n];
    }
}

}  // namespace

int64_t pair_ld(int ld) {                       // packed pair count rounded up to even (TMA strides)
    const int64_t n = tri_count(ld);
    return n + (n & 1);
}

int eri_symmetry_defect(const double *g, int ld, double *defect3, cudaStream_t stream) {
    OO_REQUIRE(g && defect3 && ld > 0);
    OO_CUDA_CHECK(cudaMemsetAsync(defect3, 0, 3 * sizeof(double), stream));
    const int64_t t = ceil_div((int64_t)ld * ld, 32);
    if (t > 65535) return OO_ERR_UNSUPPORTED;
    eri_defect_kernel<<<dim3((unsigned)t, (unsigned)t), 256, 0, stream>>>(g, ld, defect3);
    OO_LAUNCH_CHECK();
    return OO_OK;
}

int pack_eri_pairs(const double *g, double *gpk, int ld, cudaStream_t stream) {
    OO_REQUIRE(g && gpk && ld > 0 && (ld % 2) == 0);
    const int64_t rows = (int64_t)ld * ld;
    if (rows > 0x7fffffffll) return OO_ERR_UNSUPPORTED;
    pack_pairs_kernel<<<(unsigned)rows, 256, 0, stream>>>(g, gpk, ld, pair_ld(ld));
    OO_LAUNCH_CHECK();
    return OO_OK;
}

int pack_eri_8fold(const double *g, double *g8, int ld, cudaStream_t stream) {
    OO_REQUIRE(g && g8 && ld > 0 && (ld % 2) == 0);
    const int64_t rows = tri_count(ld);
    if (rows > 0x7fffffffll) return OO_ERR_UNSUPPORTED;
    pack_8fold_kernel<<<(unsigned)rows, 256, 0, stream>>>(g, g8, ld, pair_ld(ld));
    OO_LAUNCH_CHECK();
    return OO_OK;
}

size_t class_transform_sym_ws_bytes(int ld, int nIp, int batch) {
    const size_t ld2 = (size_t)ld * ld, ldp = (size_t)pair_ld(ld), npIp = (size_t)pair_ld(nIp);
    const size_t t1 = (size_t)ld * ldp * nIp, t1t = ld2 * ld * nIp;
    const size_t x = ld2 * nIp * nIp;                 // >= ldp * nIp^2 (Q2 output) as well
    const size_t xp = ld2 * npIp;
    return (size_t)batch * (t1 + t1t + x + 4 * xp) * sizeof(double);
}

// slab_ld > 0: gpk is a SLAB of the 8-fold packed tensor, g8[RS][pq_lo + j], j < pq_cnt, row pitch slab_ld (sharded
// evaluation).  Quarter 1 and the Coulomb quarter 2 then run over the slab's pairs only; every later step is linear
// in the quarter-1 result, so the class buffer this call produces is this slab's ADDITIVE share of the complete
// one (the caller sums the shares of all ranks).  The pair-unpacked quarter-1 copy and the quarter-2 output are
// zeroed first: pairs outside the slab contribute nothing.
int class_transform_sym(const double *gpk, int64_t strideG, const double *C, int64_t strideC, int N, int ld,
                        int nIp, int batch, double *cls, void *ws, size_t ws_bytes, unsigned flags,
                        cudaStream_t stream, int64_t slab_ld = 0, int64_t pq_lo = 0, int64_t pq_cnt = 0) {
    const bool g_class_unfused_pack = (flags & OO_FLAG_CLASS_UNFUSED_PACK) != 0;   // separate pack / expand passes
    const bool slab = slab_ld > 0;
    const bool direct = (flags & OO_FLAG_CLASS_DIRECT_STORES) != 0;       // no staged epilogues (A/B tests)
    if (slab && (!(flags & OO_FLAG_CLASS_ERI_8FOLD) || g_class_unfused_pack || ((flags >> 16) & 0x7fu)))
        return OO_ERR_INVALID_ARG;
    OO_REQUIRE(gpk && C && cls && ws);
    OO_REQUIRE(N > 0 && ld >= N && (ld % 2) == 0 && nIp > 0 && (nIp % 2) == 0 && nIp <= ld && batch > 0);
    if (ws_bytes < class_transform_sym_ws_bytes(ld, nIp, batch)) return OO_ERR_WORKSPACE;
    if (ld > 65535) return OO_ERR_UNSUPPORTED;
    const int64_t ld2 = (int64_t)ld * ld, ldp = pair_ld(ld), nI2 = (int64_t)nIp * nIp;
    const int64_t npI = tri_count(nIp), npIp = pair_ld(nIp);
    const int64_t sT1 = (int64_t)ld * ldp * nIp, sT1t = ld2 * ld * nIp, sX = ld2 * nI2, sXp = ld2 * npIp;
    const int64_t sCls = (2 * nI2 + 1) * ld2;
    if (npI * batch > 65535) return OO_ERR_UNSUPPORTED;
    double *T1 = reinterpret_cast<double *>(ws);
    double *T1t = T1 + (int64_t)batch * sT1;
    double *X = T1t + (int64_t)batch * sT1t;
    double *P0 = X + (int64_t)batch * sX;         // packed-class-pair buffers
    double *P1 = P0 + (int64_t)batch * sXp;
    double *Jp = P1 + (int64_t)batch * sXp;
    double *Kp = Jp + (int64_t)batch * sXp;
    double *Kout = cls, *Jout = cls + nI2 * ld2;
    int rc;
#define Q(in, sIn, out, sOut, M, Ncols)                                                                        \
    if ((rc = (direct ? dgemm_tn_direct : dgemm_tn)((in), C, (out), (M), (Ncols), ld, (M), ld, (Ncols), batch, (sIn), \
                                                    strideC, (sOut), stream)))                                     \
    return rc
    // OO_FLAG_CLASS_STAGE(k): run only the selected GEMM stages (k = 0: quarter 1; 1-3: Coulomb class; 4-6: exchange
    // class) on the intermediates a complete call left in the workspace -- per-kernel timing from the caller's side
    // quarter 2 on the triangular kernel (dgemm_tri.cu: only the class pairs n <= m are computed) unless the
    // class count is outside its range or the caller asks for the rectangular GEMM + packing epilogue
    const bool tri_q2 = dgemm_tn_tri_supported(nIp) && !(flags & OO_FLAG_CLASS_Q2_RECTANGULAR);
    const unsigned stage_mask = (flags >> 16) & 0x7fu;
    auto run = [&](int k) { return stage_mask == 0 || ((stage_mask >> k) & 1u); };
    // Evaluations that share the integrals go through quarter 1 in PAIRS where a tile configuration fits the 2 nIp
    // columns [C_2j | C_2j+1] (up to 48: e.g. 2 x 24 at 114 orbitals CAS(6,6); 81 .. 96: 2 x 44 at N=256, which
    // fill 88 of 88 computed columns where one evaluation fills 44 of 48): one GEMM reads the packed integrals once
    // for both; its output rows are 2 nIp wide, and the triangular quarter-2 launch reads each evaluation's half of
    // them.  Everything after quarter 2 is unchanged.  An odd last evaluation goes through on its own.
    const bool pair_cols = 2 * nIp <= 48 || (2 * nIp > 80 && 2 * nIp <= 96);
    const bool pair_q1 = (flags & OO_FLAG_CLASS_ERI_8FOLD) && !(flags & OO_FLAG_CLASS_Q1_UNPAIRED) && !slab && tri_q2 &&
                         !g_class_unfused_pack && batch >= 2 && strideG == 0 && strideC != 0 && pair_cols;
    const int npairs = pair_q1 ? batch / 2 : 0;
    const int64_t first_single = 2 * (int64_t)npairs;
    const int nsingle = batch - 2 * npairs;
    if (stage_mask && g_class_unfused_pack) return OO_ERR_INVALID_ARG;
    // Q1: rows (s, pq); the epilogue also writes T1t[q,p,s,m] and T1t[p,q,s,m]
    if (!run(0)) {
    } else if (flags & OO_FLAG_CLASS_ERI_8FOLD) {
        // gpk is the 8-fold packed tensor g8[RS][PQ]: the quarter-1 producer gathers its k-rows from it
        if (slab) {
            OO_CUDA_CHECK(cudaMemsetAsync(T1t, 0, (size_t)batch * sT1t * sizeof(double), stream));
            OO_CUDA_CHECK(cudaMemsetAsync(P0, 0, (size_t)batch * sXp * sizeof(double), stream));
        }
        if (npairs) {
            // two evaluations per GEMM: B operand [C_2j | C_2j+1], quarter-1 rows 2 nIp wide
            concat_class_columns_kernel<<<dim3((unsigned)ld, (unsigned)npairs), 64, 0, stream>>>(C, strideC, ld, nIp, X);
            OO_LAUNCH_CHECK();
            if ((rc = dgemm_tn_q1_packed8(gpk, ldp, 0, (int)ldp, X, T1, T1t, ld, (int)ldp, 2 * nIp, ld, 2 * nIp, 2 * nIp,
                                          npairs, 0, (int64_t)ld * 2 * nIp, 2 * sT1, 2 * sT1t, stream, direct)))
                return rc;
        }
        if (nsingle &&
            (rc = dgemm_tn_q1_packed8(gpk + first_single * strideG, slab ? slab_ld : ldp, slab ? (int)pq_lo : 0,
                                      slab ? (int)pq_cnt : (int)ldp, C + first_single * strideC, T1 + first_single * sT1,
                                      T1t + first_single * sT1t, ld, (int)ldp, nIp, ld, ld, nIp, nsingle, strideG, strideC,
                                      sT1, sT1t, stream, direct)))
            return rc;
    } else if ((rc = dgemm_tn_pair_unpack(gpk, C, T1, T1t, ld, ld, (int)ldp, nIp, ld, (int64_t)ld * ldp, ld, nIp,
                                          batch, strideG, strideC, sT1, sT1t, stream))) {
        return rc;
    }
    // ---- J: quarter 2 writes the class pairs m >= n straight into Xf[p,q,mn] (both orders of the AO pair)
    if (!run(1)) {
    } else if (g_class_unfused_pack) {
        const dim3 pgrid((unsigned)ld2, (unsigned)batch);
        Q(T1, sT1, X, sX, ldp * nIp, nIp);                               // X[pq,m,n]
        pack_class_pairs_kernel<<<pgrid, 128, 0, stream>>>(X, P0, ld, nIp, (int)npIp, 1, sX, sXp);
        OO_LAUNCH_CHECK();
    } else if (tri_q2) {
        // (a slab: only its pairs -- groups pq_lo .. pq_lo + pq_cnt -- hold anything; the rest of P0 stays zero)
        const int64_t g_lo = slab ? pq_lo : 0, g_cnt = slab ? pq_cnt : ldp;
        if (npairs &&                                      // evaluation 2 j + h: columns h nIp .. of the paired rows
            (rc = dgemm_tn_tri_class_pack(T1, C, P0, 1, nIp, ld, ldp, npIp, ld, ldp * 2 * nIp, ld, npairs, 2 * sT1,
                                          strideC, sXp, stream, 0, 2 * nIp, 2)))
            return rc;
        if (nsingle &&
            (rc = dgemm_tn_tri_class_pack(T1 + first_single * sT1 + g_lo * nIp, C + first_single * strideC,
                                          P0 + first_single * sXp, 1, nIp, ld, g_cnt, npIp, ld, ldp * nIp, ld, nsingle,
                                          sT1, strideC, sXp, stream, g_lo)))
            return rc;
    } else {
        const int64_t g_lo = slab ? pq_lo : 0, g_cnt = slab ? pq_cnt : ldp;
        if ((rc = dgemm_tn_class_pack(T1 + g_lo * nIp, C, P0, 1, nIp, ld, g_cnt, npIp, ld, ldp * nIp, ld, batch, sT1,
                                      strideC, sXp, stream, g_lo)))
            return rc;
    }
    if (run(2)) Q(P0, sXp, P1, sXp, ld * npIp, ld);                      // X'[q,mn,a]
    if (!run(3)) {
    } else if (g_class_unfused_pack) {
        Q(P1, sXp, Jp, sXp, npIp * ld, ld);                              // Jp[mn,a,b]
    } else if ((rc = dgemm_tn_class_expand(P1, C, Jout, 0, nIp, ld, npIp, ld, npIp * ld, ld, ld, batch, sXp,
                                           strideC, sCls, stream, direct))) {    // J[m,n,a,b] = J[n,m,a,b]
        return rc;
    }
    // ---- K: X2[p,s,m,n] = sum_q T1t[q,(p s m)] C[q,n], kept as X2p[p,s,mn]
    if (!run(4)) {
    } else if (g_class_unfused_pack) {
        const dim3 pgrid((unsigned)ld2, (unsigned)batch);
        Q(T1t, sT1t, X, sX, ld2 * nIp, nIp);
        pack_class_pairs_kernel<<<pgrid, 128, 0, stream>>>(X, P0, ld, nIp, (int)npIp, 0, sX, sXp);
        OO_LAUNCH_CHECK();
    } else if (tri_q2) {
        if (npairs &&
            (rc = dgemm_tn_tri_class_pack(T1t, C, P0, 0, nIp, ld, ld2, npIp, ld, ld2 * 2 * nIp, ld, npairs, 2 * sT1t,
                                          strideC, sXp, stream, 0, 2 * nIp, 2)))
            return rc;
        if (nsingle &&
            (rc = dgemm_tn_tri_class_pack(T1t + first_single * sT1t, C + first_single * strideC, P0 + first_single * sXp,
                                          0, nIp, ld, ld2, npIp, ld, ld2 * nIp, ld, nsingle, sT1t, strideC, sXp, stream)))
            return rc;
    } else if ((rc = dgemm_tn_class_pack(T1t, C, P0, 0, nIp, ld, ld2, npIp, ld, ld2 * nIp, ld, batch, sT1t, strideC,
                                         sXp, stream))) {
        return rc;
    }
    if (run(5)) Q(P0, sXp, P1, sXp, ld * npIp, ld);                      // X3[s,mn,a]
    if (!run(6)) return OO_OK;
    if (g_class_unfused_pack) {
        Q(P1, sXp, Kp, sXp, npIp * ld, ld);                              // Kp[mn,a,b]
    } else {
        if ((rc = dgemm_tn_class_expand(P1, C, Kout, 1, nIp, ld, npIp, ld, npIp * ld, ld, ld, batch, sXp, strideC,
                                        sCls, stream, direct)))                  // K[m,n,a,b], K[n,m,b,a]
            return rc;
        return OO_OK;
    }
#undef Q
    const unsigned t = (unsigned)ceil_div(ld, 32);
    expand_class_kernel<<<dim3(t, t, (unsigned)(npI * batch)), 256, 0, stream>>>(Jp, Kp, cls, ld, nIp, (int)npI,
                                                                                 sXp, sCls);
    OO_LAUNCH_CHECK();
    return OO_OK;
}

}  // namespace oo

extern "C" {

int oo_transpose_f64(const double *src, double *dst, int64_t rows, int64_t cols, void *stream) {
    return oo::transpose(src, dst, rows, cols, (cudaStream_t)stream);
}

int oo_eri_symmetry_defect_f64(const double *g_ao, int ld, double *defect3, void *stream) {
    return oo::eri_symmetry_defect(g_ao, ld, defect3, (cudaStream_t)stream);
}

int64_t oo_pair_ld(int ld) { return ld > 0 ? oo::pair_ld(ld) : 0; }

int oo_pack_eri_8fold_f64(const double *g_ao, double *g_packed8, int ld, void *stream) {
    return oo::pack_eri_8fold(g_ao, g_packed8, ld, (cudaStream_t)stream);
}

int oo_pack_eri_pairs_f64(const double *g_ao, double *g_packed, int ld, void *stream) {
    return oo::pack_eri_pairs(g_ao, g_packed, ld, (cudaStream_t)stream);
}

int oo_class_transform_sym_f64(const double *g_packed, int64_t strideG, const double *C, int64_t strideC, int N,
                               int ld, int nIp, int batch, double *cls, void *ws, size_t ws_bytes,
                               unsigned flags, void *stream) {
    return oo::class_transform_sym(g_packed, strideG, C, strideC, N, ld, nIp, batch, cls, ws, ws_bytes, flags,
                                   (cudaStream_t)stream);
}

int oo_class_transform_sym_slab_f64(const double *g_packed8_slab, int64_t slab_ld, int64_t pq_lo, int64_t pq_cnt,
                                    const double *C, int64_t strideC, int N, int ld, int nIp, int batch, double *cls,
                                    void *ws, size_t ws_bytes, unsigned flags, void *stream) {
    if (slab_ld <= 0 || pq_cnt <= 0) return OO_ERR_INVALID_ARG;
    return oo::class_transform_sym(g_packed8_slab, 0, C, strideC, N, ld, nIp, batch, cls, ws, ws_bytes,
                                   flags | OO_FLAG_CLASS_ERI_8FOLD, (cudaStream_t)stream, slab_ld, pq_lo, pq_cnt);
}

int oo_class_transform_f64(const double *g_pairT, int64_t strideG, const double *C, int64_t strideC, int N,
                           int ld, int nIp, int batch, double *cls, void *ws, size_t ws_bytes, void *stream) {
    return oo::class_transform(g_pairT, strideG, C, strideC, N, ld, nIp, batch, cls, ws, ws_bytes,
                               (cudaStream_t)stream);
}
}
