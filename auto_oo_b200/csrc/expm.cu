// K1: kappa -> skew matrix -> U = expm(-K) (reference oo_energy.py:213-230, :63-87),
// plus the N x N products around it: C' = X C_oao U (:173-176, :201, :235) and
// h' = C^T h C (:44-46).
//
// expm: scaling and squaring around a degree-18 Taylor polynomial.  With A = -K / 2^s, ||A||_1 <= 0.95, the
// truncation error 0.95^19 / 19! = 3e-18 is below the unit round-off, and for skew A every term is bounded by
// ||A||^k / k! (exp(A) is orthogonal: no cancellation to lose digits to).  The polynomial is evaluated by
// Paterson-Stockmeyer in blocks of four,
//   A2 = A A, A3 = A2 A, A4 = A2 A2                                            (3 products)
//   B_j = c_4j I + c_4j+1 A + c_4j+2 A2 + c_4j+3 A3   (j = 0..3),  B_4 = c_16 I + c_17 A + c_18 A2,   c_k = 1/k!
//   R = B_4;  R <- R A4 + B_j  for j = 3, 2, 1, 0                              (4 products, B_j added in the epilogue)
//   U = R^(2^s)                                                                (s products)
// i.e. 7 + s DMMA GEMMs with no inverse, no pivoting and no host synchronisation (the first version used the
// Pade-[7/7] approximant with a Newton-Schulz inverse: 17 + s products for the same accuracy).  Bases of up to 64
// orbitals run the whole chain in ONE launch out of shared memory (expm_fused_kernel below).
#include <stdlib.h>

#include <cooperative_groups.h>

#include "common.cuh"
#include "panel.cuh"

namespace oo {

namespace {

// A[b] = scale * K(kappa[b]):  K[l,r] = +kappa_j, K[r,l] = -kappa_j
__global__ void skew_scatter_kernel(const double *__restrict__ kappa, const int32_t *__restrict__ pl,
                                    const int32_t *__restrict__ pr, int nk, int ld, double scale,
                                    double *__restrict__ A) {
    const int b = blockIdx.y;
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= nk) return;
    const double v = scale * kappa[(int64_t)b * nk + j];
    double *Ab = A + (int64_t)b * ld * ld;
    const int l = pl[j], r = pr[j];
    Ab[(int64_t)l * ld + r] = v;
    Ab[(int64_t)r * ld + l] = -v;
}

// out = c1 X1 + c2 X2 + c3 X3 + cI I   (batched ld x ld, contiguous)
__global__ void lincomb_kernel(double *__restrict__ out, double c1, const double *__restrict__ X1,
                               double c2, const double *__restrict__ X2, double c3,
                               const double *__restrict__ X3, double cI, int N, int ld, int64_t total) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        const int64_t e = i % ((int64_t)ld * ld);
        const int row = (int)(e / ld), col = (int)(e % ld);
        double v = 0.0;
        if (X1) v += c1 * X1[i];
        if (X2) v += c2 * X2[i];
        if (X3) v += c3 * X3[i];
        if (row == col && row < N) v += cI;
        out[i] = v;
    }
}

int lincomb(double *out, double c1, const double *X1, double c2, const double *X2, double c3,
            const double *X3, double cI, int N, int ld, int batch, cudaStream_t stream) {
    const int64_t total = (int64_t)batch * ld * ld;
    int blocks = (int)ceil_div(total, 256);
    if (blocks > 4 * sm_count()) blocks = 4 * sm_count();
    lincomb_kernel<<<blocks, 256, 0, stream>>>(out, c1, X1, c2, X2, c3, X3, cI, N, ld, total);
    OO_LAUNCH_CHECK();
    return OO_OK;
}

constexpr int kExpmSlots = 10;
constexpr int kTaylorDegree = 18;

// c_k = 1 / k!
__host__ __device__ inline double inv_factorial(int k) {
    double f = 1.0;
    for (int i = 2; i <= k; ++i) f *= (double)i;
    return 1.0 / f;
}

// B_j = c_4j I + c_4j+1 A + c_4j+2 A2 + c_4j+3 A3 for j = 0..4 (terms past the degree dropped), all in one pass
__global__ void taylor_blocks_kernel(const double *__restrict__ A, const double *__restrict__ A2,
                                     const double *__restrict__ A3, double *__restrict__ B, int64_t slot, int N, int ld,
                                     int64_t total) {
    double c[kTaylorDegree + 1];
#pragma unroll
    for (int k = 0; k <= kTaylorDegree; ++k) c[k] = inv_factorial(k);
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        const int64_t e = i % ((int64_t)ld * ld);
        const int row = (int)(e / ld), col = (int)(e % ld);
        const double a1 = A[i], a2 = A2[i], a3 = A3[i];
        const double eye = (row == col && row < N) ? 1.0 : 0.0;
#pragma unroll
        for (int j = 0; j < 5; ++j) {
            double v = c[4 * j] * eye + c[4 * j + 1] * a1 + c[4 * j + 2] * a2;
            if (4 * j + 3 <= kTaylorDegree) v += c[4 * j + 3] * a3;
            B[j * slot + i] = v;
        }
    }
}

// expm of A (already scaled by 2^-s), in place workspace; result in U
int expm_scaled(const double *A, int N, int ld, int batch, int squarings, double *U, double *ws,
                cudaStream_t stream) {
    const int64_t mat = (int64_t)ld * ld;
    const int64_t sl = mat * batch;
    double *A2 = ws + 0 * sl, *A3 = ws + 1 * sl, *A4 = ws + 2 * sl, *B = ws + 3 * sl;      // B_0 .. B_4: slots 3-7
    double *T0 = ws + 8 * sl, *T1 = ws + 9 * sl;
    int rc;
#define GEMM(a, b, e, beta, d)                                                                          \
    if ((rc = dgemm_small(0, 0, ld, ld, ld, 1.0, (a), ld, mat, (b), ld, mat, (beta), (e), ld, mat, 0.0, \
                          (d), ld, mat, batch, stream, N)))                                             \
    return rc
    GEMM(A, A, nullptr, 0.0, A2);
    GEMM(A2, A, nullptr, 0.0, A3);
    GEMM(A2, A2, nullptr, 0.0, A4);
    {
        int blocks = (int)ceil_div(sl, 256);
        if (blocks > 4 * sm_count()) blocks = 4 * sm_count();
        taylor_blocks_kernel<<<blocks, 256, 0, stream>>>(A, A2, A3, B, sl, N, ld, sl);
        OO_LAUNCH_CHECK();
    }
    // Horner in A4; the chain and the squarings ping-pong so that the last product lands in U
    const int products = 4 + squarings;
    double *Rc = B + 4 * sl;
    for (int i = 0; i < products; ++i) {
        double *Rn = (i == products - 1) ? U : ((i % 2 == 0) ? T0 : T1);
        if (i < 4) {
            GEMM(Rc, A4, B + (3 - i) * sl, 1.0, Rn);                    // R <- R A4 + B_(3-i)
        } else {
            GEMM(Rc, Rc, nullptr, 0.0, Rn);
        }
        Rc = Rn;
    }
#undef GEMM
    return OO_OK;
}


// ---- fused expm for ld <= 64: one CTA per matrix, everything resident in shared memory -------------
// The unfused route above costs 21 + s launches whose kernels are a few microseconds each; for the
// small bases of the reference's molecules (7 ... 43 orbitals) the whole Taylor / squaring
// chain fits six n8 x n8 shared-memory slots (n8 = N rounded up to 8; 209 KB at n8 = 64), so one launch does all of it:
// 16 warps, DMMA.8x8x4 straight from shared memory (row stride = 4 mod 16 doubles: conflict-free A and B
// fragment loads), same arithmetic in the same order as expm_scaled().
constexpr int kFusedMaxN8 = 64;
constexpr int kFusedThreads = 512;

__host__ __device__ inline int fused_row_stride(int n8) { return ((n8 + 11) / 16) * 16 + 4; }   // >= n8, = 4 mod 16

size_t fused_smem_bytes(int n8) { return (size_t)6 * n8 * fused_row_stride(n8) * sizeof(double); }

// D = alpha X Y + beta E + gamma I(rows < eyeN); D must not alias X, Y or E
// P1, P2, P3 (optional): the epilogue also adds p1 P1 + p2 P2 + p3 P3 -- a Taylor block B_j formed on the fly
template <int GR, int GC>
__device__ __forceinline__ void smem_gemm(double *__restrict__ D, const double *X, const double *Y, int n8,
                                          int LS, double alpha, const double *E, double beta, double gamma,
                                          int eyeN, const double *P1 = nullptr, double p1 = 0.0,
                                          const double *P2 = nullptr, double p2 = 0.0, const double *P3 = nullptr,
                                          double p3 = 0.0) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarp = blockDim.x >> 5;
    const int g = lane >> 2, t = lane & 3;
    const int nt = n8 >> 3;
    const int ngr = (nt + GR - 1) / GR, ngc = (nt + GC - 1) / GC;
    for (int grp = warp; grp < ngr * ngc; grp += nwarp) {
        const int r0 = (grp / ngc) * GR, c0 = (grp % ngc) * GC;
        double acc[GR][GC][2];
#pragma unroll
        for (int i = 0; i < GR; ++i)
#pragma unroll
            for (int j = 0; j < GC; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
        for (int k = 0; k < n8; k += 4) {
            double a[GR], b[GC];
#pragma unroll
            for (int i = 0; i < GR; ++i) a[i] = (r0 + i < nt) ? X[(8 * (r0 + i) + g) * LS + k + t] : 0.0;
#pragma unroll
            for (int j = 0; j < GC; ++j) b[j] = (c0 + j < nt) ? Y[(k + t) * LS + 8 * (c0 + j) + g] : 0.0;
#pragma unroll
            for (int i = 0; i < GR; ++i)
#pragma unroll
                for (int j = 0; j < GC; ++j) dmma884(acc[i][j][0], acc[i][j][1], a[i], b[j]);
        }
#pragma unroll
        for (int i = 0; i < GR; ++i) {
            if (r0 + i >= nt) continue;
            const int row = 8 * (r0 + i) + g;
#pragma unroll
            for (int j = 0; j < GC; ++j) {
                if (c0 + j >= nt) continue;
#pragma unroll
                for (int c = 0; c < 2; ++c) {
                    const int col = 8 * (c0 + j) + 2 * t + c;
                    double v = alpha * acc[i][j][c];
                    if (E) v += beta * E[row * LS + col];
                    if (P1) v += p1 * P1[row * LS + col];
                    if (P2) v += p2 * P2[row * LS + col];
                    if (P3) v += p3 * P3[row * LS + col];
                    if (row == col && row < eyeN) v += gamma;
                    D[row * LS + col] = v;
                }
            }
        }
    }
    __syncthreads();
}

// out = c1 X1 + c2 X2 + c3 X3 + cI I(rows < N)   (elementwise; out may alias an input)
__device__ __forceinline__ void smem_lincomb(double *out, double c1, const double *X1, double c2, const double *X2,
                                             double c3, const double *X3, double cI, int N, int n8, int LS) {
    for (int e = threadIdx.x; e < n8 * n8; e += blockDim.x) {
        const int row = e / n8, col = e - row * n8, o = row * LS + col;
        double v = 0.0;
        if (X1) v += c1 * X1[o];
        if (X2) v += c2 * X2[o];
        if (X3) v += c3 * X3[o];
        if (row == col && row < N) v += cI;
        out[o] = v;
    }
    __syncthreads();
}

struct FusedExpmArgs {
    const double *kappa;          // (batch, nk) packed rotation parameters, or nullptr
    const int32_t *pl, *pr;
    int nk;
    const double *Ain;            // (batch, ld, ld) dense input when kappa == nullptr
    double scale;                 // A = scale * K(kappa)   resp.   A = scale * Ain
    int N, ld, n8, squarings;    // squarings < 0: chosen on the device from ||A||_1, per matrix
    double *U;                    // (batch, ld, ld)
};

template <int GR, int GC>
__global__ void __launch_bounds__(kFusedThreads) expm_fused_kernel(const FusedExpmArgs p) {
    extern __shared__ __align__(16) double sm[];
    const int n8 = p.n8, LS = fused_row_stride(n8), N = p.N;
    const int slot = n8 * LS;
    double *S0 = sm, *S1 = sm + slot, *S2 = sm + 2 * slot, *S3 = sm + 3 * slot, *S4 = sm + 4 * slot;
    double *S5 = sm + 5 * slot;
    const int b = blockIdx.x;
    // ---- A = scale * input into S0 (zero padded to n8)
    for (int e = threadIdx.x; e < slot; e += blockDim.x) S0[e] = 0.0;
    __syncthreads();
    if (p.kappa) {
        const double *kap = p.kappa + (int64_t)b * p.nk;
        for (int j = threadIdx.x; j < p.nk; j += blockDim.x) {
            const double v = p.scale * kap[j];
            const int l = p.pl[j], r = p.pr[j];
            S0[l * LS + r] = v;
            S0[r * LS + l] = -v;
        }
    } else {
        const double *Ab = p.Ain + (int64_t)b * p.ld * p.ld;
        for (int e = threadIdx.x; e < N * N; e += blockDim.x) {
            const int row = e / N, col = e - row * N;
            S0[row * LS + col] = p.scale * Ab[(int64_t)row * p.ld + col];
        }
    }
    __syncthreads();
    int squarings = p.squarings;
    if (squarings < 0) {
        // device-side choice, per matrix: s = max(0, ceil(log2(||A||_1 / 0.95))), A <- A / 2^s (exact scaling);
        // the same rule the host applies (engine.squarings_for) without its device->host round trip
        double *colsum = S1;
        for (int col = threadIdx.x; col < n8; col += blockDim.x) {
            double acc = 0.0;
            for (int row = 0; row < n8; ++row) acc += fabs(S0[row * LS + col]);
            colsum[col] = acc;
        }
        __syncthreads();
        double norm1 = 0.0;
        for (int col = 0; col < n8; ++col) norm1 = fmax(norm1, colsum[col]);     // every thread: same order, same value
        squarings = 0;
        if (norm1 > 0.95 && norm1 < 1e300) squarings = min(64, (int)ceil(log2(norm1 / 0.95)));
        __syncthreads();
        if (squarings > 0) {
            const double sc = ldexp(1.0, -squarings);
            for (int e = threadIdx.x; e < slot; e += blockDim.x) S0[e] *= sc;
            __syncthreads();
        }
    }
    // degree-18 Taylor polynomial by Paterson-Stockmeyer (same arithmetic, same order as expm_scaled())
    double c[kTaylorDegree + 1];
#pragma unroll
    for (int k = 0; k <= kTaylorDegree; ++k) c[k] = inv_factorial(k);
    double *A = S0, *A2 = S1, *A3 = S2, *A4 = S3;
    smem_gemm<GR, GC>(A2, A, A, n8, LS, 1.0, nullptr, 0.0, 0.0, 0);
    smem_gemm<GR, GC>(A3, A2, A, n8, LS, 1.0, nullptr, 0.0, 0.0, 0);
    smem_gemm<GR, GC>(A4, A2, A2, n8, LS, 1.0, nullptr, 0.0, 0.0, 0);
    double *Rc = S4, *Rn = S5;
    smem_lincomb(Rc, c[17], A, c[18], A2, 0.0, nullptr, c[16], N, n8, LS);               // B_4
#pragma unroll
    for (int j = 3; j >= 0; --j) {                                                        // R <- R A4 + B_j
        smem_gemm<GR, GC>(Rn, Rc, A4, n8, LS, 1.0, nullptr, 0.0, c[4 * j], N, A, c[4 * j + 1], A2, c[4 * j + 2], A3,
                          c[4 * j + 3]);
        double *tmp = Rc; Rc = Rn; Rn = tmp;
    }
    for (int s = 0; s < squarings; ++s) {
        smem_gemm<GR, GC>(Rn, Rc, Rc, n8, LS, 1.0, nullptr, 0.0, 0.0, 0);
        double *tmp = Rc; Rc = Rn; Rn = tmp;
    }
    double *Ub = p.U + (int64_t)b * p.ld * p.ld;
    for (int e = threadIdx.x; e < p.ld * p.ld; e += blockDim.x) {
        const int row = e / p.ld, col = e - row * p.ld;
        Ub[e] = Rc[row * LS + col];
    }
}

bool expm_fused_enabled() {
    static const bool on = getenv("OO_OPT_EXPM_UNFUSED") == nullptr;
    return on;
}

template <int GR, int GC>
int launch_expm_fused(const FusedExpmArgs &p, int batch, cudaStream_t stream) {
    static unsigned long long configured = 0;
    const size_t smem = fused_smem_bytes(p.n8);
    if (once_per_device(configured)) {
        OO_CUDA_CHECK(cudaFuncSetAttribute(expm_fused_kernel<GR, GC>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           (int)fused_smem_bytes(kFusedMaxN8)));
    }
    expm_fused_kernel<GR, GC><<<batch, kFusedThreads, smem, stream>>>(p);
    OO_LAUNCH_CHECK();
    return OO_OK;
}

int expm_fused(FusedExpmArgs p, int batch, cudaStream_t stream) {
    p.n8 = (p.N + 7) / 8 * 8;
    const int nt = p.n8 / 8;
    if (nt <= 4) return launch_expm_fused<1, 1>(p, batch, stream);
    if (nt == 5) return launch_expm_fused<1, 2>(p, batch, stream);
    if (nt == 6) return launch_expm_fused<1, 3>(p, batch, stream);
    return launch_expm_fused<2, 2>(p, batch, stream);
}


// ---- single-launch chain for 64 < N <= 256: one cooperative kernel, a grid barrier between the products -----------
// The multi-launch route costs 1 memset + 1 scatter + 1 block kernel + 7 + s GEMM launches of 4-8 us each (and, when
// the caller has not fixed s, a host round trip to choose it).  Here the grid stays resident: every product of the
// chain is a phase whose 32 x 32 output tiles (panel GEMM of panel.cuh: both K panels staged at once, DMMA from shared
// memory) are dealt round-robin to the CTAs, the Taylor blocks B_j are formed in the epilogues from the A, A2, A3
// tiles, and grid.sync() stands where a kernel boundary was: 8 + s barriers, same arithmetic in the same order as
// expm_scaled().  s < 0: chosen on the device, max over the batch of ceil(log2(||A_b||_1 / 0.95)) -- the rule of
// engine.squarings_for, without its device->host round trip.  (The column sums of |K| are accumulated with shared-memory
// atomics, as the host rule's index_add_ is: their last bits depend on the order of the adds, which can only matter
// for a norm within round-off of 0.95 * 2^s -- either count is then equally valid.)
namespace cg = cooperative_groups;

struct ChainArgs {
    const double *kappa;          // (batch, nk) packed rotation parameters, or nullptr
    const int32_t *pl, *pr;
    int nk;
    const double *Ain;            // (batch, ld, ld) dense input when kappa == nullptr
    double sign;                  // A = sign * K(kappa) / 2^s   resp.   A = sign * Ain / 2^s
    int N, ld, batch, squarings;
    double *ws;                   // rotation_ws_bytes(ld, batch)
    double *U;                    // (batch, ld, ld)
};

struct ChainProduct {             // D = X Y (+ X2 Y2) (+ B),  B = c0 I + c1 P1 + c2 P2 (+ c3 P3);  D2 = d0 I + d1 P1 + d2 D
    const double *X, *Y;
    double *D;
    const double *P1, *P2, *P3;
    double c0, c1, c2, c3;
    double *D2;
    double d0, d1, d2;
    const double *X2, *Y2;        // second operand pair (the dual products of the Frechet chain), or nullptr
};

// acc = X[m0.., :] Y[:, n0..] of one 32 x 32 tile, staged whole (K <= PK_MAX); true for the warps that own the output
__device__ __forceinline__ bool chain_tile_mma(const double *X, const double *Y, int64_t off, int m0, int n0, int ld,
                                               int K, double *psm, double (&acc)[2][2][2]) {
    using namespace panel;
    const int K4 = (K + 3) & ~3;
    double *sA = psm, *sB = psm + TS * panel_ls(K);
    stage_panel(sA, X + off, ld, true, m0, ld, K, K4);
    stage_panel(sB, Y + off, ld, false, n0, ld, K, K4);
    asm volatile("cp.async.commit_group;" ::: "memory");
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncthreads();
    return tile_mma(sA, sB, true, false, K, K4, psm, acc);
}

__device__ __forceinline__ void chain_tile(const ChainProduct &q, int b, int m0, int n0, int N, int ld, int K,
                                           double *psm) {
    const int64_t off = (int64_t)b * ld * ld;
    double acc[2][2][2];
    const bool own = chain_tile_mma(q.X, q.Y, off, m0, n0, ld, K, psm, acc);
    if (q.X2) {
        // second staging pass into the same panels (the reduction buffer of the first aliases them)
        double acc2[2][2][2];
        __syncthreads();
        chain_tile_mma(q.X2, q.Y2, off, m0, n0, ld, K, psm, acc2);
#pragma unroll
        for (int i = 0; i < 2; ++i)
#pragma unroll
            for (int j = 0; j < 2; ++j)
#pragma unroll
                for (int c = 0; c < 2; ++c) acc[i][j][c] += acc2[i][j][c];
    }
    if (own) {
        const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
        const int g = lane >> 2, t = lane & 3;
        const int wm = ((warp & 3) >> 1) * 16, wn = (warp & 1) * 16;
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const int row = m0 + wm + i * 8 + g;
#pragma unroll
            for (int j = 0; j < 2; ++j)
#pragma unroll
                for (int c = 0; c < 2; ++c) {
                    const int col = n0 + wn + j * 8 + 2 * t + c;
                    if (row >= ld || col >= ld) continue;
                    const int64_t o = off + (int64_t)row * ld + col;
                    const double eye = (row == col && row < N) ? 1.0 : 0.0;
                    double v = acc[i][j][c];
                    if (q.P2) {
                        double bj = q.c0 * eye + q.c1 * q.P1[o] + q.c2 * q.P2[o];
                        if (q.P3) bj += q.c3 * q.P3[o];
                        v += bj;
                    }
                    q.D[o] = v;
                    if (q.D2) q.D2[o] = q.d0 * eye + q.d1 * q.P1[o] + q.d2 * v;
                }
        }
    }
    __syncthreads();                                              // the reduction buffer aliases the next tile's panels
}

__device__ __forceinline__ void chain_phase(const ChainProduct *q, int nprod, int batch, int N, int ld, int K,
                                            double *psm) {
    const int nt = (ld + panel::TS - 1) / panel::TS;
    const int items = nprod * batch * nt * nt;
    for (int it = blockIdx.x; it < items; it += gridDim.x) {
        const int tile = it % (nt * nt), rest = it / (nt * nt);
        chain_tile(q[rest % nprod], rest / nprod, (tile / nt) * panel::TS, (tile % nt) * panel::TS, N, ld, K, psm);
    }
}

// Phase 0 of the single-launch chains: the squaring count (s < 0: max over the batch of ceil(log2(||A_b||_1 / 0.95)),
// from the packed kappa or the dense Ain), ending in a grid barrier either way.  Every CTA returns the same s.
__device__ int chain_squarings(cg::grid_group &grid, const double *kappa, const int32_t *pl, const int32_t *pr, int nk,
                               const double *Ain, int N, int ld, int batch, int squarings, double *norms, double *psm) {
    const int64_t mat = (int64_t)ld * ld;
    if (squarings < 0) {
        double *colsum = psm;
        for (int b = blockIdx.x; b < batch; b += gridDim.x) {
            for (int c = threadIdx.x; c < ld; c += blockDim.x) colsum[c] = 0.0;
            __syncthreads();
            if (kappa) {
                const double *kap = kappa + (int64_t)b * nk;
                for (int j = threadIdx.x; j < nk; j += blockDim.x) {
                    const double v = fabs(kap[j]);
                    atomicAdd(&colsum[pl[j]], v);
                    atomicAdd(&colsum[pr[j]], v);
                }
            } else {
                const double *Ab = Ain + (int64_t)b * mat;
                for (int c = threadIdx.x; c < N; c += blockDim.x) {
                    double acc = 0.0;
                    for (int r = 0; r < N; ++r) acc += fabs(Ab[(int64_t)r * ld + c]);
                    colsum[c] = acc;
                }
            }
            __syncthreads();
            if (threadIdx.x < 32) {
                double m = 0.0;
                for (int c = threadIdx.x; c < ld; c += 32) m = fmax(m, colsum[c]);
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
                if (threadIdx.x == 0) norms[b] = m;
            }
            __syncthreads();
        }
        grid.sync();
        double m = 0.0;
        for (int b = threadIdx.x; b < batch; b += blockDim.x) m = fmax(m, norms[b]);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
        double *wmax = psm;                                       // one value per warp
        __syncthreads();
        if ((threadIdx.x & 31) == 0) wmax[threadIdx.x >> 5] = m;
        __syncthreads();
        double norm1 = 0.0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) norm1 = fmax(norm1, wmax[w]);
        __syncthreads();
        squarings = 0;
        if (norm1 > 0.95 && norm1 < 1e300) squarings = min(64, (int)ceil(log2(norm1 / 0.95)));
    } else {
        grid.sync();
    }
    return squarings;
}

__global__ void __launch_bounds__(panel::PTHREADS) expm_chain_kernel(const ChainArgs p) {
    extern __shared__ __align__(16) double psm[];
    cg::grid_group grid = cg::this_grid();
    const int N = p.N, ld = p.ld, batch = p.batch;
    const int64_t mat = (int64_t)ld * ld, sl = mat * batch;
    double *A2 = p.ws + 0 * sl, *A3 = p.ws + 1 * sl, *A4 = p.ws + 2 * sl, *norms = p.ws + 3 * sl;
    double *R0 = p.ws + 7 * sl, *T0 = p.ws + 8 * sl, *T1 = p.ws + 9 * sl, *A = p.ws + (int64_t)kExpmSlots * sl;
    const int64_t gtid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, gthreads = (int64_t)gridDim.x * blockDim.x;

    // ---- phase 0: A = 0 (packed input) and, when s is ours to choose, ||sign * input_b||_1 per matrix
    if (p.kappa)
        for (int64_t i = gtid; i < sl; i += gthreads) A[i] = 0.0;
    const int squarings =
        chain_squarings(grid, p.kappa, p.pl, p.pr, p.nk, p.Ain, N, ld, batch, p.squarings, norms, psm);
    // ---- phase 1: A = sign * input / 2^s
    const double scale = p.sign * ldexp(1.0, -squarings);
    if (p.kappa) {
        for (int64_t i = gtid; i < (int64_t)batch * p.nk; i += gthreads) {
            const int b = (int)(i / p.nk), j = (int)(i - (int64_t)b * p.nk);
            const double v = scale * p.kappa[i];
            double *Ab = A + (int64_t)b * mat;
            const int l = p.pl[j], r = p.pr[j];
            Ab[(int64_t)l * ld + r] = v;
            Ab[(int64_t)r * ld + l] = -v;
        }
    } else {
        for (int64_t i = gtid; i < sl; i += gthreads) {
            const int64_t e = i % mat;
            const int row = (int)(e / ld), col = (int)(e % ld);
            A[i] = (row < N && col < N) ? scale * p.Ain[i] : 0.0;
        }
    }
    grid.sync();

    double c[kTaylorDegree + 1];
#pragma unroll
    for (int k = 0; k <= kTaylorDegree; ++k) c[k] = inv_factorial(k);
    const int K = ld;
    ChainProduct q[2];
    // A2 = A A, and R0 = B_4 = c16 I + c17 A + c18 A2 from the same tile
    q[0] = ChainProduct{A, A, A2, A, nullptr, nullptr, 0.0, 0.0, 0.0, 0.0, R0, c[16], c[17], c[18]};
    chain_phase(q, 1, batch, N, ld, K, psm);
    grid.sync();
    // A3 = A2 A and A4 = A2 A2 in one phase
    q[0] = ChainProduct{A2, A, A3, nullptr, nullptr, nullptr, 0.0, 0.0, 0.0, 0.0, nullptr, 0.0, 0.0, 0.0};
    q[1] = ChainProduct{A2, A2, A4, nullptr, nullptr, nullptr, 0.0, 0.0, 0.0, 0.0, nullptr, 0.0, 0.0, 0.0};
    chain_phase(q, 2, batch, N, ld, K, psm);
    grid.sync();
    // Horner in A4, then the squarings; the products ping-pong so that the last one lands in U
    const int products = 4 + squarings;
    const double *Rc = R0;
    for (int i = 0; i < products; ++i) {
        double *Rn = (i == products - 1) ? p.U : ((i % 2 == 0) ? T0 : T1);
        if (i < 4) {
            const int j = 3 - i;                                  // R <- R A4 + B_j
            q[0] = ChainProduct{Rc, A4, Rn, A, A2, A3, c[4 * j], c[4 * j + 1], c[4 * j + 2], c[4 * j + 3],
                                nullptr, 0.0, 0.0, 0.0};
        } else {
            q[0] = ChainProduct{Rc, Rc, Rn, nullptr, nullptr, nullptr, 0.0, 0.0, 0.0, 0.0, nullptr, 0.0, 0.0, 0.0};
        }
        chain_phase(q, 1, batch, N, ld, K, psm);
        if (i + 1 < products) grid.sync();
        Rc = Rn;
    }
}

constexpr int kChainMaxN = panel::PK_MAX;

bool expm_chain_enabled() {
    static const bool on = getenv("OO_OPT_EXPM_UNFUSED") == nullptr && getenv("OO_OPT_EXPM_MULTI_LAUNCH") == nullptr;
    return on;
}

// The chain applies when the panel GEMM does (even ld <= 256, 16-byte aligned slots) and the device can hold a
// cooperative grid; *launched = false leaves the work to the multi-launch route.
int expm_chain(const ChainArgs &p, cudaStream_t stream, bool *launched) {
    *launched = false;
    if (!expm_chain_enabled() || p.ld > kChainMaxN || p.ld < 8 || (p.ld & 1)) return OO_OK;
    if ((reinterpret_cast<uintptr_t>(p.ws) | reinterpret_cast<uintptr_t>(p.U)) & 15) return OO_OK;
    static unsigned long long configured = 0;
    static int coop[64] = {};
    int dev = 0;
    OO_CUDA_CHECK(cudaGetDevice(&dev));
    if (once_per_device(configured)) {
        OO_CUDA_CHECK(cudaFuncSetAttribute(expm_chain_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           (int)panel::smem_bytes(kChainMaxN, 0, 0)));
        int v = 0;
        OO_CUDA_CHECK(cudaDeviceGetAttribute(&v, cudaDevAttrCooperativeLaunch, dev));
        if (dev < 64) coop[dev] = v;
    }
    if (dev >= 64 || !coop[dev]) return OO_OK;
    size_t smem = panel::smem_bytes(p.ld, 0, 0);
    if (smem < (size_t)p.ld * sizeof(double)) smem = (size_t)p.ld * sizeof(double);       // column sums of phase 0
    int per_sm = 0;
    OO_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, expm_chain_kernel, panel::PTHREADS, smem));
    if (per_sm < 1) return OO_OK;
    const int nt = (p.ld + panel::TS - 1) / panel::TS;
    int64_t grid = (int64_t)2 * p.batch * nt * nt;                 // the widest phase: A3 and A4
    if (grid > (int64_t)per_sm * sm_count()) grid = (int64_t)per_sm * sm_count();
    void *args[] = {const_cast<ChainArgs *>(&p)};
    OO_CUDA_CHECK(cudaLaunchCooperativeKernel((const void *)expm_chain_kernel, dim3((unsigned)grid),
                                              dim3(panel::PTHREADS), args, smem, stream));
    OO_LAUNCH_CHECK();
    *launched = true;
    return OO_OK;
}


// ---- adjoint of the rotation: kappa_bar from L(K, Ubar), the Frechet derivative of exp at K -----------------------
// For U = exp(-K) and a cotangent Ubar, Kbar = -L(-K)^*(Ubar) = -L(K, Ubar) (the adjoint of L(-K, .) is L(-K^T, .) and
// K is skew), and kappa_bar_j = Kbar[l_j,r_j] - Kbar[r_j,l_j].  L(K, E) is carried through the same scaling-and-squaring
// chain as the rotation as a dual matrix next to every product (Al-Mohy & Higham 2009): with A = K / 2^s, E_1 = E / 2^s,
//   E2 = E_1 A + A E_1,  E3 = E2 A + A2 E_1,  E4 = E2 A2 + A2 E2,  dB_j = c_4j+1 E_1 + c_4j+2 E2 + c_4j+3 E3,
//   Horner: (R, L) <- (R A4 + B_j, L A4 + R E4 + dB_j),   squarings: (R, L) <- (R R, R L + L R).
// Every dual product is two GEMMs summed into one tile.  Workspace slots (ld^2 x batch each):
//   A A2 A3 A4 | E1 E2 E3 E4 | R0 R1 | L0 L1 | T Bt (multi-launch route only) | norms (batch doubles)
constexpr int kVjpSlots = 14;

// out = scale * X on the N x N block, 0 on the padding (the caller's padding is not read into the chain)
__global__ void scaled_block_kernel(double *__restrict__ out, const double *__restrict__ X, double scale, int N, int ld,
                                    int64_t total) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        const int64_t e = i % ((int64_t)ld * ld);
        const int row = (int)(e / ld), col = (int)(e % ld);
        out[i] = (row < N && col < N) ? scale * X[i] : 0.0;
    }
}

// kappa_bar[b][j] = -(L_b[l_j,r_j] - L_b[r_j,l_j])
__device__ __forceinline__ void skew_gather(const double *L, const int32_t *pl, const int32_t *pr, int nk, int ld,
                                            int64_t i, double *kbar) {
    const int b = (int)(i / nk), j = (int)(i - (int64_t)b * nk);
    const double *Lb = L + (int64_t)b * ld * ld;
    const int l = pl[j], r = pr[j];
    kbar[i] = -(Lb[(int64_t)l * ld + r] - Lb[(int64_t)r * ld + l]);
}

__global__ void skew_gather_kernel(const double *__restrict__ L, const int32_t *__restrict__ pl,
                                   const int32_t *__restrict__ pr, int nk, int ld, int64_t total,
                                   double *__restrict__ kbar) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < total) skew_gather(L, pl, pr, nk, ld, i, kbar);
}

struct VjpArgs {
    const double *kappa;          // (batch, nk)
    const int32_t *pl, *pr;
    int nk;
    const double *Ubar;           // (batch, ld, ld)
    int N, ld, batch, squarings;  // squarings < 0: chosen on the device (max over the batch), as in expm_chain_kernel
    double *ws;                   // rotation_vjp_ws_bytes(ld, batch)
    double *kbar;                 // (batch, nk)
};

// One cooperative launch for 8 <= ld <= 256: the phases of expm_chain_kernel with the dual products beside the
// primal ones (2, 4, then 2 per Horner step and squaring), a grid barrier between phases, the gather at the end.
__global__ void __launch_bounds__(panel::PTHREADS) expm_frechet_chain_kernel(const VjpArgs p) {
    extern __shared__ __align__(16) double psm[];
    cg::grid_group grid = cg::this_grid();
    const int N = p.N, ld = p.ld, batch = p.batch;
    const int64_t mat = (int64_t)ld * ld, sl = mat * batch;
    double *A = p.ws, *A2 = p.ws + sl, *A3 = p.ws + 2 * sl, *A4 = p.ws + 3 * sl;
    double *E1 = p.ws + 4 * sl, *E2 = p.ws + 5 * sl, *E3 = p.ws + 6 * sl, *E4 = p.ws + 7 * sl;
    double *Rs[2] = {p.ws + 8 * sl, p.ws + 9 * sl}, *Ls[2] = {p.ws + 10 * sl, p.ws + 11 * sl};
    double *norms = p.ws + (int64_t)kVjpSlots * sl;
    const int64_t gtid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, gthreads = (int64_t)gridDim.x * blockDim.x;

    // ---- phase 0: A = 0, s;  phase 1: A = K / 2^s, E1 = Ubar / 2^s
    for (int64_t i = gtid; i < sl; i += gthreads) A[i] = 0.0;
    const int squarings =
        chain_squarings(grid, p.kappa, p.pl, p.pr, p.nk, nullptr, N, ld, batch, p.squarings, norms, psm);
    const double scale = ldexp(1.0, -squarings);
    for (int64_t i = gtid; i < (int64_t)batch * p.nk; i += gthreads) {
        const int b = (int)(i / p.nk), j = (int)(i - (int64_t)b * p.nk);
        const double v = scale * p.kappa[i];
        double *Ab = A + (int64_t)b * mat;
        const int l = p.pl[j], r = p.pr[j];
        Ab[(int64_t)l * ld + r] = v;
        Ab[(int64_t)r * ld + l] = -v;
    }
    for (int64_t i = gtid; i < sl; i += gthreads) {
        const int64_t e = i % mat;
        const int row = (int)(e / ld), col = (int)(e % ld);
        E1[i] = (row < N && col < N) ? scale * p.Ubar[i] : 0.0;
    }
    grid.sync();

    double c[kTaylorDegree + 1];
#pragma unroll
    for (int k = 0; k <= kTaylorDegree; ++k) c[k] = inv_factorial(k);
    const int K = ld;
    ChainProduct q[4];
    // A2 = A A with R = B_4 = c16 I + c17 A + c18 A2;  E2 = E1 A + A E1 with L = c17 E1 + c18 E2
    q[0] = ChainProduct{A, A, A2, A, nullptr, nullptr, 0.0, 0.0, 0.0, 0.0, Rs[0], c[16], c[17], c[18]};
    q[1] = ChainProduct{E1, A, E2, E1, nullptr, nullptr, 0.0, 0.0, 0.0, 0.0, Ls[0], 0.0, c[17], c[18], A, E1};
    chain_phase(q, 2, batch, N, ld, K, psm);
    grid.sync();
    q[0] = ChainProduct{A2, A, A3};
    q[1] = ChainProduct{A2, A2, A4};
    q[2] = ChainProduct{E2, A, E3, nullptr, nullptr, nullptr, 0.0, 0.0, 0.0, 0.0, nullptr, 0.0, 0.0, 0.0, A2, E1};
    q[3] = ChainProduct{E2, A2, E4, nullptr, nullptr, nullptr, 0.0, 0.0, 0.0, 0.0, nullptr, 0.0, 0.0, 0.0, A2, E2};
    chain_phase(q, 4, batch, N, ld, K, psm);
    grid.sync();
    // Horner in A4, then the squarings; R is not formed in the last phase (only L is read)
    const int products = 4 + squarings;
    int cur = 0;
    for (int i = 0; i < products; ++i) {
        const double *Rc = Rs[cur], *Lc = Ls[cur];
        double *Rn = Rs[cur ^ 1], *Ln = Ls[cur ^ 1];
        if (i < 4) {
            const int j = 3 - i;
            q[0] = ChainProduct{Lc, A4, Ln, E1, E2, E3, 0.0, c[4 * j + 1], c[4 * j + 2], c[4 * j + 3],
                                nullptr, 0.0, 0.0, 0.0, Rc, E4};
            q[1] = ChainProduct{Rc, A4, Rn, A, A2, A3, c[4 * j], c[4 * j + 1], c[4 * j + 2], c[4 * j + 3]};
        } else {
            q[0] = ChainProduct{Rc, Lc, Ln, nullptr, nullptr, nullptr, 0.0, 0.0, 0.0, 0.0, nullptr, 0.0, 0.0, 0.0,
                                Lc, Rc};
            q[1] = ChainProduct{Rc, Rc, Rn};
        }
        chain_phase(q, i + 1 < products ? 2 : 1, batch, N, ld, K, psm);
        grid.sync();
        cur ^= 1;
    }
    // ---- kappa_bar from L(K, Ubar)
    for (int64_t i = gtid; i < (int64_t)batch * p.nk; i += gthreads) skew_gather(Ls[cur], p.pl, p.pr, p.nk, ld, i, p.kbar);
}

int frechet_chain(const VjpArgs &p, cudaStream_t stream, bool *launched) {
    *launched = false;
    if (p.ld > kChainMaxN || p.ld < 8 || (p.ld & 1)) return OO_OK;
    if (reinterpret_cast<uintptr_t>(p.ws) & 15) return OO_OK;
    static unsigned long long configured = 0;
    static int coop[64] = {};
    int dev = 0;
    OO_CUDA_CHECK(cudaGetDevice(&dev));
    if (once_per_device(configured)) {
        OO_CUDA_CHECK(cudaFuncSetAttribute(expm_frechet_chain_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           (int)panel::smem_bytes(kChainMaxN, 0, 0)));
        int v = 0;
        OO_CUDA_CHECK(cudaDeviceGetAttribute(&v, cudaDevAttrCooperativeLaunch, dev));
        if (dev < 64) coop[dev] = v;
    }
    if (dev >= 64 || !coop[dev]) return OO_OK;
    size_t smem = panel::smem_bytes(p.ld, 0, 0);
    if (smem < (size_t)p.ld * sizeof(double)) smem = (size_t)p.ld * sizeof(double);
    int per_sm = 0;
    OO_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, expm_frechet_chain_kernel, panel::PTHREADS,
                                                                smem));
    if (per_sm < 1) return OO_OK;
    const int nt = (p.ld + panel::TS - 1) / panel::TS;
    int64_t grid = (int64_t)4 * p.batch * nt * nt;                 // the widest phase: A3, A4, E3, E4
    if (grid > (int64_t)per_sm * sm_count()) grid = (int64_t)per_sm * sm_count();
    void *args[] = {const_cast<VjpArgs *>(&p)};
    OO_CUDA_CHECK(cudaLaunchCooperativeKernel((const void *)expm_frechet_chain_kernel, dim3((unsigned)grid),
                                              dim3(panel::PTHREADS), args, smem, stream));
    OO_LAUNCH_CHECK();
    *launched = true;
    return OO_OK;
}

// Multi-launch route (ld < 8, ld > 256): the same chain on dgemm_small, each dual product as T = X2 Y2 (+ dB) followed
// by X Y + T in the beta epilogue; needs the host's squaring count.
int frechet_multi_launch(const VjpArgs &p, cudaStream_t stream) {
    const int N = p.N, ld = p.ld, batch = p.batch, s = p.squarings;
    const int64_t mat = (int64_t)ld * ld, sl = mat * batch;
    double *w = p.ws;
    double *A = w, *A2 = w + sl, *A3 = w + 2 * sl, *A4 = w + 3 * sl;
    double *E1 = w + 4 * sl, *E2 = w + 5 * sl, *E3 = w + 6 * sl, *E4 = w + 7 * sl;
    double *Rs[2] = {w + 8 * sl, w + 9 * sl}, *Ls[2] = {w + 10 * sl, w + 11 * sl};
    double *T = w + 12 * sl, *Bt = w + 13 * sl;
    const double scale = ldexp(1.0, -s);
    int rc;
#define GEMM(a, b, e, d)                                                                                  \
    if ((rc = dgemm_small(0, 0, ld, ld, ld, 1.0, (a), ld, mat, (b), ld, mat, (e) ? 1.0 : 0.0, (e), ld, mat, \
                          0.0, (d), ld, mat, batch, stream, N)))                                        \
    return rc
#define LINCOMB(out, c1, X1, c2, X2, c3, X3, cI) \
    if ((rc = lincomb((out), (c1), (X1), (c2), (X2), (c3), (X3), (cI), N, ld, batch, stream))) return rc
    OO_CUDA_CHECK(cudaMemsetAsync(A, 0, sl * sizeof(double), stream));
    {
        dim3 grid((unsigned)ceil_div(p.nk, 256), (unsigned)batch);
        skew_scatter_kernel<<<grid, 256, 0, stream>>>(p.kappa, p.pl, p.pr, p.nk, ld, scale, A);     // A = K / 2^s
        OO_LAUNCH_CHECK();
        int blocks = (int)ceil_div(sl, 256);
        if (blocks > 4 * sm_count()) blocks = 4 * sm_count();
        scaled_block_kernel<<<blocks, 256, 0, stream>>>(E1, p.Ubar, scale, N, ld, sl);                // E1 = Ubar / 2^s
        OO_LAUNCH_CHECK();
    }
    double c[kTaylorDegree + 1];
    for (int k = 0; k <= kTaylorDegree; ++k) c[k] = inv_factorial(k);
    GEMM(A, A, nullptr, A2);
    GEMM(A2, A, nullptr, A3);
    GEMM(A2, A2, nullptr, A4);
    GEMM(A, E1, nullptr, T);
    GEMM(E1, A, T, E2);
    GEMM(A2, E1, nullptr, T);
    GEMM(E2, A, T, E3);
    GEMM(A2, E2, nullptr, T);
    GEMM(E2, A2, T, E4);
    LINCOMB(Rs[0], c[17], A, c[18], A2, 0.0, nullptr, c[16]);
    LINCOMB(Ls[0], c[17], E1, c[18], E2, 0.0, nullptr, 0.0);
    const int products = 4 + s;
    int cur = 0;
    for (int i = 0; i < products; ++i) {
        const bool last = i + 1 == products;
        double *Rc = Rs[cur], *Lc = Ls[cur], *Rn = Rs[cur ^ 1], *Ln = Ls[cur ^ 1];
        if (i < 4) {
            const int j = 3 - i;
            LINCOMB(Bt, c[4 * j + 1], E1, c[4 * j + 2], E2, c[4 * j + 3], E3, 0.0);
            GEMM(Rc, E4, Bt, T);
            GEMM(Lc, A4, T, Ln);
            if (!last) {
                LINCOMB(Bt, c[4 * j + 1], A, c[4 * j + 2], A2, c[4 * j + 3], A3, c[4 * j]);
                GEMM(Rc, A4, Bt, Rn);
            }
        } else {
            GEMM(Lc, Rc, nullptr, T);
            GEMM(Rc, Lc, T, Ln);
            if (!last) GEMM(Rc, Rc, nullptr, Rn);
        }
        cur ^= 1;
    }
#undef GEMM
#undef LINCOMB
    const int64_t total = (int64_t)batch * p.nk;
    skew_gather_kernel<<<(unsigned)ceil_div(total, 256), 256, 0, stream>>>(Ls[cur], p.pl, p.pr, p.nk, ld, total, p.kbar);
    OO_LAUNCH_CHECK();
    return OO_OK;
}

}  // namespace

size_t rotation_vjp_ws_bytes(int ld, int batch) {
    return ((size_t)kVjpSlots * batch * ld * ld + batch) * sizeof(double);
}

int kappa_rotation_vjp(const double *kappa, const int32_t *pl, const int32_t *pr, int nk, int N, int ld, int batch,
                       int squarings, const double *Ubar, double *kbar, void *ws, size_t ws_bytes,
                       cudaStream_t stream) {
    OO_REQUIRE(kappa && Ubar && kbar && ws && (nk == 0 || (pl && pr)));
    OO_REQUIRE(nk >= 0 && N > 0 && ld >= N && (ld % 2) == 0 && batch > 0 && squarings >= -1 && squarings <= 64);
    if (ws_bytes < rotation_vjp_ws_bytes(ld, batch)) return OO_ERR_WORKSPACE;
    if (batch > 65535) return OO_ERR_UNSUPPORTED;
    if (nk == 0) return OO_OK;                                     // no parameters: nothing to write
    VjpArgs p{kappa, pl, pr, nk, Ubar, N, ld, batch, squarings, reinterpret_cast<double *>(ws), kbar};
    bool launched = false;
    const int rc = frechet_chain(p, stream, &launched);
    if (rc || launched) return rc;
    if (squarings < 0) return OO_ERR_UNSUPPORTED;                  // the multi-launch route needs the host's choice
    return frechet_multi_launch(p, stream);
}

size_t rotation_ws_bytes(int ld, int batch) {
    return (size_t)(kExpmSlots + 1) * batch * ld * ld * sizeof(double);
}

int kappa_rotation(const double *kappa, const int32_t *pl, const int32_t *pr, int nk, int N, int ld,
                   int batch, int squarings, double *U, void *ws, size_t ws_bytes,
                   cudaStream_t stream) {
    OO_REQUIRE(kappa && U && ws && (nk == 0 || (pl && pr)));
    OO_REQUIRE(N > 0 && ld >= N && (ld % 2) == 0 && batch > 0 && squarings >= -1 && squarings <= 64);
    if (ws_bytes < rotation_ws_bytes(ld, batch)) return OO_ERR_WORKSPACE;
    if (batch > 65535) return OO_ERR_UNSUPPORTED;
    if (N <= kFusedMaxN8 && expm_fused_enabled()) {
        FusedExpmArgs p{kappa, pl, pr, nk, nullptr, squarings < 0 ? -1.0 : -ldexp(1.0, -squarings), N, ld, 0,
                        squarings, U};
        return expm_fused(p, batch, stream);
    }
    double *w = reinterpret_cast<double *>(ws);
    {
        ChainArgs c{kappa, pl, pr, nk, nullptr, -1.0, N, ld, batch, squarings, w, U};
        bool launched = false;
        const int rc = expm_chain(c, stream, &launched);
        if (rc || launched) return rc;
    }
    if (squarings < 0) return OO_ERR_UNSUPPORTED;      // the multi-launch route needs the host's choice
    const int64_t sl = (int64_t)batch * ld * ld;
    double *A = w + (int64_t)kExpmSlots * sl;
    OO_CUDA_CHECK(cudaMemsetAsync(A, 0, sl * sizeof(double), stream));
    if (nk > 0) {
        dim3 grid((unsigned)ceil_div(nk, 256), (unsigned)batch);
        // A = -K / 2^s
        skew_scatter_kernel<<<grid, 256, 0, stream>>>(kappa, pl, pr, nk, ld, -ldexp(1.0, -squarings), A);
        OO_LAUNCH_CHECK();
    }
    return expm_scaled(A, N, ld, batch, squarings, U, w, stream);
}

int expm_general(const double *Ain, double sign, int N, int ld, int batch, int squarings, double *U,
                 void *ws, size_t ws_bytes, cudaStream_t stream) {
    OO_REQUIRE(Ain && U && ws);
    OO_REQUIRE(N > 0 && ld >= N && (ld % 2) == 0 && batch > 0 && squarings >= 0 && squarings <= 64);
    if (ws_bytes < rotation_ws_bytes(ld, batch)) return OO_ERR_WORKSPACE;
    if (N <= kFusedMaxN8 && batch <= 65535 && expm_fused_enabled()) {
        FusedExpmArgs p{nullptr, nullptr, nullptr, 0, Ain, sign * ldexp(1.0, -squarings), N, ld, 0, squarings, U};
        return expm_fused(p, batch, stream);
    }
    double *w = reinterpret_cast<double *>(ws);
    {
        ChainArgs c{nullptr, nullptr, nullptr, 0, Ain, sign, N, ld, batch, squarings, w, U};
        bool launched = false;
        const int rc = expm_chain(c, stream, &launched);
        if (rc || launched) return rc;
    }
    const int64_t sl = (int64_t)batch * ld * ld;
    double *A = w + (int64_t)kExpmSlots * sl;
    int rc = lincomb(A, sign * ldexp(1.0, -squarings), Ain, 0.0, nullptr, 0.0, nullptr, 0.0, N, ld,
                     batch, stream);
    if (rc) return rc;
    return expm_scaled(A, N, ld, batch, squarings, U, w, stream);
}

size_t int1e_ws_bytes(int ld, int batch) { return (size_t)batch * ld * ld * sizeof(double); }

int mo_coeff(const double *X, int64_t strideX, const double *Coao, int64_t strideCoao, const double *U,
             int64_t strideU, int N, int ld, int batch, double *Cout, void *ws, size_t ws_bytes,
             cudaStream_t stream) {
    OO_REQUIRE(X && Coao && Cout);
    OO_REQUIRE(N > 0 && ld >= N && batch > 0);
    const int64_t mat = (int64_t)ld * ld;
    if (!U)
        return dgemm_small(0, 0, ld, ld, ld, 1.0, X, ld, strideX, Coao, ld, strideCoao, 0.0, nullptr, ld, 0, 0.0,
                           Cout, ld, mat, batch, stream, 0);
    OO_REQUIRE(ws);
    if (ws_bytes < int1e_ws_bytes(ld, batch)) return OO_ERR_WORKSPACE;
    double *T = reinterpret_cast<double *>(ws);
    int rc = dgemm_small(0, 0, ld, ld, ld, 1.0, Coao, ld, strideCoao, U, ld, strideU, 0.0, nullptr, ld, 0,
                         0.0, T, ld, mat, batch, stream, 0);
    if (rc) return rc;
    return dgemm_small(0, 0, ld, ld, ld, 1.0, X, ld, strideX, T, ld, mat, 0.0, nullptr, ld, 0, 0.0, Cout, ld,
                       mat, batch, stream, 0);
}

int int1e_transform(const double *h, int64_t stride_h, const double *C, int64_t strideC, int N, int ld,
                    int batch, double *hmo, void *ws, size_t ws_bytes, cudaStream_t stream) {
    OO_REQUIRE(h && C && hmo && ws);
    OO_REQUIRE(N > 0 && ld >= N && batch > 0);
    if (ws_bytes < int1e_ws_bytes(ld, batch)) return OO_ERR_WORKSPACE;
    const int64_t mat = (int64_t)ld * ld;
    double *T = reinterpret_cast<double *>(ws);
    // T = h C ; h' = C^T T
    int rc = dgemm_small(0, 0, ld, ld, ld, 1.0, h, ld, stride_h, C, ld, strideC, 0.0, nullptr, ld, 0, 0.0, T, ld,
                         mat, batch, stream, 0);
    if (rc) return rc;
    return dgemm_small(1, 0, ld, ld, ld, 1.0, C, ld, strideC, T, ld, mat, 0.0, nullptr, ld, 0, 0.0, hmo,
                       ld, mat, batch, stream, 0);
}

}  // namespace oo

extern "C" {

int oo_expm_device_squarings_max_n(void) {
    if (oo::expm_chain_enabled()) return oo::kChainMaxN;      // single-launch chain (cooperative grid)
    return oo::expm_fused_enabled() ? oo::kFusedMaxN8 : 0;
}

int oo_kappa_rotation_f64(const double *kappa, const int32_t *pair_l, const int32_t *pair_r, int nk,
                          int N, int ld, int batch, int squarings, double *U, void *ws,
                          size_t ws_bytes, void *stream) {
    return oo::kappa_rotation(kappa, pair_l, pair_r, nk, N, ld, batch, squarings, U, ws, ws_bytes,
                              (cudaStream_t)stream);
}

int oo_kappa_rotation_vjp_f64(const double *kappa, const int32_t *pair_l, const int32_t *pair_r, int nk, int N,
                              int ld, int batch, int squarings, const double *Ubar, double *kappa_bar, void *ws,
                              size_t ws_bytes, void *stream) {
    return oo::kappa_rotation_vjp(kappa, pair_l, pair_r, nk, N, ld, batch, squarings, Ubar, kappa_bar, ws, ws_bytes,
                                  (cudaStream_t)stream);
}

int oo_expm_f64(const double *A, double sign, int N, int ld, int batch, int squarings, double *U,
                void *ws, size_t ws_bytes, void *stream) {
    return oo::expm_general(A, sign, N, ld, batch, squarings, U, ws, ws_bytes, (cudaStream_t)stream);
}

int oo_mo_coeff_f64(const double *X, int64_t strideX, const double *Coao, int64_t strideCoao, const double *U,
                    int64_t strideU, int N, int ld, int batch, double *Cout, void *ws, size_t ws_bytes,
                    void *stream) {
    return oo::mo_coeff(X, strideX, Coao, strideCoao, U, strideU, N, ld, batch, Cout, ws, ws_bytes,
                        (cudaStream_t)stream);
}

int oo_int1e_transform_f64(const double *h_ao, int64_t stride_h, const double *C, int64_t strideC, int N,
                           int ld, int batch, double *h_mo, void *ws, size_t ws_bytes, void *stream) {
    return oo::int1e_transform(h_ao, stride_h, C, strideC, N, ld, batch, h_mo, ws, ws_bytes,
                               (cudaStream_t)stream);
}
}
