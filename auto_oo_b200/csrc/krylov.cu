// Krylov-subspace arithmetic between Hessian-vector products: the lowest orbital-Hessian eigenpair by Davidson-Liu
// and the shifted Newton solve by deflated preconditioned CG (auto_oo_b200/krylov.py), without forming H.
//
//  subspace_eigh_kernel    one CTA per k x k symmetric matrix (k <= 64): cyclic Jacobi in shared memory, the
//                          k/2 disjoint rotations of a round-robin round applied together; ascending eigenvalues
//  dav_project_kernel      out[j] = V_j . u, one CTA per basis vector (the new row/column of S = V^T H V)
//  dav_expand_kernel /     Ritz vector x = V y, HV y, residual r = HV y - theta x, correction t = r / (D - theta)
//  dav_orth_kernel         (|D - theta| floored), two-pass classical Gram-Schmidt against the basis, normalised new
//                          basis row; thick restart to [x, x_prev] when the basis is full
//  pcg_partial_kernel /    one step of deflated PCG on (H + sigma) x = b: alpha, x, r, z = r / (D + sigma), beta, p;
//  pcg_update_kernel       the shift is applied here, so the product needs none
//
// Vectors are split into P contiguous slices, one per CTA; every reduction is a per-CTA block sum followed by a sum
// over the P partials in CTA order, done identically by every CTA that needs it.  No atomics, no host
// synchronisation: repeats are bit-identical and the calls can be captured in a CUDA graph.
#include "common.cuh"

#include <cooperative_groups.h>

namespace cg = cooperative_groups;

namespace oo {

namespace {

constexpr int kKryThreads = 256;
constexpr int kSubMaxK = 64;                 // largest projected matrix / basis
constexpr int kMaxSlices = 1024;             // upper bound on P used for workspace sizing
constexpr int kPartW = kSubMaxK + 4;         // doubles per CTA in a partial-sum row

int slice_count(int64_t n) {
    int64_t p = ceil_div(n, kKryThreads);
    const int cap = sm_count() < kMaxSlices ? sm_count() : kMaxSlices;
    if (p > cap) p = cap;
    return p < 1 ? 1 : (int)p;
}

__device__ __forceinline__ void slice_of(int64_t n, int P, int b, int64_t &lo, int64_t &hi) {
    const int64_t c = (n + P - 1) / P;
    lo = (int64_t)b * c;
    hi = lo + c < n ? lo + c : n;
}

// sum over the P partial rows of column `col`, in CTA order
__device__ __forceinline__ double reduce_partials(const double *part, int P, int col) {
    double s = 0.0;
    for (int b = 0; b < P; ++b) s += part[(int64_t)b * kPartW + col];
    return s;
}

// ---------------------------------------------------------------------------------------------- subspace eigh
__global__ void __launch_bounds__(kKryThreads) subspace_eigh_kernel(const double *__restrict__ S, int k, int lds,
                                                                    int64_t strideS, double *__restrict__ w,
                                                                    int64_t stridew, double *__restrict__ Y, int ldy,
                                                                    int64_t strideY) {
    extern __shared__ double sm[];
    const int st = k | 1;                                   // odd row stride: column sweeps hit distinct banks
    double *A = sm, *V = A + k * st;
    __shared__ double rc[kSubMaxK / 2], rs[kSubMaxK / 2], rt[kSubMaxK / 2], rpq[kSubMaxK / 2];
    __shared__ double rpp[kSubMaxK / 2], rqq[kSubMaxK / 2], red[32];
    __shared__ int rp[kSubMaxK / 2], rq[kSubMaxK / 2], rank[kSubMaxK];
    __shared__ int rotated;
    const int tid = threadIdx.x;
    const double *Sb = S + (int64_t)blockIdx.x * strideS;
    double fro = 0.0;
    for (int e = tid; e < k * k; e += kKryThreads) {
        const int i = e / k, j = e % k;
        const double a = i >= j ? Sb[(int64_t)i * lds + j] : Sb[(int64_t)j * lds + i];   // lower triangle
        A[i * st + j] = a;
        V[i * st + j] = i == j ? 1.0 : 0.0;
        fro += a * a;
    }
    fro = sqrt(block_sum(fro, red));
    // a rotation that would remove less than this changes no eigenvalue by more than it: skipped
    const double skip = 0x1p-56 * fro;
    const int m = k + (k & 1), half = m / 2;                 // round-robin players (one dummy when k is odd)
    for (int sweep = 0; sweep < 60; ++sweep) {
        if (tid == 0) rotated = 0;
        __syncthreads();
        for (int r = 0; r < m - 1; ++r) {
            if (tid < half) {
                int a, b;
                if (tid == 0) {
                    a = r;
                    b = m - 1;
                } else {
                    a = (r + tid) % (m - 1);
                    b = (r - tid + (m - 1)) % (m - 1);
                }
                const int p = a < b ? a : b, q = a < b ? b : a;
                int use = 0;
                if (q < k) {
                    const double app = A[p * st + p], aqq = A[q * st + q], apq = A[p * st + q];
                    if (fabs(apq) > skip) {
                        const double tau = (aqq - app) / (2.0 * apq);
                        const double t = (tau >= 0.0 ? 1.0 : -1.0) / (fabs(tau) + sqrt(1.0 + tau * tau));
                        const double c = 1.0 / sqrt(1.0 + t * t);
                        rc[tid] = c;
                        rs[tid] = t * c;
                        rt[tid] = t;
                        rpp[tid] = app;
                        rqq[tid] = aqq;
                        rpq[tid] = apq;
                        use = 1;
                        rotated = 1;
                    }
                }
                rp[tid] = use ? p : -1;
                rq[tid] = q;
            }
            __syncthreads();
            // rows p, q  <-  J^T A
            for (int e = tid; e < half * k; e += kKryThreads) {
                const int i = e / k, j = e % k, p = rp[i];
                if (p < 0) continue;
                const int q = rq[i];
                const double c = rc[i], s = rs[i], ap = A[p * st + j], aq = A[q * st + j];
                A[p * st + j] = c * ap - s * aq;
                A[q * st + j] = s * ap + c * aq;
            }
            __syncthreads();
            // columns p, q  <-  A J,  V J
            for (int e = tid; e < half * k; e += kKryThreads) {
                const int i = e / k, j = e % k, p = rp[i];
                if (p < 0) continue;
                const int q = rq[i];
                const double c = rc[i], s = rs[i];
                double ap = A[j * st + p], aq = A[j * st + q];
                A[j * st + p] = c * ap - s * aq;
                A[j * st + q] = s * ap + c * aq;
                ap = V[j * st + p];
                aq = V[j * st + q];
                V[j * st + p] = c * ap - s * aq;
                V[j * st + q] = s * ap + c * aq;
            }
            __syncthreads();
            // the rotated 2 x 2 block exactly
            if (tid < half && rp[tid] >= 0) {
                const int p = rp[tid], q = rq[tid];
                A[p * st + p] = rpp[tid] - rt[tid] * rpq[tid];
                A[q * st + q] = rqq[tid] + rt[tid] * rpq[tid];
                A[p * st + q] = 0.0;
                A[q * st + p] = 0.0;
            }
            __syncthreads();
        }
        const int any = rotated;
        __syncthreads();
        if (!any) break;
    }
    // ascending order; equal values keep their index order
    if (tid < k) {
        const double d = A[tid * st + tid];
        int pos = 0;
        for (int j = 0; j < k; ++j) {
            const double e = A[j * st + j];
            pos += (e < d) || (e == d && j < tid);
        }
        rank[tid] = pos;
        w[(int64_t)blockIdx.x * stridew + pos] = d;
    }
    __syncthreads();
    double *Yb = Y + (int64_t)blockIdx.x * strideY;
    for (int e = tid; e < k * k; e += kKryThreads) {
        const int i = e / k, j = e % k;
        Yb[(int64_t)i * ldy + rank[j]] = V[i * st + j];
    }
}

size_t eigh_smem_bytes(int k) { return (size_t)2 * k * (k | 1) * sizeof(double); }

// ---------------------------------------------------------------------------------------------- Davidson
__global__ void __launch_bounds__(kKryThreads) dav_project_kernel(const double *__restrict__ Vt, int64_t ldv,
                                                                  int64_t n, const double *__restrict__ u,
                                                                  double *out, int inc, double *out2, int inc2) {
    __shared__ double red[32];
    const int j = blockIdx.x;
    const double *v = Vt + (int64_t)j * ldv;
    double s = 0.0;
    for (int64_t i = threadIdx.x; i < n; i += kKryThreads) s += v[i] * u[i];
    s = block_sum(s, red);
    if (threadIdx.x == 0) {
        out[(int64_t)j * inc] = s;
        if (out2) out2[(int64_t)j * inc2] = s;
    }
}

struct ExpandArgs {
    double *Vt, *HVt;
    int64_t n, ldv;
    int k, restart, P;
    const double *Y;
    int ldy;
    const double *theta, *D;
    double floor_;
    double *S;
    int lds;
    double *x, *hx, *yprev, *rnorm;
    double *t, *xp, *hxp, *part1, *part2, *coef;
};

// coefficients (in the current basis) of the previous Ritz vector made orthonormal to y: the second restart vector
__device__ void restart_coefficients(const double *y, const double *yp, int k, double *c) {
    double dot = 0.0;
    for (int j = 0; j < k; ++j) dot += y[j] * yp[j];
    for (int j = 0; j < k; ++j) c[j] = yp[j] - dot * y[j];
    double nrm = 0.0;
    for (int j = 0; j < k; ++j) nrm += c[j] * c[j];
    if (!(nrm > 1e-24)) {                                   // x_prev parallel to x: any direction orthogonal to y
        int jm = 0;
        for (int j = 1; j < k; ++j)
            if (fabs(y[j]) < fabs(y[jm])) jm = j;
        for (int j = 0; j < k; ++j) c[j] = (j == jm ? 1.0 : 0.0) - y[jm] * y[j];
    }
    for (int pass = 0; pass < 2; ++pass) {
        dot = 0.0;
        for (int j = 0; j < k; ++j) dot += y[j] * c[j];
        for (int j = 0; j < k; ++j) c[j] -= dot * y[j];
    }
    nrm = 0.0;
    for (int j = 0; j < k; ++j) nrm += c[j] * c[j];
    nrm = sqrt(nrm);
    for (int j = 0; j < k; ++j) c[j] /= nrm;
}

__global__ void __launch_bounds__(kKryThreads) dav_expand_kernel(ExpandArgs a) {
    __shared__ double y[kSubMaxK], c[kSubMaxK], red[32];
    const int tid = threadIdx.x, k = a.k;
    if (tid < k) y[tid] = a.Y[(int64_t)tid * a.ldy];
    __syncthreads();
    if (a.restart && tid == 0) {
        restart_coefficients(y, a.yprev, k, c);
        if (blockIdx.x == 0)
            for (int j = 0; j < k; ++j) a.coef[j] = c[j];
    }
    __syncthreads();
    const double theta = *a.theta;
    int64_t lo, hi;
    slice_of(a.n, a.P, blockIdx.x, lo, hi);
    double rr = 0.0, tt = 0.0;
    for (int64_t i = lo + tid; i < hi; i += kKryThreads) {
        double xi = 0.0, hxi = 0.0;
        for (int j = 0; j < k; ++j) {
            xi += y[j] * a.Vt[(int64_t)j * a.ldv + i];
            hxi += y[j] * a.HVt[(int64_t)j * a.ldv + i];
        }
        const double ri = hxi - theta * xi;
        double d = a.D[i] - theta;
        if (fabs(d) < a.floor_) d = d < 0.0 ? -a.floor_ : a.floor_;
        a.x[i] = xi;
        a.hx[i] = hxi;
        a.t[i] = ri / d;
        rr += ri * ri;
        tt += (ri / d) * (ri / d);
        if (a.restart) {
            double pi = 0.0, hpi = 0.0;
            for (int j = 0; j < k; ++j) {
                pi += c[j] * a.Vt[(int64_t)j * a.ldv + i];
                hpi += c[j] * a.HVt[(int64_t)j * a.ldv + i];
            }
            a.xp[i] = pi;
            a.hxp[i] = hpi;
        }
    }
    // first Gram-Schmidt pass: t against the basis the new vector joins (V, or [x, x_prev] on a restart)
    const int nb = a.restart ? 2 : k;
    double *prow = a.part1 + (int64_t)blockIdx.x * kPartW;
    for (int j = 0; j < nb; ++j) {
        const double *bj = a.restart ? (j == 0 ? a.x : a.xp) : a.Vt + (int64_t)j * a.ldv;
        double s = 0.0;
        for (int64_t i = lo + tid; i < hi; i += kKryThreads) s += bj[i] * a.t[i];
        s = block_sum(s, red);
        if (tid == 0) prow[j] = s;
    }
    rr = block_sum(rr, red);
    tt = block_sum(tt, red);
    if (tid == 0) {
        prow[kSubMaxK] = rr;
        prow[kSubMaxK + 2] = tt;                            // ||t||^2 before Gram-Schmidt: breakdown test
    }
}

__global__ void __launch_bounds__(kKryThreads) dav_orth_kernel(ExpandArgs a) {
    cg::grid_group grid = cg::this_grid();
    __shared__ double cf[kSubMaxK], red[32];
    __shared__ double rr;
    const int tid = threadIdx.x, k = a.k, nb = a.restart ? 2 : k;
    int64_t lo, hi;
    slice_of(a.n, a.P, blockIdx.x, lo, hi);
    auto basis = [&](int j) -> const double * {
        return a.restart ? (j == 0 ? a.x : a.xp) : a.Vt + (int64_t)j * a.ldv;
    };
    const double *part[2] = {a.part1, a.part2};
    for (int pass = 0; pass < 2; ++pass) {
        if (tid < nb) cf[tid] = reduce_partials(part[pass], a.P, tid);
        if (pass == 0 && tid == kKryThreads - 1) rr = reduce_partials(a.part1, a.P, kSubMaxK);
        __syncthreads();
        for (int64_t i = lo + tid; i < hi; i += kKryThreads) {
            double ti = a.t[i];
            for (int j = 0; j < nb; ++j) ti -= cf[j] * basis(j)[i];
            a.t[i] = ti;
        }
        double *prow = (pass == 0 ? a.part2 : a.part1) + (int64_t)blockIdx.x * kPartW;
        if (pass == 0) {                                    // dots of the second pass
            for (int j = 0; j < nb; ++j) {
                double s = 0.0;
                for (int64_t i = lo + tid; i < hi; i += kKryThreads) s += basis(j)[i] * a.t[i];
                s = block_sum(s, red);
                if (tid == 0) prow[j] = s;
            }
        } else {                                            // squared norm of the result (part1 is read by now)
            double s = 0.0;
            for (int64_t i = lo + tid; i < hi; i += kKryThreads) s += a.t[i] * a.t[i];
            s = block_sum(s, red);
            if (tid == 0) prow[kSubMaxK + 1] = s;
        }
        grid.sync();
    }
    // breakdown: the correction lies in the span of the basis (what is left is round-off, or not finite).  The new
    // row is then zero instead of amplified noise, and rnorm[1] = 1 tells the caller.
    const double tt = reduce_partials(a.part1, a.P, kSubMaxK + 1), tt0 = reduce_partials(a.part1, a.P, kSubMaxK + 2);
    const bool breakdown = !(tt > 1e-24 * tt0) || !isfinite(tt);
    const double inv = breakdown ? 0.0 : 1.0 / sqrt(tt);
    const int row = a.restart ? 2 : k;
    for (int64_t i = lo + tid; i < hi; i += kKryThreads) {
        a.Vt[(int64_t)row * a.ldv + i] = a.t[i] * inv;
        if (a.restart) {
            a.Vt[i] = a.x[i];
            a.HVt[i] = a.hx[i];
            a.Vt[a.ldv + i] = a.xp[i];
            a.HVt[a.ldv + i] = a.hxp[i];
        }
    }
    if (blockIdx.x == 0 && tid == 0) {
        a.rnorm[0] = sqrt(rr);
        a.rnorm[1] = breakdown ? 1.0 : 0.0;
        if (a.restart) {
            // S' = C^T S C for C = [y, c]: the projected matrix of the two restart vectors
            const double *y = a.Y, *c = a.coef;
            double s00 = 0.0, s01 = 0.0, s11 = 0.0;
            for (int i = 0; i < k; ++i)
                for (int j = 0; j < k; ++j) {
                    const double sij = a.S[(int64_t)i * a.lds + j];
                    const double yi = y[(int64_t)i * a.ldy], yj = y[(int64_t)j * a.ldy];
                    s00 += yi * sij * yj;
                    s01 += yi * sij * c[j];
                    s11 += c[i] * sij * c[j];
                }
            a.S[0] = s00;
            a.S[1] = s01;
            a.S[a.lds] = s01;
            a.S[a.lds + 1] = s11;
            for (int j = 0; j < k; ++j) a.yprev[j] = j == 0 ? 1.0 : 0.0;      // x is basis vector 0 now
        } else {
            for (int j = 0; j < k; ++j) a.yprev[j] = a.Y[(int64_t)j * a.ldy];
            a.yprev[k] = 0.0;
        }
    }
}

// ---------------------------------------------------------------------------------------------- PCG
struct PcgArgs {
    int64_t n;
    int P, init;
    const double *Ap, *D, *w, *aw;
    double shift;
    double *x, *r, *p, *z, *state, *rnorm, *part;
};

__global__ void __launch_bounds__(kKryThreads) pcg_partial_kernel(PcgArgs a) {
    __shared__ double red[32];
    int64_t lo, hi;
    slice_of(a.n, a.P, blockIdx.x, lo, hi);
    double s0 = 0.0, s1 = 0.0;
    for (int64_t i = lo + threadIdx.x; i < hi; i += kKryThreads) {
        if (a.init) {                                       // w . b  and  w . (H + sigma) w
            if (a.w) {
                s0 += a.w[i] * a.r[i];
                s1 += a.w[i] * a.aw[i];
            }
        } else {                                            // p . (H + sigma) p
            s0 += a.p[i] * (a.Ap[i] + a.shift * a.p[i]);
        }
    }
    s0 = block_sum(s0, red);
    s1 = block_sum(s1, red);
    if (threadIdx.x == 0) {
        a.part[(int64_t)blockIdx.x * kPartW + 0] = s0;
        a.part[(int64_t)blockIdx.x * kPartW + 1] = s1;
    }
}

__global__ void __launch_bounds__(kKryThreads) pcg_update_kernel(PcgArgs a) {
    cg::grid_group grid = cg::this_grid();
    __shared__ double red[32];
    int64_t lo, hi;
    slice_of(a.n, a.P, blockIdx.x, lo, hi);
    const int tid = threadIdx.x;
    const double s0 = reduce_partials(a.part, a.P, 0), s1 = reduce_partials(a.part, a.P, 1);
    const double rz_old = a.init ? 0.0 : a.state[0];
    const double waw = a.w == nullptr ? 1.0 : (a.init ? s1 : a.state[1]);
    const double step = a.init ? (a.w == nullptr ? 0.0 : s0 / waw) : rz_old / s0;
    double rz = 0.0, rr = 0.0, awz = 0.0;
    for (int64_t i = lo + tid; i < hi; i += kKryThreads) {
        double xi, ri;
        if (a.init) {                                       // Galerkin start in span{w}: x = w (w.b) / (w.Aw)
            xi = a.w == nullptr ? 0.0 : step * a.w[i];
            ri = a.w == nullptr ? a.r[i] : a.r[i] - step * a.aw[i];
        } else {
            const double pi = a.p[i];
            xi = a.x[i] + step * pi;
            ri = a.r[i] - step * (a.Ap[i] + a.shift * pi);
        }
        const double zi = ri / (a.D[i] + a.shift);
        a.x[i] = xi;
        a.r[i] = ri;
        a.z[i] = zi;
        rz += ri * zi;
        rr += ri * ri;
        if (a.w) awz += a.aw[i] * zi;
    }
    rz = block_sum(rz, red);
    rr = block_sum(rr, red);
    awz = block_sum(awz, red);
    grid.sync();                                            // every CTA has read part: it can be overwritten
    if (tid == 0) {
        double *prow = a.part + (int64_t)blockIdx.x * kPartW;
        prow[2] = rz;
        prow[3] = rr;
        prow[4] = awz;
    }
    grid.sync();
    const double rz_new = reduce_partials(a.part, a.P, 2);
    const double beta = a.init ? 0.0 : rz_new / rz_old;
    const double mu = a.w == nullptr ? 0.0 : reduce_partials(a.part, a.P, 4) / waw;
    for (int64_t i = lo + tid; i < hi; i += kKryThreads) {
        double pi = a.z[i] + (a.init ? 0.0 : beta * a.p[i]);
        if (a.w) pi -= mu * a.w[i];                         // search directions stay (H + sigma)-orthogonal to w
        a.p[i] = pi;
    }
    if (blockIdx.x == 0 && tid == 0) {
        a.state[0] = rz_new;
        if (a.init) a.state[1] = waw;
        *a.rnorm = sqrt(reduce_partials(a.part, a.P, 3));
    }
}

int launch_cooperative(const void *fn, int P, void *arg, cudaStream_t stream) {
    static unsigned long long checked = 0;
    static int coop[64] = {};
    int dev = 0;
    OO_CUDA_CHECK(cudaGetDevice(&dev));
    if (once_per_device(checked)) {
        int v = 0;
        OO_CUDA_CHECK(cudaDeviceGetAttribute(&v, cudaDevAttrCooperativeLaunch, dev));
        if (dev < 64) coop[dev] = v;
    }
    if (dev >= 64 || !coop[dev]) return OO_ERR_NO_DEVICE;
    void *args[] = {arg};
    OO_CUDA_CHECK(cudaLaunchCooperativeKernel(fn, dim3((unsigned)P), dim3(kKryThreads), args, 0, stream));
    OO_LAUNCH_CHECK();
    return OO_OK;
}

struct KrylovLayout {
    size_t off_part1, off_part2, off_t, off_xp, off_hxp, off_coef, total;
};

KrylovLayout krylov_layout(int64_t n) {
    KrylovLayout L;
    const size_t part = align_up((size_t)kMaxSlices * kPartW * sizeof(double), 256);
    const size_t vec = align_up((size_t)n * sizeof(double), 256);
    L.off_part1 = 0;
    L.off_part2 = part;
    L.off_t = 2 * part;
    L.off_xp = L.off_t + vec;
    L.off_hxp = L.off_xp + vec;
    L.off_coef = L.off_hxp + vec;
    L.total = L.off_coef + align_up(kSubMaxK * sizeof(double), 256);
    return L;
}

}  // namespace

size_t krylov_ws_bytes(int64_t n, int k) {
    if (n <= 0 || k <= 0 || k > kSubMaxK) return 0;
    return krylov_layout(n).total;
}

int subspace_eigh(const double *S, int k, int lds, int64_t strideS, int batch, double *w, int64_t stridew, double *Y,
                  int ldy, int64_t strideY, cudaStream_t stream) {
    OO_REQUIRE(S && w && Y);
    OO_REQUIRE(k > 0 && k <= kSubMaxK && lds >= k && ldy >= k && batch > 0 && batch <= 65535);
    OO_REQUIRE(batch == 1 || (strideS >= (int64_t)lds * k && stridew >= k && strideY >= (int64_t)ldy * k));
    static unsigned long long cfgd = 0;
    if (once_per_device(cfgd))
        OO_CUDA_CHECK(cudaFuncSetAttribute(subspace_eigh_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           (int)eigh_smem_bytes(kSubMaxK)));
    subspace_eigh_kernel<<<(unsigned)batch, kKryThreads, eigh_smem_bytes(k), stream>>>(S, k, lds, strideS, w, stridew,
                                                                                      Y, ldy, strideY);
    OO_LAUNCH_CHECK();
    return OO_OK;
}

int davidson_project(const double *Vt, int64_t ldv, int64_t n, int k, const double *u, double *out, int inc,
                     double *out2, int inc2, cudaStream_t stream) {
    OO_REQUIRE(Vt && u && out && n > 0 && ldv >= n && k > 0 && k <= kSubMaxK && inc > 0);
    OO_REQUIRE(out2 == nullptr || inc2 > 0);
    dav_project_kernel<<<(unsigned)k, kKryThreads, 0, stream>>>(Vt, ldv, n, u, out, inc, out2, inc2);
    OO_LAUNCH_CHECK();
    return OO_OK;
}

int davidson_expand(double *Vt, double *HVt, int64_t n, int64_t ldv, int k, int kmax, const double *Y, int ldy,
                    const double *theta, const double *D, double floor_, double *S, int lds, double *x, double *hx,
                    double *yprev, double *rnorm, void *ws, size_t ws_bytes, cudaStream_t stream) {
    OO_REQUIRE(Vt && HVt && Y && theta && D && S && x && hx && yprev && rnorm && ws);
    OO_REQUIRE(n > 0 && ldv >= n && kmax >= 3 && kmax <= kSubMaxK && k > 0 && k <= kmax);
    OO_REQUIRE(ldy >= k && lds >= kmax && floor_ > 0.0);
    const KrylovLayout L = krylov_layout(n);
    if (ws_bytes < L.total) return OO_ERR_WORKSPACE;
    uint8_t *wb = reinterpret_cast<uint8_t *>(ws);
    ExpandArgs a;
    a.Vt = Vt;
    a.HVt = HVt;
    a.n = n;
    a.ldv = ldv;
    a.k = k;
    a.restart = k == kmax;
    a.P = slice_count(n);
    a.Y = Y;
    a.ldy = ldy;
    a.theta = theta;
    a.D = D;
    a.floor_ = floor_;
    a.S = S;
    a.lds = lds;
    a.x = x;
    a.hx = hx;
    a.yprev = yprev;
    a.rnorm = rnorm;
    a.t = reinterpret_cast<double *>(wb + L.off_t);
    a.xp = reinterpret_cast<double *>(wb + L.off_xp);
    a.hxp = reinterpret_cast<double *>(wb + L.off_hxp);
    a.part1 = reinterpret_cast<double *>(wb + L.off_part1);
    a.part2 = reinterpret_cast<double *>(wb + L.off_part2);
    a.coef = reinterpret_cast<double *>(wb + L.off_coef);
    dav_expand_kernel<<<(unsigned)a.P, kKryThreads, 0, stream>>>(a);
    OO_LAUNCH_CHECK();
    return launch_cooperative((const void *)dav_orth_kernel, a.P, &a, stream);
}

int pcg_step(int64_t n, const double *Ap, double shift, const double *D, const double *w, const double *aw,
             double *x, double *r, double *p, double *state, double *rnorm, int init, void *ws, size_t ws_bytes,
             cudaStream_t stream) {
    OO_REQUIRE(D && x && r && p && state && rnorm && ws && n > 0);
    OO_REQUIRE(init || Ap);
    OO_REQUIRE((w == nullptr) == (aw == nullptr));
    const KrylovLayout L = krylov_layout(n);
    if (ws_bytes < L.total) return OO_ERR_WORKSPACE;
    uint8_t *wb = reinterpret_cast<uint8_t *>(ws);
    PcgArgs a;
    a.n = n;
    a.P = slice_count(n);
    a.init = init != 0;
    a.Ap = Ap;
    a.D = D;
    a.w = w;
    a.aw = aw;
    a.shift = shift;
    a.x = x;
    a.r = r;
    a.p = p;
    a.z = reinterpret_cast<double *>(wb + L.off_t);
    a.state = state;
    a.rnorm = rnorm;
    a.part = reinterpret_cast<double *>(wb + L.off_part1);
    pcg_partial_kernel<<<(unsigned)a.P, kKryThreads, 0, stream>>>(a);
    OO_LAUNCH_CHECK();
    return launch_cooperative((const void *)pcg_update_kernel, a.P, &a, stream);
}

}  // namespace oo

extern "C" int oo_subspace_eigh_f64(const double *S, int k, int lds, int64_t strideS, int batch, double *w,
                                    int64_t stridew, double *Y, int ldy, int64_t strideY, void *stream) {
    return oo::subspace_eigh(S, k, lds, strideS, batch, w, stridew, Y, ldy, strideY, (cudaStream_t)stream);
}

extern "C" int oo_davidson_project_f64(const double *Vt, int64_t ldv, int64_t n, int k, const double *u, double *out,
                                       int inc, double *out2, int inc2, void *stream) {
    return oo::davidson_project(Vt, ldv, n, k, u, out, inc, out2, inc2, (cudaStream_t)stream);
}

extern "C" int oo_davidson_expand_f64(double *Vt, double *HVt, int64_t n, int64_t ldv, int k, int kmax,
                                      const double *Y, int ldy, const double *theta, const double *D, double floor_,
                                      double *S, int lds, double *x, double *hx, double *yprev, double *rnorm,
                                      void *ws, size_t ws_bytes, void *stream) {
    return oo::davidson_expand(Vt, HVt, n, ldv, k, kmax, Y, ldy, theta, D, floor_, S, lds, x, hx, yprev, rnorm, ws,
                               ws_bytes, (cudaStream_t)stream);
}

extern "C" int oo_pcg_step_f64(int64_t n, const double *Ap, double shift, const double *D, const double *w,
                               const double *aw, double *x, double *r, double *p, double *state, double *rnorm,
                               int init, void *ws, size_t ws_bytes, void *stream) {
    return oo::pcg_step(n, Ap, shift, D, w, aw, x, r, p, state, rnorm, init, ws, ws_bytes, (cudaStream_t)stream);
}
