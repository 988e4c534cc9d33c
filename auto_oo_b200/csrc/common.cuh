// Shared device/host helpers for the sm_100a kernels of the orbital-optimization hot path.
#pragma once

#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>

#include "../../include/oo_b200.h"

namespace oo {

// ---- error plumbing ---------------------------------------------------------
extern int g_last_cuda_error;
extern unsigned long long g_launch_count;   // kernels launched by this library (oo_launch_count)

inline int cuda_fail(cudaError_t e) {
    g_last_cuda_error = (int)e;
    return OO_ERR_CUDA;
}

#define OO_CUDA_CHECK(expr)                                   \
    do {                                                      \
        cudaError_t _e = (expr);                              \
        if (_e != cudaSuccess) return ::oo::cuda_fail(_e);    \
    } while (0)

#define OO_LAUNCH_CHECK()                      \
    do {                                       \
        ++::oo::g_launch_count;                \
        OO_CUDA_CHECK(cudaGetLastError());     \
    } while (0)

#define OO_REQUIRE(cond)                          \
    do {                                          \
        if (!(cond)) return OO_ERR_INVALID_ARG;   \
    } while (0)

inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }
inline size_t align_up(size_t a, size_t b) { return (a + b - 1) / b * b; }

int sm_count();   // cached cudaDevAttrMultiProcessorCount of the current device

// Function attributes (opt-in dynamic shared memory) are per DEVICE: `once_per_device(mask)` is true the first time
// it is called with the calling thread's current device for a given call-site mask (devices 0..63; a process that
// drives several GPUs configures each of them).  Benign race: two threads may both configure the same device.
inline bool once_per_device(unsigned long long &mask) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev > 63) return true;
    const unsigned long long bit = 1ull << dev;
    if (mask & bit) return false;
    mask |= bit;
    return true;
}

// compile-time booleans for generic lambdas, e.g. a GEMM main loop's k-block body called with TrueTag{} for the last
// k-block only
struct FalseTag { static constexpr bool value = false; };
struct TrueTag { static constexpr bool value = true; };

// ---- FP64 tensor-core MMA (DMMA.8x8x4) --------------------------------------
// Fragment ownership for lane = 4*g + t (g = 0..7, t = 0..3):
//   a = A[g][t]   (row-major 8x4),  b = B[t][g]  (col-major 4x8),
//   c0,c1 = C[g][2t], C[g][2t+1]
__device__ __forceinline__ void dmma884(double &c0, double &c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

// ---- shared-memory / mbarrier / TMA wrappers ---------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) {
    return (uint32_t)__cvta_generic_to_shared(p);
}

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}

__device__ __forceinline__ void fence_barrier_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}

__device__ __forceinline__ void fence_proxy_async() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
                 "r"(bytes)
                 : "memory");
}

__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

__device__ __forceinline__ void mbar_arrive_addr(uint32_t bar_smem_addr) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar_smem_addr) : "memory");
}

__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, uint32_t parity) {
    uint32_t done;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(done)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return done != 0;
}

__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    while (!mbar_try_wait(bar, parity)) {
    }
}

__device__ __forceinline__ void tma_load_3d(void *smem_dst, const CUtensorMap *map, uint64_t *bar,
                                            int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(smem_u32(smem_dst)),
        "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}

__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap *map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}

__device__ __forceinline__ double lds_f64(uint32_t addr) {
    double v;
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(addr));
    return v;
}

// ---- reductions -----------------------------------------------------------------
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// block-wide sum; every thread gets the result.  `scratch` >= 32 doubles of smem.
__device__ __forceinline__ double block_sum(double v, double *scratch) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int nwarp = (blockDim.x + 31) >> 5;
    v = warp_sum(v);
    __syncthreads();
    if (lane == 0) scratch[warp] = v;
    __syncthreads();
    double r = (lane < nwarp) ? scratch[lane] : 0.0;
    r = warp_sum(r);
    return r;
}

// ---- views of the transformed two-electron integrals ----------------------------
// Every contraction of the hot path touches g' only through two access patterns with at
// least two indices m, n in I = occ + act:
//   coul(a,b,m,n) = g'[a,b,m,n]     (Coulomb class  (ab|mn))
//   exch(a,m,n,b) = g'[a,m,n,b]     (exchange class (am|nb))
// FullView reads them from the complete ld^4 tensor of the four-index transform;
// ClassView from the two class tensors of the partial transform (classes.cu):
//   J[m,n,a,b] = g'[a,b,m,n],  K[n,m,a,b] = g'[a,m,n,b],  each [nIp][nIp][ld][ld].
struct FullView {
    const double *g;
    int ld;
    int64_t batch_stride;
    __device__ __forceinline__ FullView at(int b) const { return {g + (int64_t)b * batch_stride, ld, batch_stride}; }
    __device__ __forceinline__ double coul(int a, int b, int m, int n) const {
        return g[(((int64_t)a * ld + b) * ld + m) * ld + n];
    }
    __device__ __forceinline__ double exch(int a, int m, int n, int b) const {
        return g[(((int64_t)a * ld + m) * ld + n) * ld + b];
    }
};

struct ClassView {
    const double *K, *J;      // K first: the Hessian's B operand is [K rows; J rows; h row]
    int ld, nIp;
    int64_t batch_stride;
    __device__ __forceinline__ ClassView at(int b) const {
        return {K + (int64_t)b * batch_stride, J + (int64_t)b * batch_stride, ld, nIp, batch_stride};
    }
    __device__ __forceinline__ double coul(int a, int b, int m, int n) const {
        return J[(((int64_t)m * nIp + n) * ld + a) * ld + b];
    }
    __device__ __forceinline__ double exch(int a, int m, int n, int b) const {
        return K[(((int64_t)n * nIp + m) * ld + a) * ld + b];
    }
};

// ---- host: TMA descriptor encode (driver entry point fetched at run time) -----
int encode_tmap_3d_f64(CUtensorMap *map, const void *base, uint64_t dim0, uint64_t dim1,
                       uint64_t dim2, uint64_t stride1_elems, uint64_t stride2_elems,
                       uint32_t box0, uint32_t box1);
int encode_tmap_4d_f64(CUtensorMap *map, const void *base, const uint64_t dims[4], const uint64_t strides_elems[3],
                       const uint32_t box[4]);

// ---- host: functions one source file defines and others call ------------------
// TN-GEMMs on the FP64 tensor pipe (dgemm_tn.cu, dgemm_tri.cu)
int dgemm_tn(const double *At, const double *B, double *C, int64_t M, int64_t N, int64_t K,
             int64_t lda, int64_t ldb, int64_t ldc, int batch, int64_t strideA, int64_t strideB,
             int64_t strideC, cudaStream_t stream);
int dgemm_tn_direct(const double *At, const double *B, double *C, int64_t M, int64_t N, int64_t K,
                    int64_t lda, int64_t ldb, int64_t ldc, int batch, int64_t strideA, int64_t strideB,
                    int64_t strideC, cudaStream_t stream);
int dgemm_tn_swap02(const double *At, const double *B, double *C, double *C2, int d0, int d1, int d2,
                    int64_t N, int64_t K, int64_t lda, int64_t ldb, int64_t ldc, int batch, int64_t strideA,
                    int64_t strideB, int64_t strideC, cudaStream_t stream);
int dgemm_tn_pair_unpack(const double *At, const double *B, double *C, double *C2, int d0, int dorb, int dP,
                         int64_t N, int64_t K, int64_t lda, int64_t ldb, int64_t ldc, int batch,
                         int64_t strideA, int64_t strideB, int64_t strideC, int64_t strideC2,
                         cudaStream_t stream);
int dgemm_tn_class_pack(const double *At, const double *B, double *P, int tri_rows, int nclass, int dorb,
                        int64_t nrows2, int64_t npair_ld, int64_t K, int64_t lda, int64_t ldb, int batch,
                        int64_t strideA, int64_t strideB, int64_t strideP, cudaStream_t stream, int64_t r2_offset = 0);
int dgemm_tn_q1_packed8(const double *A8, int64_t a8_ld, int pq_lo, int pq_cnt, const double *B, double *C,
                        double *C2, int dorb, int dP, int64_t N, int64_t K, int64_t ldb, int64_t ldc, int batch,
                        int64_t strideA8, int64_t strideB, int64_t strideC, int64_t strideC2, cudaStream_t stream,
                        bool direct_epilogue);
int dgemm_tn_class_expand(const double *At, const double *B, double *Out, int transpose_mirror, int nclass, int dorb,
                          int64_t npair_ld, int64_t K, int64_t lda, int64_t ldb, int64_t ld_out, int batch,
                          int64_t strideA, int64_t strideB, int64_t strideOut, cudaStream_t stream,
                          bool direct_epilogue = false);
bool dgemm_tn_tri_supported(int nclass);
int dgemm_tn_tri_class_pack(const double *At, const double *B, double *P, int tri_rows, int nclass, int dorb,
                            int64_t ngroups, int64_t npair_ld, int64_t K, int64_t lda, int64_t ldb, int batch,
                            int64_t strideA, int64_t strideB, int64_t strideP, cudaStream_t stream,
                            int64_t group_offset = 0, int64_t group_ld = 0, int halves = 1);
// small GEMM on the FP64 tensor pipe (dgemm_small.cu)
int dgemm_small(int transA, int transB, int M, int N, int K, double alpha, const double *A, int lda,
                int64_t strideA, const double *B, int ldb, int64_t strideB, double beta,
                const double *E, int lde, int64_t strideE, double gamma, double *D, int ldd,
                int64_t strideD, int batch, cudaStream_t stream, int eye_n);

// the class Hessian and the gathered class layout of the (h', g') forms (hessian.cu)
int class_hessian(const double *cls, const double *F, const double *d1, int64_t sd1, const double *d2,
                  int64_t sd2, int no, int na, int N, int ld, int nIp, int batch, const int32_t *pl,
                  const int32_t *pr, int nk, double *H, void *ws, size_t ws_bytes, unsigned flags,
                  cudaStream_t stream);
int gather_class_layout(const double *h, const double *g, int nI, int ld, double *B, cudaStream_t stream);
size_t full_hessian_b_bytes(int ld, int nIp);

// workspace and buffer sizes (oo_workspace_bytes)
size_t rotation_ws_bytes(int ld, int batch);
size_t rotation_vjp_ws_bytes(int ld, int batch);
size_t int1e_ws_bytes(int ld, int batch);
size_t hessian_ws_bytes(int ld, int nI);
size_t y_matrix_ws_bytes(int ld, int N);
size_t class_transform_ws_bytes(int ld, int nIp, int batch);
size_t class_buffer_bytes(int ld, int nIp);
size_t class_transform_sym_ws_bytes(int ld, int nIp, int batch);
size_t class_hessian_ws_bytes(int ld, int nIp, int no, int na, int batch);
size_t class_hessian_vector_ws_bytes(int ld, int nIp, int no, int na, int nv);
size_t hessian_vector_ws_bytes(int ld, int nI, int na, int nv);
size_t hessian_diagonal_ws_bytes(int ld, int nI);
size_t krylov_ws_bytes(int64_t n, int k);

}  // namespace oo
