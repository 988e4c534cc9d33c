// C-ABI glue: versioning, error strings, device info, TMA descriptor encoding,
// workspace sizing, and K2b -- the four-index transform driver.
#include "common.cuh"

#include <mutex>

namespace oo {

int g_last_cuda_error = 0;
unsigned long long g_launch_count = 0;

int sm_count() {
    static int cached[64] = {};                         // per device
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev > 63) return 148;
    if (cached[dev] > 0) return cached[dev];
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
        return 148;
    cached[dev] = n;
    return n;
}

// cuTensorMapEncodeTiled is a driver-API symbol; fetch it through the runtime so the
// library links against cudart only (and loads on a machine without libcuda).
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *,
                                  const cuuint64_t *, const cuuint64_t *, const cuuint32_t *,
                                  const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    });
    return fn;
}

int encode_tmap_3d_f64(CUtensorMap *map, const void *base, uint64_t dim0, uint64_t dim1, uint64_t dim2,
                       uint64_t stride1_elems, uint64_t stride2_elems, uint32_t box0, uint32_t box1) {
    EncodeTiledFn fn = get_encode_fn();
    if (!fn) return OO_ERR_NO_DEVICE;
    cuuint64_t dims[3] = {dim0, dim1, dim2};
    cuuint64_t strides[2] = {stride1_elems * sizeof(double), stride2_elems * sizeof(double)};
    cuuint32_t box[3] = {box0, box1, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 3, const_cast<void *>(base), dims, strides, box,
                    estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                    CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        g_last_cuda_error = (int)r;
        return OO_ERR_CUDA;
    }
    return OO_OK;
}

int encode_tmap_4d_f64(CUtensorMap *map, const void *base, const uint64_t dims_in[4], const uint64_t strides_elems[3],
                       const uint32_t box_in[4]) {
    EncodeTiledFn fn = get_encode_fn();
    if (!fn) return OO_ERR_NO_DEVICE;
    cuuint64_t dims[4] = {dims_in[0], dims_in[1], dims_in[2], dims_in[3]};
    cuuint64_t strides[3] = {strides_elems[0] * sizeof(double), strides_elems[1] * sizeof(double),
                             strides_elems[2] * sizeof(double)};
    cuuint32_t box[4] = {box_in[0], box_in[1], box_in[2], box_in[3]};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 4, const_cast<void *>(base), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        g_last_cuda_error = (int)r;
        return OO_ERR_CUDA;
    }
    return OO_OK;
}

// K2b.  Each quarter is  Out[(q r s), i] = sum_p In[p, (q r s)] C[p, i]: the contracted
// (leading) index leaves at the front and its image arrives at the back, so after four
// quarters [p,q,r,s] -> [q,r,s,i] -> [r,s,i,j] -> [s,i,j,k] -> [i,j,k,l].
int int2e_transform(const double *g_ao, int64_t strideG, const double *C0, const double *C1,
                    const double *C2, const double *C3, int64_t strideC, int N, int ld, int batch,
                    double *g_mo, void *ws, size_t ws_bytes, cudaStream_t stream) {
    OO_REQUIRE(g_ao && C0 && C1 && C2 && C3 && g_mo && ws);
    OO_REQUIRE(N > 0 && ld >= N && (ld % 2) == 0 && batch > 0);
    const int64_t ld3 = (int64_t)ld * ld * ld;
    const int64_t ld4 = ld3 * ld;
    if (ws_bytes < (size_t)batch * ld4 * sizeof(double)) return OO_ERR_WORKSPACE;
    double *tmp = reinterpret_cast<double *>(ws);
    const double *Cs[4] = {C0, C1, C2, C3};
    const double *in = g_ao;
    int64_t in_stride = strideG;
    for (int q = 0; q < 4; ++q) {
        double *out = (q % 2 == 0) ? tmp : g_mo;
        int rc = dgemm_tn(in, Cs[q], out, ld3, ld, ld, ld3, ld, ld, batch, in_stride, strideC, ld4, stream);
        if (rc) return rc;
        in = out;
        in_stride = ld4;
    }
    return OO_OK;
}

}  // namespace oo

extern "C" {

int oo_abi_version(void) { return OO_ABI_VERSION; }

const char *oo_error_string(int code) {
    switch (code) {
        case OO_OK: return "success";
        case OO_ERR_INVALID_ARG: return "invalid argument";
        case OO_ERR_UNSUPPORTED: return "unsupported size";
        case OO_ERR_WORKSPACE: return "workspace too small";
        case OO_ERR_CUDA: return "CUDA error (see oo_last_cuda_error)";
        case OO_ERR_NO_DEVICE: return "no usable CUDA device / driver entry point";
        default: return "unknown error";
    }
}

int oo_last_cuda_error(void) { return oo::g_last_cuda_error; }

unsigned long long oo_launch_count(void) { return oo::g_launch_count; }

int oo_device_info(int *sm_count, int *cc_major, int *cc_minor) {
    int dev = 0;
    cudaDeviceProp prop;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaGetDeviceProperties(&prop, dev) != cudaSuccess)
        return OO_ERR_NO_DEVICE;
    if (sm_count) *sm_count = prop.multiProcessorCount;
    if (cc_major) *cc_major = prop.major;
    if (cc_minor) *cc_minor = prop.minor;
    return OO_OK;
}

size_t oo_workspace_bytes(int which, int N, int ld, int nI, int batch) {
    (void)N;
    if (ld <= 0 || batch <= 0) return 0;
    switch (which) {
        case OO_WS_ROTATION: return oo::rotation_ws_bytes(ld, batch);
        case OO_WS_INT2E: return (size_t)batch * ld * ld * ld * ld * sizeof(double);
        case OO_WS_HESSIAN: return oo::hessian_ws_bytes(ld, nI);
        case OO_WS_INT1E: return oo::int1e_ws_bytes(ld, batch);
        case OO_WS_YMATRIX: return oo::y_matrix_ws_bytes(ld, N);
        case OO_WS_CLASS_TRANSFORM: return oo::class_transform_ws_bytes(ld, nI + (nI & 1), batch);
        case OO_WS_CLASS_TRANSFORM_SYM: return oo::class_transform_sym_ws_bytes(ld, nI + (nI & 1), batch);
        case OO_WS_CLASS_BUFFER: return (size_t)batch * oo::class_buffer_bytes(ld, nI + (nI & 1));
        case OO_WS_CLASS_HESSIAN:   /* N carries na here (the sparse layout depends on no, na, not on N) */
            return oo::class_hessian_ws_bytes(ld, nI + (nI & 1), nI - N, N, batch);
        case OO_WS_CLASS_HESSIAN_VECTOR:   /* N carries na, batch the number of vectors */
            return (N > 0 && N <= nI) ? oo::class_hessian_vector_ws_bytes(ld, nI + (nI & 1), nI - N, N, batch) : 0;
        case OO_WS_HESSIAN_VECTOR:
            return (N > 0 && N <= nI) ? oo::hessian_vector_ws_bytes(ld, nI, N, batch) : 0;
        case OO_WS_HESSIAN_DIAGONAL: return oo::hessian_diagonal_ws_bytes(ld, nI);
        case OO_WS_KRYLOV: return oo::krylov_ws_bytes(N, nI);   /* N carries the vector length, nI the basis size */
        case OO_WS_ROTATION_VJP: return oo::rotation_vjp_ws_bytes(ld, batch);
        default: return 0;
    }
}

int oo_int2e_transform_f64(const double *g_ao, int64_t strideG, const double *C0, const double *C1,
                           const double *C2, const double *C3, int64_t strideC, int N, int ld,
                           int batch, double *g_mo, void *ws, size_t ws_bytes, void *stream) {
    return oo::int2e_transform(g_ao, strideG, C0, C1, C2, C3, strideC, N, ld, batch, g_mo, ws, ws_bytes,
                               (cudaStream_t)stream);
}
}
