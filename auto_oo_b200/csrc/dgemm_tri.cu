// Quarter 2 of the symmetric class transform as a TRIANGULAR TN-GEMM (sm_100a).
//
//   X[(g, m), n] = sum_k At[k, (g, m)] C[k, n],     m, n < nclass  (class indices, occ + act)
//
// where only the class pairs n <= m are kept (J[m,n] = J[n,m], K[n,m] = K[m,n]^T: classes.cu) and written packed,
// P[g'][m(m+1)/2 + n].  Rows come in GROUPS of nclass consecutive rows (one group g per AO pair of the quarter-1
// result, the class index m fastest); dgemm_tn.cu treats them as a flat row index, so a 256-row tile mixes all m
// and has to compute every column n for every row -- half of those products are thrown away by its epilogue.
// Here a group is the unit of tiling:
//   * the A operand is fetched through a 4-D tensor map (m, group, k, batch) with boxes [BK k][1 group][16 m]
//     (128-byte swizzle, m >= nclass zero-filled), so that in shared memory every group occupies GP = 16 ceil(nclass/16)
//     rows and an 8-row MMA tile holds the class indices 8 mi .. 8 mi + 7 of ONE group;
//   * one consumer warp per group: warp tile GP x GP, of which only the MMA tiles on and below the diagonal
//     (ni <= mi) are issued: 21 of 36 DMMA.8x8x4 per k4-step at GP = 48 (nclass = 44), 10 of 16 at GP = 32;
//   * the epilogue writes P[g'][m(m+1)/2 + n], n <= m, where g' = g (exchange class: rows (p, s)) or both (p, q) and
//     (q, p) of the packed pair g = p(p+1)/2 + q (Coulomb class).
// Same pipeline as dgemm_tn.cu: one producer warpgroup (one lane issues TMA), STAGES-deep ring with full / empty
// mbarriers, two consumer warpgroups on the FP64 tensor pipe, setmaxnreg 40 / 232, persistent grid, and the
// register-dependent stage release (TnArgs::zero in dgemm_tn.cu explains why).
#include "common.cuh"

namespace oo {

namespace {

// MTC_: 8-row MMA tiles per group that hold class indices (ceil(nclass / 8) <= GP / 8); tiles past it are padding
template <int GP_, int MTC_, int STAGES_>
struct TriCfg {
    static constexpr int GP = GP_, STAGES = STAGES_, BK = 16;
    static constexpr int NCW = 8;                         // consumer warps = groups per tile
    static constexpr int THREADS = (NCW + 4) * 32;
    static constexpr int MT = MTC_;                       // MMA tiles per side of the warp tile
    static_assert(MTC_ * 8 <= GP_, "class tiles exceed the group");
    static constexpr int CPG = GP / 16;                   // 16-wide TMA chunks per group
    static constexpr int CHUNK_BYTES = BK * 128;
    static constexpr int A_BYTES = NCW * CPG * CHUNK_BYTES;
    static constexpr int B_BYTES = CPG * CHUNK_BYTES;
    static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
    static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 2 * STAGES * 8 + 1024;
    static_assert((STAGES & (STAGES - 1)) == 0, "STAGES must be a power of two");
    static_assert(SMEM_BYTES <= 227 * 1024, "stage ring exceeds the shared memory of an SM");
};

struct TriArgs {
    double *P;              // packed output rows of length npair_ld
    int64_t npair_ld, strideP;
    int nclass;             // valid class indices per group (<= GP)
    int tri_rows;           // 1: group = packed pair p(p+1)/2 + q of dorb orbitals, written at (p q) and (q p)
    int dorb;
    int64_t ngroups;
    int64_t group_offset;   // tri_rows: the packed pair of group g is group_offset + g (a slab of the pairs)
    int kblocks, tiles_per_batch, batch;
    int halves;             // 2: every group row holds the class columns of TWO evaluations side by side (quarter 1 ran
                            // on [C_2j | C_2j+1]); tile u of batch element j is half u % 2 of group tile u / 2, reads
                            // columns h nclass .., multiplies by C_(2j+h) and writes P_(2j+h).  The two halves of a
                            // group tile run back to back, so the second finds the rows in L2.
    int a_batched, b_batched;
    int last_subs;          // substeps of the last k-block with rows below K
    uint32_t zero;
};

__device__ __forceinline__ void tma_load_4d(void *smem_dst, const CUtensorMap *map, uint64_t *bar, int c0, int c1,
                                            int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(smem_u32(smem_dst)),
        "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}

template <class Cfg>
__global__ void __launch_bounds__(Cfg::THREADS, 1)
dgemm_tn_tri_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB,
                    const TriArgs args) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t *smem = smem_raw + (smem_base - smem_u32(smem_raw));
    uint64_t *full_bar = reinterpret_cast<uint64_t *>(smem + Cfg::STAGES * Cfg::STAGE_BYTES);
    uint64_t *empty_bar = full_bar + Cfg::STAGES;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
#pragma unroll
        for (int s = 0; s < Cfg::STAGES; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], Cfg::NCW);
        }
        fence_barrier_init();
        tma_prefetch_desc(&mapA);
        tma_prefetch_desc(&mapB);
    }
    __syncthreads();
    const int64_t total_tiles = (int64_t)args.tiles_per_batch * args.batch;

    if (warp >= Cfg::NCW) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
        if (warp == Cfg::NCW && lane == 0) {                 // ---- TMA producer
            int stage = 0;
            uint32_t phase = 0;
            for (int64_t tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
                const int b = (int)(tile / args.tiles_per_batch);
                const int u = (int)(tile - (int64_t)b * args.tiles_per_batch);
                const int h = u % args.halves, g0 = (u / args.halves) * Cfg::NCW;
                const int ba = args.a_batched ? b : 0, bb = args.b_batched ? b * args.halves + h : 0;
                const int m0 = h * args.nclass;
                for (int kb = 0; kb < args.kblocks; ++kb) {
                    mbar_wait(&empty_bar[stage], phase ^ 1u);
                    mbar_arrive_expect_tx(&full_bar[stage], Cfg::STAGE_BYTES);
                    uint8_t *sA = smem + stage * Cfg::STAGE_BYTES;
                    uint8_t *sB = sA + Cfg::A_BYTES;
                    const int k0 = kb * Cfg::BK;
#pragma unroll
                    for (int w = 0; w < Cfg::NCW; ++w)
#pragma unroll
                        for (int c = 0; c < Cfg::CPG; ++c)
                            tma_load_4d(sA + (w * Cfg::CPG + c) * Cfg::CHUNK_BYTES, &mapA, &full_bar[stage],
                                        m0 + 16 * c, g0 + w, k0, ba);
#pragma unroll
                    for (int c = 0; c < Cfg::CPG; ++c)
                        tma_load_3d(sB + c * Cfg::CHUNK_BYTES, &mapB, &full_bar[stage], 16 * c, k0, bb);
                    if (++stage == Cfg::STAGES) {
                        stage = 0;
                        phase ^= 1u;
                    }
                }
            }
        }
        return;
    }
    asm volatile("setmaxnreg.inc.sync.aligned.u32 232;");
    // ---- DMMA consumers: warp w owns group g0 + w of the tile
    const int g = lane >> 2, t = lane & 3;
    uint32_t x[2][2];                                        // swizzled in-chunk offsets, as in dgemm_tn.cu
#pragma unroll
    for (int h = 0; h < 2; ++h)
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const uint32_t krow = 2 * t + j;
            x[h][j] = krow * 128u + ((((uint32_t)(h * 8 + g)) * 8u) ^ (krow << 4));
        }
    const uint32_t a_warp_off = (uint32_t)(warp * Cfg::CPG) * Cfg::CHUNK_BYTES;
    constexpr int MT = Cfg::MT;
    constexpr int SUB = Cfg::BK / 4;

    uint32_t it = 0;
    for (uint32_t tile = blockIdx.x; tile < (uint32_t)total_tiles; tile += gridDim.x) {
        double acc[MT][MT][2];                               // only ni <= mi is ever touched
#pragma unroll
        for (int mi = 0; mi < MT; ++mi)
#pragma unroll
            for (int ni = 0; ni <= mi; ++ni) acc[mi][ni][0] = acc[mi][ni][1] = 0.0;
        double a[2][MT], bf[2][MT];
        uint32_t loaded = 0, loaded_next = 0;
        auto load_frags = [&](int buf, uint32_t st, int sub, uint32_t &lx) {
            const uint32_t sbase = smem_base + st * Cfg::STAGE_BYTES;
            const uint32_t abase = sbase + a_warp_off, bbase = sbase + Cfg::A_BYTES;
            const int kk = sub >> 1, j = sub & 1;
#pragma unroll
            for (int mi = 0; mi < MT; ++mi)
                a[buf][mi] = lds_f64(abase + (mi >> 1) * Cfg::CHUNK_BYTES + kk * 1024 + x[mi & 1][j]);
#pragma unroll
            for (int ni = 0; ni < MT; ++ni)
                bf[buf][ni] = lds_f64(bbase + (ni >> 1) * Cfg::CHUNK_BYTES + kk * 1024 + x[ni & 1][j]);
#pragma unroll
            for (int mi = 0; mi < MT; ++mi) lx ^= (uint32_t)__double2hiint(a[buf][mi]);
#pragma unroll
            for (int ni = 0; ni < MT; ++ni) lx ^= (uint32_t)__double2hiint(bf[buf][ni]);
        };
        {
            const uint32_t stage = it & (Cfg::STAGES - 1);
            mbar_wait(&full_bar[stage], (it / Cfg::STAGES) & 1u);
            load_frags(0, stage, 0, loaded);
        }
        // one k-block; LAST: no next stage to prefetch, 8-row atoms entirely past K skipped (as in dgemm_tn.cu)
        auto kblock = [&](auto last_tag) {
            constexpr bool LAST = decltype(last_tag)::value;
            const uint32_t stage = it & (Cfg::STAGES - 1);
#pragma unroll
            for (int sub = 0; sub < SUB; ++sub) {
                const int cur = sub & 1, nxt = cur ^ 1;
                if (sub + 1 < SUB) {
                    load_frags(nxt, stage, sub + 1, loaded);
                } else if (!LAST) {
                    const uint32_t nstage = (it + 1) & (Cfg::STAGES - 1);
                    mbar_wait(&full_bar[nstage], ((it + 1) / Cfg::STAGES) & 1u);
                    load_frags(nxt, nstage, 0, loaded_next);
                }
                if (!LAST || sub < args.last_subs) {
#pragma unroll
                    for (int mi = 0; mi < MT; ++mi)
#pragma unroll
                        for (int ni = 0; ni <= mi; ++ni)     // the diagonal and below: columns n <= 8 mi + 7
                            dmma884(acc[mi][ni][0], acc[mi][ni][1], a[cur][mi], bf[cur][ni]);
                }
            }
            if (lane == 0) mbar_arrive_addr(smem_u32(&empty_bar[stage]) + (loaded & args.zero));
            loaded = loaded_next;
            loaded_next = 0;
            ++it;
        };
        for (int kb = 0; kb + 1 < args.kblocks; ++kb) kblock(FalseTag{});
        kblock(TrueTag{});

        // ---- epilogue: P[g'][m(m+1)/2 + n] for n <= m < nclass
        const int b = (int)(tile / (uint32_t)args.tiles_per_batch);
        const int u = (int)(tile - (uint32_t)b * (uint32_t)args.tiles_per_batch);
        const int64_t grp = (int64_t)(u / args.halves) * Cfg::NCW + warp;
        if (grp >= args.ngroups) continue;
        double *row0 = nullptr, *row1 = nullptr;
        double *base = args.P + (int64_t)(b * args.halves + u % args.halves) * args.strideP;
        if (args.tri_rows) {
            const int64_t pq = grp + args.group_offset;
            int p = (int)((sqrt(8.0 * (double)pq + 1.0) - 1.0) * 0.5);
            while ((int64_t)(p + 1) * (p + 2) / 2 <= pq) ++p;
            while ((int64_t)p * (p + 1) / 2 > pq) --p;
            const int q = (int)(pq - (int64_t)p * (p + 1) / 2);
            if (p >= args.dorb) continue;                    // padding of the pair index
            row0 = base + ((int64_t)p * args.dorb + q) * args.npair_ld;
            row1 = base + ((int64_t)q * args.dorb + p) * args.npair_ld;
        } else {
            row0 = row1 = base + grp * args.npair_ld;
        }
#pragma unroll
        for (int mi = 0; mi < MT; ++mi) {
            const int m = mi * 8 + g;
            if (m >= args.nclass) continue;
            const int64_t off = (int64_t)m * (m + 1) / 2;
#pragma unroll
            for (int ni = 0; ni <= mi; ++ni)
#pragma unroll
                for (int c = 0; c < 2; ++c) {
                    const int n = ni * 8 + 2 * t + c;
                    if (n <= m) {
                        row0[off + n] = acc[mi][ni][c];
                        if (row1 != row0) row1[off + n] = acc[mi][ni][c];
                    }
                }
        }
    }
}

template <class Cfg>
int launch_tri(const double *At, const double *B, double *P, int tri_rows, int nclass, int dorb, int64_t ngroups,
               int64_t npair_ld, int64_t K, int64_t lda, int64_t ldb, int batch, int64_t strideA, int64_t strideB,
               int64_t strideP, cudaStream_t stream, int64_t group_offset, int64_t group_ld, int halves) {
    CUtensorMap mapA, mapB;
    const int a_batched = (batch > 1 && strideA != 0);
    const int b_batched = ((batch > 1 || halves > 1) && strideB != 0);
    // (halves = 2: the innermost extent is the whole paired row, of which a tile reads the columns of its half)
    const uint64_t dimsA[4] = {(uint64_t)(halves > 1 ? group_ld : nclass), (uint64_t)ngroups, (uint64_t)K,
                               (uint64_t)(a_batched ? batch : 1)};
    const uint64_t strA[3] = {(uint64_t)group_ld, (uint64_t)lda, (uint64_t)(a_batched ? strideA : lda * K)};
    const uint32_t boxA[4] = {16, 1, (uint32_t)Cfg::BK, 1};
    int rc = encode_tmap_4d_f64(&mapA, At, dimsA, strA, boxA);
    if (rc) return rc;
    rc = encode_tmap_3d_f64(&mapB, B, (uint64_t)nclass, (uint64_t)K, b_batched ? batch * halves : 1, (uint64_t)ldb,
                            b_batched ? (uint64_t)strideB : (uint64_t)ldb * K, 16, Cfg::BK);
    if (rc) return rc;
    TriArgs args;
    args.P = P;
    args.npair_ld = npair_ld;
    args.strideP = strideP;
    args.nclass = nclass;
    args.tri_rows = tri_rows;
    args.dorb = dorb;
    args.ngroups = ngroups;
    args.group_offset = group_offset;
    args.kblocks = (int)ceil_div(K, Cfg::BK);
    args.tiles_per_batch = (int)ceil_div(ngroups, Cfg::NCW) * halves;
    args.batch = batch;
    args.halves = halves;
    args.a_batched = a_batched;
    args.b_batched = b_batched;
    args.last_subs = 2 * (int)ceil_div(K - (int64_t)(args.kblocks - 1) * Cfg::BK, 8);
    args.zero = 0;
    static unsigned long long attr_set = 0;
    if (once_per_device(attr_set))
        OO_CUDA_CHECK(cudaFuncSetAttribute(dgemm_tn_tri_kernel<Cfg>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           Cfg::SMEM_BYTES));
    const int64_t total = (int64_t)args.tiles_per_batch * batch;
    const int grid = (int)(total < sm_count() ? total : sm_count());
    dgemm_tn_tri_kernel<Cfg><<<grid, Cfg::THREADS, Cfg::SMEM_BYTES, stream>>>(mapA, mapB, args);
    OO_LAUNCH_CHECK();
    return OO_OK;
}

}  // namespace

// true when the triangular kernel covers this class count (otherwise the caller uses dgemm_tn_class_pack)
bool dgemm_tn_tri_supported(int nclass) { return nclass > 16 && nclass <= 48 && (nclass % 2) == 0; }

// X[(g, m), n] = sum_k At[k, (g m)] B[k, n] for n <= m only, stored as P[g'][m(m+1)/2 + n] (rows of npair_ld doubles).
// At: K x (ngroups * nclass), leading dimension lda (= ngroups * nclass rows back to back), B: K x nclass (ldb).
// tri_rows: g = p(p+1)/2 + q is a packed pair of `dorb` orbitals and both P[(p q)] and P[(q p)] are written.
// group_ld > nclass: the groups lie group_ld doubles apart (a column slice of a wider quarter-1 result).
// halves = 2 (group_ld >= 2 nclass): every group row holds two evaluations side by side; batch counts such PAIRS
// (strideA between pairs), B and P hold 2 batch matrices (strideB, strideP between consecutive evaluations).
int dgemm_tn_tri_class_pack(const double *At, const double *B, double *P, int tri_rows, int nclass, int dorb,
                            int64_t ngroups, int64_t npair_ld, int64_t K, int64_t lda, int64_t ldb, int batch,
                            int64_t strideA, int64_t strideB, int64_t strideP, cudaStream_t stream,
                            int64_t group_offset, int64_t group_ld, int halves) {
    OO_REQUIRE(At && B && P && nclass > 0 && ngroups > 0 && K > 0 && batch > 0 && dorb > 0);
    if (group_ld == 0) group_ld = nclass;
    OO_REQUIRE((halves == 1 || halves == 2) && group_ld >= (int64_t)halves * nclass && (group_ld % 2) == 0);
    OO_REQUIRE(lda >= (ngroups - 1) * group_ld + (int64_t)halves * nclass);
    OO_REQUIRE(dgemm_tn_tri_supported(nclass) && npair_ld >= (int64_t)nclass * (nclass + 1) / 2);
    OO_REQUIRE((lda % 2) == 0 && (ldb % 2) == 0 && (strideA % 2) == 0 && (strideB % 2) == 0);
    OO_REQUIRE(((uintptr_t)At % 16) == 0 && ((uintptr_t)B % 16) == 0);
    if (ngroups * halves >= (1ll << 31) || K >= (1ll << 31)) return OO_ERR_UNSUPPORTED;
#define OO_TRI(GP, MTC)                                                                                              \
    return launch_tri<TriCfg<GP, MTC, 4>>(At, B, P, tri_rows, nclass, dorb, ngroups, npair_ld, K, lda, ldb, batch, strideA, \
                                          strideB, strideP, stream, group_offset, group_ld, halves)
    if (nclass <= 24) OO_TRI(32, 3);
    if (nclass <= 32) OO_TRI(32, 4);
    if (nclass <= 40) OO_TRI(48, 5);
    OO_TRI(48, 6);
#undef OO_TRI
}

}  // namespace oo
