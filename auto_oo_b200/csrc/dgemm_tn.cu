// TN DGEMM for sm_100a:  C[b][m][n] = sum_k At[b][k][m] * B[b][k][n]
//
// This is the dense contraction behind the four-index transform
// (reference oo_energy.py:26-29, one launch per quarter) and the Hessian
// Y-matrix (oo_energy.py:390-392).  Both operands are K-major with the free
// index contiguous, so both are fetched by the same TMA path:
//   * cp.async.bulk.tensor 3-D boxes of [BK k-rows][16 doubles] with 128-byte
//     swizzle, landing in a STAGES-deep shared-memory ring guarded by
//     full/empty mbarriers (one producer warp, NCW consumer warps);
//   * consumers issue FP64 tensor-core MMAs (mma.sync m8n8k4 -> DMMA.8x8x4;
//     tcgen05 has no f64 kind).  Within a k8 step lane (g,t) takes k = 2t and
//     k = 2t+1 for its two MMAs; with the 128B swizzle that makes every
//     fragment load (LDS.64) bank-conflict free;
//   * persistent CTAs (one per SM) walk the tile list with n-tiles adjacent so
//     the A tile shared by neighbouring n-tiles is served from L2; the producer
//     runs ahead into the next tile while consumers store the finished one.
// OOB rows/cols/k are zero-filled by TMA, so M, N, K need no alignment; only the
// leading dimensions must be even (16-byte global strides).
#include "common.cuh"

namespace oo {

// NTC_ > 0: only the first NTC_ 8-column MMA tiles of the (single) warp column are computed and stored -- the
// 24- and 40-column variants of the 32- and 48-wide tiles (the TMA boxes still fetch 16-column chunks of B).
template <int BM_, int BN_, int BK_, int WGM_, int WGN_, int STAGES_, int NTC_ = 0>
struct TnCfg {
    static constexpr int BM = BM_, BN = BN_, BK = BK_, WGM = WGM_, WGN = WGN_, STAGES = STAGES_;
    static constexpr int NCW = WGM * WGN;            // consumer warps (two warpgroups)
    static constexpr int THREADS = (NCW + 4) * 32;   // + one producer warpgroup (its first warp issues TMA)
    static_assert(NCW == 8, "register re-allocation below assumes 2 consumer warpgroups + 1 producer warpgroup");
    static constexpr int WTM = BM / WGM, WTN = BN / WGN;
    static constexpr int MT = WTM / 8, NT = NTC_ ? NTC_ : WTN / 8;
    static_assert(NTC_ == 0 || (WGN_ == 1 && NTC_ * 8 <= WTN), "a trimmed warp tile needs a single warp column");
    static constexpr int CHUNK_BYTES = BK * 128;     // one TMA box: [BK][16 doubles]
    static constexpr int A_BYTES = (BM / 16) * CHUNK_BYTES;
    static constexpr int B_BYTES = (BN / 16) * CHUNK_BYTES;
    static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
    static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 2 * STAGES * 8 + 1024;
    // "linear A" stages (AMODE 1 below): BK rows of BM doubles, each fetched by ONE bulk copy from an arbitrary
    // global address, row pitch BM*8 + 16 bytes.  The pitch is 4 banks mod 32, which makes the fragment loads
    // (lane (g,t): k = 2t + j, row 8 mi + g) conflict free without any swizzle.
    static constexpr int LIN_PITCH = BM * 8 + 16;
    static constexpr int LIN_A_BYTES = (BK * LIN_PITCH + 1023) / 1024 * 1024;      // B chunks stay 1024-aligned
    static constexpr int LIN_STAGE_BYTES = LIN_A_BYTES + B_BYTES;
    static constexpr int LIN_SMEM_BYTES = STAGES * LIN_STAGE_BYTES + 2 * STAGES * 8 + 1024;
    // EPI 1 (below): a three-stage ring leaves room for one BM x BN result tile in shared memory
    static constexpr int EPI_STAGES = 3;
    static constexpr int EPI_TILE_BYTES = BM * BN * 8;
    static constexpr int EPI_SMEM_BYTES = EPI_STAGES * LIN_STAGE_BYTES + EPI_TILE_BYTES + 2 * EPI_STAGES * 8 + 1024;
    // the same for the TMA-fed kernel (plain and class-expand stores): tile rows padded by 16 bytes so that the
    // shipping warps can also read it column-wise (transposed mirror) with 4-way instead of 32-way bank conflicts;
    // as many stages as fit next to it (two for the 128 x 128 tile: a k-block is 4096 clocks of DMMA, one stage
    // in flight covers the memory latency)
    static constexpr int EPI0_PITCH = BN * 8 + 16;
    static constexpr int EPI0_TILE_BYTES = BM * EPI0_PITCH;
    static constexpr int EPI0_STAGES = (227 * 1024 - 1024 - 64 - EPI0_TILE_BYTES) / STAGE_BYTES >= 4 ? 4
                                       : (227 * 1024 - 1024 - 64 - EPI0_TILE_BYTES) / STAGE_BYTES;
    static constexpr int EPI0_SMEM_BYTES = EPI0_STAGES * STAGE_BYTES + EPI0_TILE_BYTES + 2 * 4 * 8 + 1024;
    static_assert(WTM % 16 == 0 && WTN % 16 == 0, "warp tile must cover whole 16-wide chunks");
    static_assert(BK % 8 == 0, "BK must be a multiple of 8");
    static_assert((BK / 4) % 2 == 0, "the substep double buffer assumes an even number of substeps per k-block");
    static_assert(CHUNK_BYTES % 1024 == 0, "chunks must keep the 1024B swizzle alignment");
};

struct TnArgs {
    double *C;
    // optional second copy of the result with rows permuted (a b c) -> (c b a), M = d0*d1*d2
    // (classes.cu: T1[s,p,q,m] and T1t[q,p,s,m] from the same accumulators, no separate swap pass)
    // or (mode 2, symmetric class transform) rows (a, pq) with pq = p(p+1)/2 + q a packed lower-triangular
    // pair of d1 orbitals (d2 = padded pair count): C2 receives the value at rows (q p a) AND (p q a)
    // or (modes 3 / 4, class-pair packing; C itself is NOT written) rows (r2, m) with m < d0 a class index and
    // columns n: only n <= m is kept, at C2[r2'][m(m+1)/2 + n] with row length d2 -- r2' = r2 (mode 4), or
    // both (p q) and (q p) of the packed pair r2 = p(p+1)/2 + q of d1 orbitals (mode 3)
    // or (mode 5, class-pair expansion; C itself is NOT written) rows (mn, a), mn = m(m+1)/2 + n a packed class
    // pair of d0 indices, a < d1, columns b < N = d1: C2[(m n), a, b] always and, for m != n, C2[(n m), a, b]
    // (d2 == 0) or the transposed C2[(n m), b, a] (d2 != 0)
    double *C2;
    int d0, d1, d2;
    int64_t M, N;
    int64_t ldc, strideC, strideC2;
    int kblocks;
    int tiles_m, tiles_n, batch;
    int a_batched, b_batched;
    // AMODE 1 (quarter 1 over 8-fold packed AO integrals): A8[RS][PQ] with RS = r(r+1)/2 + s (r >= s) and PQ a packed
    // pair (row length d2); the tile (s, PQ-range) takes its k-row r from row RS(max(r,s), min(r,s)).  Rows of the
    // product are (s, PQ) as in mode 2 (d0 = number of s, d2 = padded pair count); K = number of r.
    const double *A8;
    int64_t strideA8;
    int K;
    // a SLAB of the pair columns (sharded evaluation: every rank holds A8[:, pq_lo : pq_lo + pq_cnt], row pitch a8_ld):
    // the tiles cover PQ in [pq_lo, pq_lo + pq_cnt) only; the whole tensor is pq_lo = 0, pq_cnt = a8_ld = d2
    int pq_lo, pq_cnt;
    int64_t a8_ld;
    // mode 3 (tri_rows): the row groups are the packed pairs r2_offset + r2 (a slab of the quarter-1 result)
    int64_t r2_offset;
    // staged mode 5, Coulomb class: every d1 x d1 result block is symmetric, J[mn][a][b] = J[mn][b][a].  sym_T > 0
    // (= d1 / BM tiles per side) walks only the tiles on and below the block diagonal -- sym_T (sym_T + 1) / 2 per
    // block instead of sym_T^2 -- and the shipping warps also write the transpose of every off-diagonal tile.
    int sym_T, sym_tiles_per_batch;
    int last_subs;   // k4-substeps of the LAST k-block that hold rows below K (whole 8-row atoms beyond K are skipped)
    // Always 0, but opaque to the compiler: ANDed with bits of every fragment a consumer loaded from
    // a stage and added to the address of that stage's "empty" arrive.  The arrive thus has a true
    // register dependency on the LDS results, so it cannot be issued while a shared-memory load of
    // the stage is still in flight (an in-flight LDS is NOT ordered against the TMA refill that the
    // arrive releases; without this, ptxas schedules the arrive ahead of the last loads' consumers
    // and a stage was seen overwritten under a pending read).
    uint32_t zero;
};

// shared -> global bulk asynchronous copy (TMA store path; tracked by the issuing thread's bulk group)
__device__ __forceinline__ void bulk_store_1d(void *gdst, uint32_t smem_src, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(smem_src), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ void named_bar_arrive(int id, int nthreads) {
    asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

__device__ __forceinline__ void bulk_load_1d(uint32_t smem_dst, const void *gsrc, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_dst),
                 "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// DUAL: 0 = plain store, 1 = second store with rows (a b c) -> (c b a), 2 = packed-pair unpack,
// 3 / 4 = class-pair packing, 5 = class-pair expansion instead of the plain store (see TnArgs)
// AMODE: 0 = A through the tensor map (K-major matrix), 1 = A rows gathered from the 8-fold packed AO integrals
// EPI:   0 = the consumer warps store their accumulators to global memory themselves;
//        1 = (DUAL 2, AMODE 1: quarter 1) they drop the tile into shared memory (24 STS.128 per thread) and go
//            straight on to the next tile, while a warp of the producer warpgroup ships it with bulk asynchronous
//            copies (cp.async.bulk shared -> global): ONE copy for the contiguous packed rows, one per row and order
//            for the pair-unpacked rows.  The 288 KB of stores per tile then cost the tensor pipe nothing.
template <class Cfg, int DUAL, int AMODE = 0, int EPI = 0>
__global__ void __launch_bounds__(Cfg::THREADS, 1)
dgemm_tn_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB,
                const TnArgs args) {
    static_assert(EPI == 0 || (DUAL == 2 && AMODE == 1) || (AMODE == 0 && (DUAL == 0 || DUAL == 5)),
                  "the staged epilogue exists for quarter 1 and for the plain / class-expand stores");
    constexpr int STAGE_BYTES = AMODE ? Cfg::LIN_STAGE_BYTES : Cfg::STAGE_BYTES;
    constexpr int A_BYTES = AMODE ? Cfg::LIN_A_BYTES : Cfg::A_BYTES;
    constexpr int NST = !EPI ? Cfg::STAGES : (AMODE ? Cfg::EPI_STAGES : (Cfg::EPI0_STAGES > 0 ? Cfg::EPI0_STAGES : 1));
    constexpr int kShipWarps = 3;                        // the spare warps of the producer warpgroup ship the tile
    constexpr int kBarFree = 1, kBarFull = 2, kBarThreads = (Cfg::NCW + kShipWarps) * 32;   // consumers + shippers
    constexpr int TILE_BYTES = AMODE ? Cfg::EPI_TILE_BYTES : Cfg::EPI0_TILE_BYTES;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t *smem = smem_raw + (smem_base - smem_u32(smem_raw));
    const uint32_t ctile = smem_base + NST * STAGE_BYTES;                           // EPI 1: the result tile
    uint64_t *full_bar = reinterpret_cast<uint64_t *>(smem + NST * STAGE_BYTES + (EPI ? TILE_BYTES : 0));
    uint64_t *empty_bar = full_bar + NST;

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
#pragma unroll
        for (int s = 0; s < NST; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], Cfg::NCW);
        }
        fence_barrier_init();
        if (!AMODE) tma_prefetch_desc(&mapA);
        tma_prefetch_desc(&mapB);
    }
    __syncthreads();

    const bool sym = DUAL == 5 && EPI && args.sym_T > 0;
    const int tiles_per_batch = sym ? args.sym_tiles_per_batch : args.tiles_m * args.tiles_n;
    const int64_t total_tiles = (int64_t)tiles_per_batch * args.batch;
    // tile number within a batch entry -> (m-tile, n-tile); `offdiag`: a tile below the diagonal of a symmetric block
    auto tile_mn = [&](int rem, int &mt, int &nt, bool &offdiag) {
        offdiag = false;
        if (sym) {
            const int TT = args.sym_T * (args.sym_T + 1) / 2;
            const int blk = rem / TT, k = rem - blk * TT;
            int ta = (int)((sqrtf(8.0f * (float)k + 1.0f) - 1.0f) * 0.5f);
            while ((ta + 1) * (ta + 2) / 2 <= k) ++ta;
            while (ta * (ta + 1) / 2 > k) --ta;
            nt = k - ta * (ta + 1) / 2;
            mt = blk * args.sym_T + ta;
            offdiag = nt != ta;
        } else {
            mt = rem / args.tiles_n;
            nt = rem - mt * args.tiles_n;
        }
    };
    // AMODE 1 walks the m-tiles as (PQ-tile outer, s inner): the CTAs that run together share one PQ panel of
    // A8, and every row RS(r, s) of that panel is needed twice -- by tile s at step r and by tile r at step s --
    // so the second use is served from L2 (the 8-fold packed tensor is read from HBM about once).
    auto lin_tile = [&](int mt, int &s, int &pq0) {      // pq0: offset inside the slab
        s = mt % args.d0;
        pq0 = (mt / args.d0) * Cfg::BM;
    };

    // Register re-allocation (setmaxnreg): the CTA starts with 168 registers per thread (384 threads,
    // three warps per SM sub-partition); the producer warpgroup gives most of its share back and the
    // two consumer warpgroups grow to 232, which holds the 128 accumulator registers of the 64x32 /
    // 32x48 warp tiles plus fragments and addressing without spilling.
    if (warp >= Cfg::NCW) {
        // (the shipping warps of the staged epilogue do address arithmetic a 40-register budget makes ptxas spill:
        //  64 / 216 there.  The registers the consumers gain must not exceed what this warpgroup gives back --
        //  128 x (168 - 64) >= 256 x (216 - 168) -- or setmaxnreg.inc waits for ever.)
        static_assert(128 * (168 - 64) >= 256 * (216 - 168) && 128 * (168 - 40) >= 256 * (232 - 168),
                      "setmaxnreg.inc would wait for registers the producer warpgroup never releases");
        if (EPI) asm volatile("setmaxnreg.dec.sync.aligned.u32 64;");
        else asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
        // ===================== TMA producer =====================
        if (AMODE && warp == Cfg::NCW) {
            // linear-A producer: the whole warp takes part, lane k issues the bulk copy of k-row k
            int stage = 0;
            uint32_t phase = 0;
            for (int64_t tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
                const int b = (int)(tile / tiles_per_batch);
                const int rem = (int)(tile - (int64_t)b * tiles_per_batch);
                int s, pq0;
                lin_tile(rem / args.tiles_n, s, pq0);
                const int n0 = (rem % args.tiles_n) * Cfg::BN;
                const int bb = args.b_batched ? b : 0;
                const int rows = (args.pq_cnt - pq0) < Cfg::BM ? (args.pq_cnt - pq0) : Cfg::BM;   // even: pq_cnt, BM are
                const uint32_t row_bytes = (uint32_t)rows * 8u;
                const double *Ab = args.A8 + (int64_t)b * args.strideA8 + pq0;
                for (int kb = 0; kb < args.kblocks; ++kb) {
                    if (lane == 0) {
                        mbar_wait(&empty_bar[stage], phase ^ 1u);
                        mbar_arrive_expect_tx(&full_bar[stage], Cfg::BK * row_bytes + Cfg::B_BYTES);
                    }
                    __syncwarp();
                    const uint32_t sA = smem_base + stage * STAGE_BYTES;
                    const int k0 = kb * Cfg::BK;
                    if (lane < Cfg::BK) {
                        int r = k0 + lane;
                        r = r < args.K ? r : args.K - 1;         // rows past K meet zero rows of B (TMA fill)
                        const int hi = r > s ? r : s, lo = r > s ? s : r;
                        const double *src = Ab + ((int64_t)hi * (hi + 1) / 2 + lo) * args.a8_ld;
                        bulk_load_1d(sA + lane * Cfg::LIN_PITCH, src, row_bytes, &full_bar[stage]);
                    }
                    if (lane == 0) {
                        uint8_t *sB = smem + stage * STAGE_BYTES + A_BYTES;
#pragma unroll
                        for (int c = 0; c < Cfg::BN / 16; ++c)
                            tma_load_3d(sB + c * Cfg::CHUNK_BYTES, &mapB, &full_bar[stage], n0 + 16 * c, k0, bb);
                    }
                    if (++stage == NST) {
                        stage = 0;
                        phase ^= 1u;
                    }
                }
            }
        } else if (EPI && !AMODE && warp > Cfg::NCW) {
            // ===================== shipping warps, plain / class-expand stores (EPI 1) =====================
            // warp NCW+1 issues one bulk copy per tile row (and per mirror row of the Coulomb class); the transposed
            // mirror of the exchange class, K[n,m][b][a] = K[m,n][a][b], is read column-wise from the tile by all
            // three warps and written with coalesced stores.
            const int sw = warp - Cfg::NCW - 1;                      // 0, 1, 2
            named_bar_arrive(kBarFree, kBarThreads);                // the tile buffer starts out free
            for (int64_t tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
                const int b = (int)(tile / tiles_per_batch);
                const int rem = (int)(tile - (int64_t)b * tiles_per_batch);
                int mt, nt;
                bool offdiag;
                tile_mn(rem, mt, nt, offdiag);
                const int64_t m0 = (int64_t)mt * Cfg::BM;
                const int n0 = nt * Cfg::BN;
                const int rows = (args.M - m0) < Cfg::BM ? (int)(args.M - m0) : Cfg::BM;
                const int ncols = (args.N - n0) < Cfg::BN ? (int)(args.N - n0) : Cfg::BN;   // even (N and BN are)
                named_bar_sync(kBarFull, kBarThreads);
                if (DUAL == 0) {
                    if (sw == 0) {
                        double *Cb = args.C + (int64_t)b * args.strideC + n0;
                        for (int r = lane; r < rows; r += 32)
                            bulk_store_1d(Cb + (m0 + r) * args.ldc, ctile + (uint32_t)r * Cfg::EPI0_PITCH, (uint32_t)ncols * 8u);
                    }
                } else {
                    double *base2 = args.C2 + (int64_t)b * args.strideC2;
                    const int64_t plane = (int64_t)args.d1 * args.ldc;
                    const bool transposed = args.d2 != 0;
                    for (int r = lane; r < rows; r += 32) {
                        const int64_t row = m0 + r;
                        const int a = (int)(row % args.d1);
                        const int mn = (int)(row / args.d1);
                        int m = (int)((sqrtf(8.0f * (float)mn + 1.0f) - 1.0f) * 0.5f);
                        while ((m + 1) * (m + 2) / 2 <= mn) ++m;
                        while (m * (m + 1) / 2 > mn) --m;
                        const int n = mn - m * (m + 1) / 2;
                        if (m >= args.d0) continue;                  // padding of the pair index
                        const uint32_t src = ctile + (uint32_t)r * Cfg::EPI0_PITCH;
                        if (sw == 0) {
                            bulk_store_1d(base2 + ((int64_t)m * args.d0 + n) * plane + (int64_t)a * args.ldc + n0, src,
                                          (uint32_t)ncols * 8u);
                            if (m != n && !transposed)
                                bulk_store_1d(base2 + ((int64_t)n * args.d0 + m) * plane + (int64_t)a * args.ldc + n0, src,
                                              (uint32_t)ncols * 8u);
                        }
                        if (m != n && transposed) {                  // lanes = consecutive a: coalesced rows of the mirror
                            double *mir = base2 + ((int64_t)n * args.d0 + m) * plane + a;
                            for (int c = sw; c < ncols; c += kShipWarps)
                                mir[(int64_t)(n0 + c) * args.ldc] = lds_f64(src + (uint32_t)c * 8u);
                        }
                        if (offdiag) {                               // symmetric block: the tile above the diagonal
                            double *t1 = base2 + ((int64_t)m * args.d0 + n) * plane + a;
                            double *t2 = base2 + ((int64_t)n * args.d0 + m) * plane + a;
                            for (int c = sw; c < ncols; c += kShipWarps) {
                                const double v = lds_f64(src + (uint32_t)c * 8u);
                                t1[(int64_t)(n0 + c) * args.ldc] = v;
                                if (m != n) t2[(int64_t)(n0 + c) * args.ldc] = v;
                            }
                        }
                    }
                }
                if (sw == 0) {
                    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                    asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                }
                __syncwarp();
                named_bar_arrive(kBarFree, kBarThreads);
            }
            if (sw == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
        } else if (EPI && AMODE && warp > Cfg::NCW) {
            // ===================== shipping warps, quarter 1 (EPI 1) =====================
            // (three of them: with a short K -- 114 orbitals are 8 k-blocks -- the 500 bulk copies of a tile would
            //  take one warp longer than the tile's DMMAs)
            const int sw = warp - Cfg::NCW - 1;
            const uint32_t pitch = (uint32_t)args.N * 8u;            // tile rows hold the N valid columns, dense
            named_bar_arrive(kBarFree, kBarThreads);                // the tile buffer starts out free
            for (int64_t tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
                const int b = (int)(tile / tiles_per_batch);
                const int rem = (int)(tile - (int64_t)b * tiles_per_batch);
                int s, pq0;
                lin_tile(rem / args.tiles_n, s, pq0);
                const int rows = (args.pq_cnt - pq0) < Cfg::BM ? (args.pq_cnt - pq0) : Cfg::BM;
                const int pq_first = args.pq_lo + pq0;
                named_bar_sync(kBarFull, kBarThreads);              // consumers have written (and fenced) the tile
                if (sw == 0 && lane == 0)                            // packed rows (s, PQ): one contiguous run
                    bulk_store_1d(args.C + (int64_t)b * args.strideC + ((int64_t)s * args.d2 + pq_first) * args.ldc, ctile,
                                  (uint32_t)rows * pitch);
                double *base2 = args.C2 + (int64_t)b * args.strideC2;
                for (int r = sw * 32 + lane; r < rows; r += 32 * kShipWarps) {
                    const int pq = pq_first + r;
                    int p = (int)((sqrtf(8.0f * (float)pq + 1.0f) - 1.0f) * 0.5f);
                    while ((p + 1) * (p + 2) / 2 <= pq) ++p;
                    while (p * (p + 1) / 2 > pq) --p;
                    const int q = pq - p * (p + 1) / 2;
                    if (p >= args.d1) continue;                      // padding of the pair index
                    const uint32_t src = ctile + (uint32_t)r * pitch;
                    bulk_store_1d(base2 + (((int64_t)q * args.d1 + p) * args.d0 + s) * args.ldc, src, pitch);
                    if (p != q) bulk_store_1d(base2 + (((int64_t)p * args.d1 + q) * args.d0 + s) * args.ldc, src, pitch);
                }
                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // shared memory has been read
                __syncwarp();
                named_bar_arrive(kBarFree, kBarThreads);
            }
            asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
        } else if (warp == Cfg::NCW && lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            for (int64_t tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
                const int b = (int)(tile / tiles_per_batch);
                const int rem = (int)(tile - (int64_t)b * tiles_per_batch);
                int mt, nt;
                bool offdiag;
                tile_mn(rem, mt, nt, offdiag);
                const int m0 = mt * Cfg::BM;
                const int n0 = nt * Cfg::BN;
                const int ba = args.a_batched ? b : 0;
                const int bb = args.b_batched ? b : 0;
                for (int kb = 0; kb < args.kblocks; ++kb) {
                    mbar_wait(&empty_bar[stage], phase ^ 1u);
                    mbar_arrive_expect_tx(&full_bar[stage], Cfg::STAGE_BYTES);
                    uint8_t *sA = smem + stage * Cfg::STAGE_BYTES;
                    uint8_t *sB = sA + Cfg::A_BYTES;
                    const int k0 = kb * Cfg::BK;
#pragma unroll
                    for (int c = 0; c < Cfg::BM / 16; ++c)
                        tma_load_3d(sA + c * Cfg::CHUNK_BYTES, &mapA, &full_bar[stage], m0 + 16 * c, k0, ba);
#pragma unroll
                    for (int c = 0; c < Cfg::BN / 16; ++c)
                        tma_load_3d(sB + c * Cfg::CHUNK_BYTES, &mapB, &full_bar[stage], n0 + 16 * c, k0, bb);
                    if (++stage == NST) {
                        stage = 0;
                        phase ^= 1u;
                    }
                }
            }
        }
    } else {
        if (EPI) asm volatile("setmaxnreg.inc.sync.aligned.u32 216;");
        else asm volatile("setmaxnreg.inc.sync.aligned.u32 232;");
        // ===================== DMMA consumers =====================
        const int g = lane >> 2, t = lane & 3;
        const int wm = warp / Cfg::WGN, wn = warp % Cfg::WGN;
        // swizzled in-chunk byte offsets: x[h][j], h = which 8-column half of the
        // 16-wide chunk, j = which of the lane's two k rows (k = 2t + j)
        uint32_t x[2][2];
#pragma unroll
        for (int h = 0; h < 2; ++h)
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const uint32_t krow = 2 * t + j;
                x[h][j] = krow * 128u + ((((uint32_t)(h * 8 + g)) * 8u) ^ (krow << 4));
            }
        const uint32_t a_warp_off = AMODE ? (uint32_t)(wm * Cfg::WTM + g) * 8u + (uint32_t)(2 * t) * Cfg::LIN_PITCH
                                          : (uint32_t)(wm * Cfg::WTM / 16) * Cfg::CHUNK_BYTES;
        const uint32_t b_warp_off = A_BYTES + (uint32_t)(wn * Cfg::WTN / 16) * Cfg::CHUNK_BYTES;

        // registers are the scarce resource here (3 warps share one SM sub-partition's file: 168 per
        // thread): one running k-block counter carries both the ring slot and its phase, and the
        // tile coordinates are re-derived in the epilogue instead of living across the k loop.
        // `it % NST` / `it / NST`: NST is a compile-time constant (a mask and a shift for the power-of-two rings)
        uint32_t it = 0;
        for (uint32_t tile = blockIdx.x; tile < (uint32_t)total_tiles; tile += gridDim.x) {
            double acc[Cfg::MT][Cfg::NT][2];
#pragma unroll
            for (int mi = 0; mi < Cfg::MT; ++mi)
#pragma unroll
                for (int ni = 0; ni < Cfg::NT; ++ni) acc[mi][ni][0] = acc[mi][ni][1] = 0.0;

            // Software pipeline over the SUBSTEPS (4 k values each: kk = 8-row swizzle atom, j = k parity):
            // the fragments of substep s+1 -- or of the next k-block's first substep, after waiting for
            // its stage -- are requested before the DMMAs of substep s are issued, so shared-memory
            // latency hides behind MT*NT tensor instructions even across k-block boundaries.
            constexpr int SUB = Cfg::BK / 4;            // substeps per k-block
            double a[2][Cfg::MT], bf[2][Cfg::NT];
            uint32_t loaded = 0, loaded_next = 0;       // XOR of the high words read from the current / next stage
            auto load_frags = [&](int buf, uint32_t st, int sub, uint32_t &lx) {
                const uint32_t sbase = smem_base + st * STAGE_BYTES;
                const uint32_t abase = sbase + a_warp_off, bbase = sbase + b_warp_off;
                const int kk = sub >> 1, j = sub & 1;
#pragma unroll
                for (int mi = 0; mi < Cfg::MT; ++mi)
                    a[buf][mi] = AMODE ? lds_f64(abase + (kk * 8 + j) * Cfg::LIN_PITCH + mi * 64)
                                       : lds_f64(abase + (mi >> 1) * Cfg::CHUNK_BYTES + kk * 1024 + x[mi & 1][j]);
#pragma unroll
                for (int ni = 0; ni < Cfg::NT; ++ni)
                    bf[buf][ni] = lds_f64(bbase + (ni >> 1) * Cfg::CHUNK_BYTES + kk * 1024 + x[ni & 1][j]);
#ifndef OO_TN_DIAG_NO_RELEASE_DEPENDENCY   /* diagnostic builds only: measures what the dependency costs */
#pragma unroll
                for (int mi = 0; mi < Cfg::MT; ++mi) lx ^= (uint32_t)__double2hiint(a[buf][mi]);
#pragma unroll
                for (int ni = 0; ni < Cfg::NT; ++ni) lx ^= (uint32_t)__double2hiint(bf[buf][ni]);
#endif
            };
            {
                const uint32_t stage = it % NST;
                mbar_wait(&full_bar[stage], (it / NST) & 1u);
                load_frags(0, stage, 0, loaded);
            }
            // One k-block.  LAST = the tile's final block: no next stage to prefetch from, and the 8-row atoms
            // that lie entirely past K (zero rows: nothing to add) are skipped -- 114 orbitals are 7 1/8 blocks.
            auto kblock = [&](auto last_tag) {
                constexpr bool LAST = decltype(last_tag)::value;
                const uint32_t stage = it % NST;
#pragma unroll
                for (int sub = 0; sub < SUB; ++sub) {
                    const int cur = sub & 1, nxt = cur ^ 1;
                    if (sub + 1 < SUB) {
                        load_frags(nxt, stage, sub + 1, loaded);
                    } else if (!LAST) {
                        const uint32_t nstage = (it + 1) % NST;
                        mbar_wait(&full_bar[nstage], ((it + 1) / NST) & 1u);
                        load_frags(nxt, nstage, 0, loaded_next);
                    }
                    if (!LAST || sub < args.last_subs) {
#pragma unroll
                        for (int mi = 0; mi < Cfg::MT; ++mi)
#pragma unroll
                            for (int ni = 0; ni < Cfg::NT; ++ni)
                                dmma884(acc[mi][ni][0], acc[mi][ni][1], a[cur][mi], bf[cur][ni]);
                    }
                }
                // release the stage only once every load from it has landed in registers (see TnArgs::zero)
                if (lane == 0) mbar_arrive_addr(smem_u32(&empty_bar[stage]) + (loaded & args.zero));
                loaded = loaded_next;
                loaded_next = 0;
                ++it;
            };
            for (int kb = 0; kb + 1 < args.kblocks; ++kb) kblock(FalseTag{});
            kblock(TrueTag{});

            if (EPI) {
                // staged epilogue: accumulators -> shared-memory tile, then on to the next tile.  Quarter 1: rows of
                // the N valid columns, dense (its packed rows leave as ONE bulk copy); otherwise rows of BN + 2
                const uint32_t pitch = AMODE ? (uint32_t)args.N * 8u : (uint32_t)Cfg::EPI0_PITCH;
                named_bar_sync(kBarFree, kBarThreads);              // the previous tile has been shipped
#pragma unroll
                for (int mi = 0; mi < Cfg::MT; ++mi) {
                    const uint32_t rowaddr = ctile + (uint32_t)(wm * Cfg::WTM + mi * 8 + g) * pitch;
#pragma unroll
                    for (int ni = 0; ni < Cfg::NT; ++ni) {
                        const int col = wn * Cfg::WTN + ni * 8 + 2 * t;
                        if (!AMODE || col + 1 < args.N)
                            asm volatile("st.shared.v2.f64 [%0], {%1, %2};" ::"r"(rowaddr + (uint32_t)col * 8u),
                                         "d"(acc[mi][ni][0]), "d"(acc[mi][ni][1])
                                         : "memory");
                    }
                }
                fence_proxy_async();                                // generic-proxy writes -> visible to the bulk copies
                named_bar_arrive(kBarFull, kBarThreads);
                continue;
            }
            // epilogue: registers -> global (16-byte stores, rows of 64 B per MMA tile)
            const int b = (int)(tile / (uint32_t)tiles_per_batch);
            const int rem = (int)(tile - (uint32_t)b * (uint32_t)tiles_per_batch);
            int64_t m0 = (int64_t)(rem / args.tiles_n) * Cfg::BM, m_end = args.M;
            if (AMODE) {                                   // rows (s, PQ) of one s: global row s * d2 + PQ
                int s, pq0;
                lin_tile(rem / args.tiles_n, s, pq0);
                m0 = (int64_t)s * args.d2 + args.pq_lo + pq0;
                m_end = (int64_t)s * args.d2 + args.pq_lo + args.pq_cnt;
            }
            const int n0 = (rem % args.tiles_n) * Cfg::BN;
            double *Cb = args.C + (int64_t)b * args.strideC;
#pragma unroll
            for (int mi = 0; mi < Cfg::MT; ++mi) {
                const int64_t row = m0 + wm * Cfg::WTM + mi * 8 + g;
                if (row < m_end) {
                    double *crow = Cb + row * args.ldc;
                    double *crow2 = nullptr, *crow3 = nullptr;
                    if (DUAL == 1) {
                        const int c = (int)(row % args.d2);
                        const int64_t ab = row / args.d2;
                        const int bq = (int)(ab % args.d1), a = (int)(ab / args.d1);
                        crow2 = args.C2 + (int64_t)b * args.strideC2 + (((int64_t)c * args.d1 + bq) * args.d0 + a) * args.ldc;
                    }
                    if (DUAL == 2) {
                        const int pq = (int)(row % args.d2);
                        const int a = (int)(row / args.d2);
                        int p = (int)((sqrt(8.0 * pq + 1.0) - 1.0) * 0.5);
                        while ((p + 1) * (p + 2) / 2 <= pq) ++p;
                        while (p * (p + 1) / 2 > pq) --p;
                        const int q = pq - p * (p + 1) / 2;
                        if (p < args.d1) {                     // (padding of the pair index: nothing to unpack)
                            double *base2 = args.C2 + (int64_t)b * args.strideC2;
                            crow2 = base2 + (((int64_t)q * args.d1 + p) * args.d0 + a) * args.ldc;
                            crow3 = base2 + (((int64_t)p * args.d1 + q) * args.d0 + a) * args.ldc;
                        }
                    }
                    if (DUAL == 5) {
                        const int a = (int)(row % args.d1);
                        const int mn = (int)(row / args.d1);
                        int m = (int)((sqrt(8.0 * mn + 1.0) - 1.0) * 0.5);
                        while ((m + 1) * (m + 2) / 2 <= mn) ++m;
                        while (m * (m + 1) / 2 > mn) --m;
                        const int n = mn - m * (m + 1) / 2;
                        if (m >= args.d0) continue;                          // padding of the pair index
                        double *base2 = args.C2 + (int64_t)b * args.strideC2;
                        const int64_t plane = (int64_t)args.d1 * args.ldc;
                        crow2 = base2 + ((int64_t)m * args.d0 + n) * plane + (int64_t)a * args.ldc;
                        double *mirror = base2 + ((int64_t)n * args.d0 + m) * plane;
                        const bool second = m != n, transposed = args.d2 != 0;
#pragma unroll
                        for (int ni = 0; ni < Cfg::NT; ++ni) {
                            const int col = n0 + wn * Cfg::WTN + ni * 8 + 2 * t;
#pragma unroll
                            for (int c = 0; c < 2; ++c) {
                                if (col + c >= args.N) continue;
                                const double v = acc[mi][ni][c];
                                crow2[col + c] = v;
                                if (second) {
                                    if (transposed) mirror[(int64_t)(col + c) * args.ldc + a] = v;
                                    else mirror[(int64_t)a * args.ldc + col + c] = v;
                                }
                            }
                        }
                        continue;
                    }
                    if (DUAL >= 3) {
                        const int m = (int)(row % args.d0);
                        const int64_t r2 = row / args.d0;
                        double *base2 = args.C2 + (int64_t)b * args.strideC2 + (int64_t)m * (m + 1) / 2;
                        if (DUAL == 4) {
                            crow2 = base2 + r2 * args.d2;
                        } else {
                            const int64_t pq = r2 + args.r2_offset;
                            int p = (int)((sqrt(8.0 * (double)pq + 1.0) - 1.0) * 0.5);
                            while ((int64_t)(p + 1) * (p + 2) / 2 <= pq) ++p;
                            while ((int64_t)p * (p + 1) / 2 > pq) --p;
                            const int q = (int)(pq - (int64_t)p * (p + 1) / 2);
                            if (p < args.d1) {
                                crow2 = base2 + ((int64_t)p * args.d1 + q) * args.d2;
                                crow3 = base2 + ((int64_t)q * args.d1 + p) * args.d2;
                            }
                        }
                        if (crow2) {
#pragma unroll
                            for (int ni = 0; ni < Cfg::NT; ++ni)
#pragma unroll
                                for (int c = 0; c < 2; ++c) {
                                    const int col = n0 + wn * Cfg::WTN + ni * 8 + 2 * t + c;
                                    if (col <= m && col < args.N) {
                                        crow2[col] = acc[mi][ni][c];
                                        if (DUAL == 3) crow3[col] = acc[mi][ni][c];
                                    }
                                }
                        }
                        continue;
                    }
#pragma unroll
                    for (int ni = 0; ni < Cfg::NT; ++ni) {
                        const int64_t col = (int64_t)n0 + wn * Cfg::WTN + ni * 8 + 2 * t;
                        if (col + 1 < args.N) {
                            const double2 v = make_double2(acc[mi][ni][0], acc[mi][ni][1]);
                            *reinterpret_cast<double2 *>(crow + col) = v;
                            if (DUAL == 1) *reinterpret_cast<double2 *>(crow2 + col) = v;
                            if (DUAL == 2 && crow2) {
                                *reinterpret_cast<double2 *>(crow2 + col) = v;
                                *reinterpret_cast<double2 *>(crow3 + col) = v;
                            }
                        } else if (col < args.N) {
                            crow[col] = acc[mi][ni][0];
                            if (DUAL == 1) crow2[col] = acc[mi][ni][0];
                            if (DUAL == 2 && crow2) crow2[col] = crow3[col] = acc[mi][ni][0];
                        }
                    }
                }
            }
        }
    }
}

struct TnDual {
    double *C2 = nullptr;
    int mode = 0;               // 1 = swap02, 2 = packed-pair unpack, 3 / 4 = class-pair packing (tri / plain rows), 5 = class-pair expansion
    int d0 = 0, d1 = 0, d2 = 0;
    int64_t strideC2 = 0;
    int64_t r2_offset = 0;
    bool direct_epilogue = false;   // true: consumer warps store to global memory themselves (A/B tests)
    bool symmetric_blocks = false;  // mode 5: every d1 x d1 result block is symmetric (Coulomb class)
};

template <class Cfg>
static int launch_tn(const double *At, const double *B, double *C, int64_t M, int64_t N, int64_t K,
                     int64_t lda, int64_t ldb, int64_t ldc, int batch, int64_t strideA,
                     int64_t strideB, int64_t strideC, cudaStream_t stream, const TnDual &dual = TnDual()) {
    CUtensorMap mapA, mapB;
    const int a_batched = (batch > 1 && strideA != 0);
    const int b_batched = (batch > 1 && strideB != 0);
    int rc = encode_tmap_3d_f64(&mapA, At, (uint64_t)M, (uint64_t)K, a_batched ? batch : 1,
                                (uint64_t)lda, a_batched ? (uint64_t)strideA : (uint64_t)lda * K, 16,
                                Cfg::BK);
    if (rc) return rc;
    rc = encode_tmap_3d_f64(&mapB, B, (uint64_t)N, (uint64_t)K, b_batched ? batch : 1, (uint64_t)ldb,
                            b_batched ? (uint64_t)strideB : (uint64_t)ldb * K, 16, Cfg::BK);
    if (rc) return rc;

    TnArgs args;
    args.C = C;
    args.C2 = dual.C2;
    args.d0 = dual.d0;
    args.d1 = dual.d1;
    args.d2 = dual.d2;
    args.M = M;
    args.N = N;
    args.ldc = ldc;
    args.strideC = strideC;
    args.strideC2 = dual.strideC2;
    args.kblocks = (int)ceil_div(K, Cfg::BK);
    args.tiles_m = (int)ceil_div(M, Cfg::BM);
    args.tiles_n = (int)ceil_div(N, Cfg::BN);
    args.batch = batch;
    args.a_batched = a_batched;
    args.b_batched = b_batched;
    args.zero = 0;
    args.A8 = nullptr;
    args.strideA8 = 0;
    args.K = (int)K;
    args.pq_lo = args.pq_cnt = 0;
    args.a8_ld = 0;
    args.r2_offset = dual.r2_offset;
    args.sym_T = args.sym_tiles_per_batch = 0;
    args.last_subs = 2 * (int)ceil_div(K - (int64_t)(args.kblocks - 1) * Cfg::BK, 8);

    static unsigned long long attr_set = 0;
    if (once_per_device(attr_set)) {
        OO_CUDA_CHECK(cudaFuncSetAttribute(dgemm_tn_kernel<Cfg, 0>,
                                           cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           Cfg::SMEM_BYTES));
        OO_CUDA_CHECK(cudaFuncSetAttribute(dgemm_tn_kernel<Cfg, 1>,
                                           cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           Cfg::SMEM_BYTES));
        OO_CUDA_CHECK(cudaFuncSetAttribute(dgemm_tn_kernel<Cfg, 2>,
                                           cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           Cfg::SMEM_BYTES));
        OO_CUDA_CHECK(cudaFuncSetAttribute(dgemm_tn_kernel<Cfg, 3>,
                                           cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           Cfg::SMEM_BYTES));
        OO_CUDA_CHECK(cudaFuncSetAttribute(dgemm_tn_kernel<Cfg, 4>,
                                           cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           Cfg::SMEM_BYTES));
        OO_CUDA_CHECK(cudaFuncSetAttribute(dgemm_tn_kernel<Cfg, 5>,
                                           cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           Cfg::SMEM_BYTES));
        if constexpr (Cfg::EPI0_STAGES >= 2 && Cfg::BN >= 128) {
#ifdef OO_TN_STAGE_PLAIN_STORES
            OO_CUDA_CHECK(cudaFuncSetAttribute(dgemm_tn_kernel<Cfg, 0, 0, 1>,
                                               cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::EPI0_SMEM_BYTES));
#endif
            OO_CUDA_CHECK(cudaFuncSetAttribute(dgemm_tn_kernel<Cfg, 5, 0, 1>,
                                               cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::EPI0_SMEM_BYTES));
        }
    }
    const int64_t total = (int64_t)args.tiles_m * args.tiles_n * batch;
    const int grid = (int)(total < sm_count() ? total : sm_count());
    // staged epilogue (tile -> shared memory -> bulk copies by the producer warpgroup's spare warps): big tiles only
    // (the 128 x 128 configuration), even N (16-byte row pieces), at least two k-blocks to hide the shipping behind
    constexpr bool kCanStage = Cfg::EPI0_STAGES >= 2 && Cfg::BN >= 128;
    const bool staged = kCanStage && !dual.direct_epilogue && (N % 2) == 0 && args.kblocks >= 2;
  if constexpr (kCanStage) {
    // (the plain store is NOT staged: its epilogue is 3 % of a 128 x 128 tile, less than what the two-stage ring that
    //  makes room for the tile costs -- measured 0.99 -> 1.03 ms per quarter at N = 256; the kernel variant exists
    //  behind OO_TN_STAGE_PLAIN_STORES for experiments)
#ifdef OO_TN_STAGE_PLAIN_STORES
    if (staged && !dual.C2) {
        dgemm_tn_kernel<Cfg, 0, 0, 1><<<grid, Cfg::THREADS, Cfg::EPI0_SMEM_BYTES, stream>>>(mapA, mapB, args);
        OO_LAUNCH_CHECK();
        return OO_OK;
    }
#endif
    if (staged && dual.C2 && dual.mode == 5) {
        int sgrid = grid;
        if (dual.symmetric_blocks && Cfg::BM == Cfg::BN && dual.d1 % Cfg::BM == 0 && N == dual.d1 && M % dual.d1 == 0 &&
            dual.d1 / Cfg::BM >= 2) {
            // Coulomb class: only the tiles on and below the diagonal of every symmetric d1 x d1 block
            args.sym_T = dual.d1 / Cfg::BM;
            args.sym_tiles_per_batch = (int)(M / dual.d1) * args.sym_T * (args.sym_T + 1) / 2;
            const int64_t stotal = (int64_t)args.sym_tiles_per_batch * batch;
            sgrid = (int)(stotal < sm_count() ? stotal : sm_count());
        }
        dgemm_tn_kernel<Cfg, 5, 0, 1><<<sgrid, Cfg::THREADS, Cfg::EPI0_SMEM_BYTES, stream>>>(mapA, mapB, args);
        OO_LAUNCH_CHECK();
        return OO_OK;
    }
  }
    (void)staged;
    if (dual.C2 && dual.mode == 5)
        dgemm_tn_kernel<Cfg, 5><<<grid, Cfg::THREADS, Cfg::SMEM_BYTES, stream>>>(mapA, mapB, args);
    else if (dual.C2 && dual.mode == 4)
        dgemm_tn_kernel<Cfg, 4><<<grid, Cfg::THREADS, Cfg::SMEM_BYTES, stream>>>(mapA, mapB, args);
    else if (dual.C2 && dual.mode == 3)
        dgemm_tn_kernel<Cfg, 3><<<grid, Cfg::THREADS, Cfg::SMEM_BYTES, stream>>>(mapA, mapB, args);
    else if (dual.C2 && dual.mode == 2)
        dgemm_tn_kernel<Cfg, 2><<<grid, Cfg::THREADS, Cfg::SMEM_BYTES, stream>>>(mapA, mapB, args);
    else if (dual.C2)
        dgemm_tn_kernel<Cfg, 1><<<grid, Cfg::THREADS, Cfg::SMEM_BYTES, stream>>>(mapA, mapB, args);
    else
        dgemm_tn_kernel<Cfg, 0><<<grid, Cfg::THREADS, Cfg::SMEM_BYTES, stream>>>(mapA, mapB, args);
    OO_LAUNCH_CHECK();
    return OO_OK;
}

// Quarter 1 of the symmetric class transform straight from the 8-fold packed AO integrals (AMODE 1):
//   T1[(s, PQ), m] = sum_r A8[RS(r, s)][PQ] C[r, m],   RS(r, s) = tri(max, min),
// stored as C[(s PQ), m] and, pair unpacked, at C2 rows (q p s) and (p q s) (the mode-2 epilogue).
template <class Cfg>
static int launch_tn_q1_packed8(const double *A8, int64_t a8_ld, int pq_lo, int pq_cnt, const double *B, double *C,
                                double *C2, int S, int dorb, int dP, int64_t N, int64_t K, int64_t ldb, int64_t ldc,
                                int batch, int64_t strideA8, int64_t strideB, int64_t strideC, int64_t strideC2,
                                cudaStream_t stream, bool direct_epilogue) {
    CUtensorMap mapB;
    const int b_batched = (batch > 1 && strideB != 0);
    int rc = encode_tmap_3d_f64(&mapB, B, (uint64_t)N, (uint64_t)K, b_batched ? batch : 1, (uint64_t)ldb,
                                b_batched ? (uint64_t)strideB : (uint64_t)ldb * K, 16, Cfg::BK);
    if (rc) return rc;
    TnArgs args;
    args.C = C;
    args.C2 = C2;
    args.d0 = S;
    args.d1 = dorb;
    args.d2 = dP;
    args.M = (int64_t)S * dP;
    args.N = N;
    args.ldc = ldc;
    args.strideC = strideC;
    args.strideC2 = strideC2;
    args.kblocks = (int)ceil_div(K, Cfg::BK);
    args.tiles_m = S * (int)ceil_div(pq_cnt, Cfg::BM);
    args.tiles_n = (int)ceil_div(N, Cfg::BN);
    args.batch = batch;
    args.a_batched = (batch > 1 && strideA8 != 0);
    args.b_batched = b_batched;
    args.zero = 0;
    args.A8 = A8;
    args.strideA8 = args.a_batched ? strideA8 : 0;
    args.K = (int)K;
    args.pq_lo = pq_lo;
    args.pq_cnt = pq_cnt;
    args.a8_ld = a8_ld;
    args.r2_offset = 0;
    args.sym_T = args.sym_tiles_per_batch = 0;
    args.last_subs = 2 * (int)ceil_div(K - (int64_t)(args.kblocks - 1) * Cfg::BK, 8);
    static unsigned long long attr_set = 0;
    if (once_per_device(attr_set)) {
        OO_CUDA_CHECK(cudaFuncSetAttribute(dgemm_tn_kernel<Cfg, 2, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           Cfg::LIN_SMEM_BYTES));
        if constexpr (Cfg::EPI_SMEM_BYTES <= 227 * 1024)
            OO_CUDA_CHECK(cudaFuncSetAttribute(dgemm_tn_kernel<Cfg, 2, 1, 1>,
                                               cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::EPI_SMEM_BYTES));
    }
    const int64_t total = (int64_t)args.tiles_m * args.tiles_n * batch;
    const int grid = (int)(total < sm_count() ? total : sm_count());
    // staged epilogue: one n-tile, dense rows (ldc == N), enough shared memory, and not asked for the direct stores
    constexpr bool kCanStage = Cfg::EPI_SMEM_BYTES <= 227 * 1024;
    bool staged = false;
    if constexpr (kCanStage) {
        staged = !direct_epilogue && args.tiles_n == 1 && ldc == N && (N % 2) == 0;
        if (staged)
            dgemm_tn_kernel<Cfg, 2, 1, 1><<<grid, Cfg::THREADS, Cfg::EPI_SMEM_BYTES, stream>>>(mapB, mapB, args);
    }
    if (!staged) dgemm_tn_kernel<Cfg, 2, 1><<<grid, Cfg::THREADS, Cfg::LIN_SMEM_BYTES, stream>>>(mapB, mapB, args);
    OO_LAUNCH_CHECK();
    return OO_OK;
}

//                     BM   BN  BK WGM WGN STAGES
using TnWide = TnCfg<128, 128, 16, 2, 4, 4>;   // N > 64 : warp tile 64x32
using TnMid = TnCfg<256, 64, 16, 4, 2, 4>;     // N in (48, 64]
using TnM192 = TnCfg<192, 64, 16, 4, 2, 4>;    // 128 < M <= 192 rows, many columns: the C block of the Hessian (M = na^2 + no
                                               // = 176 at CAS(12,12), 32 core orbitals) would waste a third of 128-row tiles
using TnMid48 = TnCfg<256, 48, 16, 8, 1, 4>;   // N in (32, 48] : warp tile 32x48 (class index nIp = 44 at N=256)
using TnMid40 = TnCfg<256, 48, 16, 8, 1, 4, 5>;   // N in (32, 40] : warp tile 32x40
using TnNarrow = TnCfg<256, 32, 16, 8, 1, 4>;  // N in (24, 32] : warp tile 32x32
using TnNarrow24 = TnCfg<256, 32, 16, 8, 1, 4, 3>;  // N in (16, 24] : warp tile 32x24 (class index 24 at 114 orbitals)
using TnSlim = TnCfg<256, 16, 16, 8, 1, 4>;    // N <= 16 : warp tile 32x16
// quarter 1 of TWO evaluations side by side (classes.cu: columns [C_2j | C_2j+1], 2 x 44 at N=256): warp tile 16x88 / 16x96
// -- 88 accumulator registers, and the 128 x 88 result tile (90 KB) still fits next to a three-stage ring
using TnPair88 = TnCfg<128, 96, 16, 8, 1, 4, 11>;
using TnPair96 = TnCfg<128, 96, 16, 8, 1, 4>;

static int dgemm_tn_impl(const double *At, const double *B, double *C, int64_t M, int64_t N, int64_t K,
                         int64_t lda, int64_t ldb, int64_t ldc, int batch, int64_t strideA, int64_t strideB,
                         int64_t strideC, cudaStream_t stream, const TnDual &dual) {
    OO_REQUIRE(At && B && C);
    OO_REQUIRE(M > 0 && N > 0 && K > 0 && batch > 0);
    OO_REQUIRE(lda >= M && ldb >= N && ldc >= N);
    OO_REQUIRE((lda % 2) == 0 && (ldb % 2) == 0 && (ldc % 2) == 0);
    OO_REQUIRE((strideA % 2) == 0 && (strideB % 2) == 0 && (strideC % 2) == 0);
    OO_REQUIRE(((uintptr_t)At % 16) == 0 && ((uintptr_t)B % 16) == 0 && ((uintptr_t)C % 16) == 0);
    if (M >= (1ll << 31) || N >= (1ll << 31) || K >= (1ll << 31)) return OO_ERR_UNSUPPORTED;
    if (N > 64 && M > 128 && M <= 192 && N >= 64 * 148 && !dual.C2)
        return launch_tn<TnM192>(At, B, C, M, N, K, lda, ldb, ldc, batch, strideA, strideB, strideC, stream, dual);
    if (N > 64)
        return launch_tn<TnWide>(At, B, C, M, N, K, lda, ldb, ldc, batch, strideA, strideB, strideC, stream, dual);
    if (N > 48)
        return launch_tn<TnMid>(At, B, C, M, N, K, lda, ldb, ldc, batch, strideA, strideB, strideC, stream, dual);
    if (N > 40)
        return launch_tn<TnMid48>(At, B, C, M, N, K, lda, ldb, ldc, batch, strideA, strideB, strideC, stream, dual);
    if (N > 32)
        return launch_tn<TnMid40>(At, B, C, M, N, K, lda, ldb, ldc, batch, strideA, strideB, strideC, stream, dual);
    if (N > 24)
        return launch_tn<TnNarrow>(At, B, C, M, N, K, lda, ldb, ldc, batch, strideA, strideB, strideC, stream, dual);
    if (N > 16)
        return launch_tn<TnNarrow24>(At, B, C, M, N, K, lda, ldb, ldc, batch, strideA, strideB, strideC, stream, dual);
    return launch_tn<TnSlim>(At, B, C, M, N, K, lda, ldb, ldc, batch, strideA, strideB, strideC, stream, dual);
}

int dgemm_tn(const double *At, const double *B, double *C, int64_t M, int64_t N, int64_t K,
             int64_t lda, int64_t ldb, int64_t ldc, int batch, int64_t strideA, int64_t strideB,
             int64_t strideC, cudaStream_t stream) {
    return dgemm_tn_impl(At, B, C, M, N, K, lda, ldb, ldc, batch, strideA, strideB, strideC, stream, TnDual());
}

// the same product with the consumer warps storing their accumulators themselves (A/B tests of the staged epilogue)
int dgemm_tn_direct(const double *At, const double *B, double *C, int64_t M, int64_t N, int64_t K,
                    int64_t lda, int64_t ldb, int64_t ldc, int batch, int64_t strideA, int64_t strideB,
                    int64_t strideC, cudaStream_t stream) {
    TnDual dual;
    dual.direct_epilogue = true;
    return dgemm_tn_impl(At, B, C, M, N, K, lda, ldb, ldc, batch, strideA, strideB, strideC, stream, dual);
}

// C[(a b c), n] and C2[(c b a), n] from one pass (M = d0*d1*d2, same ldc and batch stride for both)
int dgemm_tn_swap02(const double *At, const double *B, double *C, double *C2, int d0, int d1, int d2,
                    int64_t N, int64_t K, int64_t lda, int64_t ldb, int64_t ldc, int batch, int64_t strideA,
                    int64_t strideB, int64_t strideC, cudaStream_t stream) {
    OO_REQUIRE(C2 && d0 > 0 && d1 > 0 && d2 > 0);
    TnDual dual;
    dual.C2 = C2;
    dual.mode = 1;
    dual.d0 = d0;
    dual.d1 = d1;
    dual.d2 = d2;
    dual.strideC2 = strideC;
    return dgemm_tn_impl(At, B, C, (int64_t)d0 * d1 * d2, N, K, lda, ldb, ldc, batch, strideA, strideB, strideC,
                         stream, dual);
}

// Rows (a, pq): a < d0, pq < dP a packed lower-triangular pair (p >= q) of `dorb` orbitals, dP >= dorb(dorb+1)/2
// (padding rows carry zeros).  C[(a pq), n] is stored as is; C2 receives the same value at rows (q p a) and
// (p q a), i.e. the pair index unpacked to both orders and moved to the front (M2 = dorb*dorb*d0 rows).
int dgemm_tn_pair_unpack(const double *At, const double *B, double *C, double *C2, int d0, int dorb, int dP,
                         int64_t N, int64_t K, int64_t lda, int64_t ldb, int64_t ldc, int batch,
                         int64_t strideA, int64_t strideB, int64_t strideC, int64_t strideC2,
                         cudaStream_t stream) {
    OO_REQUIRE(C2 && d0 > 0 && dorb > 0 && (int64_t)dP >= (int64_t)dorb * (dorb + 1) / 2);
    if ((int64_t)dorb * (dorb + 1) / 2 >= (1ll << 30)) return OO_ERR_UNSUPPORTED;
    TnDual dual;
    dual.C2 = C2;
    dual.mode = 2;
    dual.d0 = d0;
    dual.d1 = dorb;
    dual.d2 = dP;
    dual.strideC2 = strideC2;
    return dgemm_tn_impl(At, B, C, (int64_t)d0 * dP, N, K, lda, ldb, ldc, batch, strideA, strideB, strideC,
                         stream, dual);
}

// Quarter 1 from the 8-fold packed AO integrals A8[RS][PQ] (rows of dP doubles, RS over pairs of S = dorb orbitals):
// see launch_tn_q1_packed8.  N = number of class columns (ldb, ldc even).
// A8 may be a slab of the pair columns: row pitch a8_ld, columns PQ in [pq_lo, pq_lo + pq_cnt) (both even).
int dgemm_tn_q1_packed8(const double *A8, int64_t a8_ld, int pq_lo, int pq_cnt, const double *B, double *C,
                        double *C2, int dorb, int dP, int64_t N, int64_t K, int64_t ldb, int64_t ldc, int batch,
                        int64_t strideA8, int64_t strideB, int64_t strideC, int64_t strideC2, cudaStream_t stream,
                        bool direct_epilogue) {
    OO_REQUIRE(A8 && B && C && C2 && dorb > 0 && K > 0 && K <= dorb && N > 0 && batch > 0);
    OO_REQUIRE(pq_lo >= 0 && pq_cnt > 0 && pq_lo + pq_cnt <= dP && (pq_lo % 2) == 0 && (pq_cnt % 2) == 0);
    OO_REQUIRE(a8_ld >= pq_cnt && (a8_ld % 2) == 0);
    OO_REQUIRE((int64_t)dP >= (int64_t)dorb * (dorb + 1) / 2 && (dP % 2) == 0);
    OO_REQUIRE((ldb % 2) == 0 && (ldc % 2) == 0 && ldc >= N && (strideA8 % 2) == 0 && (strideB % 2) == 0);
    OO_REQUIRE(((uintptr_t)A8 % 16) == 0 && ((uintptr_t)B % 16) == 0 && ((uintptr_t)C % 16) == 0);
    if ((int64_t)dorb * dP >= (1ll << 31)) return OO_ERR_UNSUPPORTED;
#define OO_Q1(CFG)                                                                                                 \
    return launch_tn_q1_packed8<CFG>(A8, a8_ld, pq_lo, pq_cnt, B, C, C2, dorb, dorb, dP, N, K, ldb, ldc, batch,      \
                                     strideA8, strideB, strideC, strideC2, stream, direct_epilogue)
    if (N > 88 && N <= 96) OO_Q1(TnPair96);
    if (N > 80 && N <= 88) OO_Q1(TnPair88);
    if (N > 64) OO_Q1(TnWide);
    if (N > 48) OO_Q1(TnMid);
    if (N > 40) OO_Q1(TnMid48);
    if (N > 32) OO_Q1(TnMid40);
    if (N > 24) OO_Q1(TnNarrow);
    if (N > 16) OO_Q1(TnNarrow24);
    OO_Q1(TnSlim);
#undef OO_Q1
}

// Rows (r2, m), m < nclass, columns n < N (= nclass): only the class pairs n <= m are stored, packed, at
// P[r2'][m(m+1)/2 + n] (row length npair_ld); nothing else is written.  tri_rows: r2 = p(p+1)/2 + q is a packed
// pair of `dorb` orbitals (nrows2 >= dorb(dorb+1)/2 rows, padding skipped) and both P[(p q)] and P[(q p)] are
// written; otherwise r2' = r2.  This is the quarter-2 GEMM of the symmetric class transform with
// pack_class_pairs fused into its epilogue.
int dgemm_tn_class_pack(const double *At, const double *B, double *P, int tri_rows, int nclass, int dorb,
                        int64_t nrows2, int64_t npair_ld, int64_t K, int64_t lda, int64_t ldb, int batch,
                        int64_t strideA, int64_t strideB, int64_t strideP, cudaStream_t stream, int64_t r2_offset) {
    OO_REQUIRE(P && nclass > 0 && dorb > 0 && nrows2 > 0 && npair_ld >= (int64_t)nclass * (nclass + 1) / 2);
    TnDual dual;
    dual.C2 = P;
    dual.mode = tri_rows ? 3 : 4;
    dual.d0 = nclass;
    dual.d1 = dorb;
    dual.d2 = (int)npair_ld;
    dual.strideC2 = strideP;
    dual.r2_offset = r2_offset;
    const int64_t ldc = nclass + (nclass & 1);
    return dgemm_tn_impl(At, B, P, nrows2 * nclass, nclass, K, lda, ldb, ldc, batch, strideA, strideB, 0, stream, dual);
}

// Rows (mn, a): mn < npair_ld a packed class pair (m >= n) of `nclass` indices, a < dorb; columns b < dorb.
// Out[(m n), a, b] is written for every pair and, for m != n, Out[(n m), a, b] (transpose_mirror == 0: the
// Coulomb class, J[n,m] = J[m,n]) or Out[(n m), b, a] (the exchange class, K[n,m] = K[m,n]^T); planes of
// dorb x ld_out doubles.  The last quarter of the symmetric class transform with expand_class fused into it.
int dgemm_tn_class_expand(const double *At, const double *B, double *Out, int transpose_mirror, int nclass, int dorb,
                          int64_t npair_ld, int64_t K, int64_t lda, int64_t ldb, int64_t ld_out, int batch,
                          int64_t strideA, int64_t strideB, int64_t strideOut, cudaStream_t stream,
                          bool direct_epilogue) {
    OO_REQUIRE(Out && nclass > 0 && dorb > 0 && npair_ld >= (int64_t)nclass * (nclass + 1) / 2 && ld_out >= dorb);
    TnDual dual;
    dual.C2 = Out;
    dual.mode = 5;
    dual.d0 = nclass;
    dual.d1 = dorb;
    dual.d2 = transpose_mirror ? 1 : 0;
    dual.strideC2 = strideOut;
    dual.direct_epilogue = direct_epilogue;
    dual.symmetric_blocks = !transpose_mirror;      // J[mn][a][b] = J[mn][b][a]; the exchange class has no such symmetry
    return dgemm_tn_impl(At, B, Out, npair_ld * dorb, dorb, K, lda, ldb, ld_out, batch, strideA, strideB, 0, stream,
                         dual);
}

}  // namespace oo

extern "C" int oo_dgemm_tn_f64(const double *At, const double *B, double *C, int64_t M, int64_t N,
                               int64_t K, int64_t lda, int64_t ldb, int64_t ldc, int batch,
                               int64_t strideA, int64_t strideB, int64_t strideC, void *stream) {
    return oo::dgemm_tn(At, B, C, M, N, K, lda, ldb, ldc, batch, strideA, strideB, strideC,
                        (cudaStream_t)stream);
}

extern "C" int oo_dgemm_tn_swap02_f64(const double *At, const double *B, double *C, double *C2, int d0,
                                      int d1, int d2, int64_t N, int64_t K, int64_t lda, int64_t ldb,
                                      int64_t ldc, void *stream) {
    return oo::dgemm_tn_swap02(At, B, C, C2, d0, d1, d2, N, K, lda, ldb, ldc, 1, 0, 0, 0, (cudaStream_t)stream);
}
