// pgroup_tc.cu -- tensor-core kernel for the pattern-grouped format (kernel K4 of SURVEY.md 2.2):
// tcgen05.mma with an error-compensated TF32 + BF16 split (2 MMAs per 8 k), fp32 accumulators in TMEM.
//
// Per pattern group g (see pgroup.cu) the product  Y[rows[g], :] = V_g (G x K) . X[cols[g], :] (K x N)
// is a true small GEMM (G = 96..512 output channels, K = 9*Cin+1 = 865..4609, N = batch), which is what
// north_star allows on the tensor pipe.  Orientation: the BATCH is the UMMA M dimension (always a full
// 128 lanes), the group's rows are the UMMA N dimension (any multiple of 16 up to 256, so G = 96 or 192
// wastes nothing):
//
//     D[128 batch][Gp] (TMEM, fp32)  +=  A[128 batch][8 k] (smem, MN-major)  .  B[8 k][Gp] (smem, K-major)
//
//   * B = weight block V_g: pre-split at pack time (kn_pg_tc_split) into a hi plane (v rounded to nearest TF32) and a
//     corr plane of bf16 pairs ([w_lo ; w_hi] per 8 k, lo = v - hi), both K-contiguous 4-byte words, loaded by TMA
//     (SWIZZLE_64B boxes of 16 words x Gp rows).
//   * A = gathered activation rows X[cols[g][k], n0:n0+128], kept in TENSOR MEMORY (lane = batch element,
//     column = k): eight producer warps read coalesced 128-byte row segments, split them into TF32 hi words and bf16
//     [x_hi | x_lo] pairs in registers and write both with tcgen05.st into a TMEM ring; the MMA takes A from TMEM, so shared memory
//     carries only the weight ring.  (A first version staged A in shared memory, in the MN-major
//     SWIZZLE_128B_BASE32B layout -- the only MN-major layout tcgen05 accepts for 32-bit operands; it was
//     bound by the 128 B/clk shared-memory port: 7 KB of operands per 48-cycle N=96 MMA.)
//   * one elected thread issues, per 8-k step, x_hi.w_hi (kind::tf32, K = 8) and [x_hi | x_lo].[w_lo ; w_hi]
//     (kind::f16 in bf16, K = 16: both correction products in ONE instruction that reads as many operand bytes as a tf32
//     K = 8 one and runs at twice its rate), both into the same fp32 accumulator.  Error per product < 2^-16.9 |x||w|
//     (tc_common.cuh), inside the fp32 rtol 1e-4 parity bar, which plain TF32 (10-bit mantissa) would not be.
//   * stages of 16 k, ring of kStages (full/empty mbarriers, tcgen05.commit frees a stage), epilogue:
//     tcgen05.ld 32x32b.x16 -> ReLU -> Y[rows[g][j]][n] (32 lanes = 32 consecutive batch columns = 128 B).
//
// One CTA per (group, 128*NB batch columns); NB = 2 batch tiles share every weight stage.
#include "tc_common.cuh"
#include <string.h>

namespace {
using namespace kn_tc;

constexpr int kThreads = 384;          // warp 0: TMA(B)  warps 1,3: MMA issuers  warp 2: TMEM alloc  warps 4-11: A producers + epilogue
constexpr int kProducerThreads = 256;

// Shared memory holds only the weight ring; the activation operand lives in TMEM:
//   TMEM columns [0, NB*Gp)                      fp32 accumulators, one Gp-wide block per batch tile
//   TMEM columns [a0 + (sa*NB + b)*32, +32)      A ring: 16 TF32 hi columns (column = k), then per 8 k 4 columns of bf16
//                                                x_hi pairs and 4 of bf16 x_lo pairs (lane = batch element)
// A tf32 UMMA with N = 96 needs 4 KB of A and 3 KB of B per 48 cycles; with A in shared memory that is 146 B/clk, above
// the 128 B/clk shared-memory port, so the tensor pipe starves.  From TMEM the A operand costs no shared-memory
// bandwidth and the producers' stores (tcgen05.st) bypass shared memory as well.
// phase timestamps of one CTA (debug aid, read back with kn_debug_tc_timing): entry, prologue done, first stage full,
// last MMA issued, accumulators ready, epilogue stored, teardown
__device__ long long g_tc_timing[8];
__device__ int g_tc_timing_cta = -1;
#define KN_STAMP(i) do { if ((int)blockIdx.x == g_tc_timing_cta) g_tc_timing[i] = clock64(); } while (0)

template <int NB, bool RELU, int CS, bool PEERS>
__global__ void __launch_bounds__(kThreads, 1)
pg_tc_kernel(const __grid_constant__ CUtensorMap map_hi, const __grid_constant__ CUtensorMap map_corr,
             const int32_t *__restrict__ rows, const int32_t *__restrict__ cols, const int32_t *__restrict__ group_k, const int32_t *__restrict__ block_of,
             int G, int Gp, int K_pad, int chunks_per_group, int64_t n_items, int64_t n_tiles, int n_b, int n_a, uint32_t a0, int super_tiles,
             const float *__restrict__ X, int64_t ldx, float *__restrict__ Y, int64_t ldy, int64_t n_vecs, const __grid_constant__ KnPeers peers)
{
    extern __shared__ unsigned char smem_dyn[];
    unsigned char *smem = reinterpret_cast<unsigned char *>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023) & ~(uintptr_t)1023);
    const int b_plane_bytes = Gp * KS * 4;                       // Gp rows x 64 B
    const int stage_bytes = 2 * b_plane_bytes;                   // hi plane, corr plane
    int32_t *s_cols = reinterpret_cast<int32_t *>(smem + (size_t)n_b * stage_bytes);        // the group's gather list, K_pad entries
    uint64_t *fullB = reinterpret_cast<uint64_t *>(smem + (size_t)n_b * stage_bytes + (size_t)K_pad * 4);
    uint64_t *emptyB = fullB + n_b;
    uint64_t *fullA = emptyB + n_b;
    uint64_t *emptyA = fullA + n_a;
    uint64_t *accum_bar = emptyA + n_a;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(accum_bar + 1);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const KnRaster rt = kn_raster(blockIdx.x, n_items, n_tiles, super_tiles);
    const int64_t g = rt.item / chunks_per_group;                // pattern group
    const int gchunk = (int)(rt.item - g * chunks_per_group);    // 256-row chunk of a very tall group
    const int row0 = gchunk * 256;                               // first group row handled here
    const int64_t nbase = rt.tile * (BM * NB);
    // groups of one class share K_pad (storage) but loop only over their own K (edge / corner pixels have fewer taps)
    const int n_ksteps = group_k ? (__ldg(group_k + g) + KS - 1) / KS : K_pad / KS;
    const uint32_t crank = (CS > 1) ? cluster_ctarank() : 0u;

    if (tid == 0) KN_STAMP(0);
    if (warp == 0 && lane == 0) {
        // NB MMA issuers (one per batch tile): each commits once per stage to both rings and once to accum_bar
        // CS > 1: the CTAs of a cluster (same group, adjacent batch tiles) share every weight stage by TMA multicast, so a
        // stage is free only when the issuers of ALL cluster CTAs have retired it
        for (int s = 0; s < n_b; s++) { mbar_init(&fullB[s], 1); mbar_init(&emptyB[s], NB * CS); }
        for (int s = 0; s < n_a; s++) { mbar_init(&fullA[s], kProducerThreads); mbar_init(&emptyA[s], NB); }
        mbar_init(accum_bar, NB);
        fence_barrier_init();
    } else if (warp == 2) {
        tmem_alloc512(tmem_slot);
    }
    // the column list is read once per CTA: a gather then never waits for an index load before it can issue
    for (int i = tid; i < n_ksteps * KS; i += kThreads) s_cols[i] = __ldg(cols + g * (int64_t)K_pad + i);
    tc_fence_before();
    __syncthreads();
    if (CS > 1) cluster_sync_all();                              // partner barriers are initialised before any multicast
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    if (tid == 0) KN_STAMP(1);

    if (warp == 0) {
        // ===== TMA producer: weight block planes (hi, corr), 16 k x Gp rows per stage =====
        if (elect_one()) {
            const int grow = (int)((block_of ? (int64_t)__ldg(block_of + g) : g) * G) + row0;      // rows of the group's unique value block
            int s = 0; uint32_t ph = 0;                          // ring position / phase kept incrementally (no runtime div/mod)
            for (int ks = 0; ks < n_ksteps; ks++) {
                mbar_wait(&emptyB[s], ph ^ 1u);
                unsigned char *bs = smem + (size_t)s * stage_bytes;
                mbar_arrive_expect_tx(&fullB[s], 2u * (uint32_t)b_plane_bytes);
                if (CS == 1) {
                    tma_load_2d(bs, &map_hi, ks * KS, grow, &fullB[s]);
                    tma_load_2d(bs + b_plane_bytes, &map_corr, ks * KS, grow, &fullB[s]);
                } else {
                    // this CTA fetches rows [rank*Gp/CS, (rank+1)*Gp/CS) of both planes and multicasts them to the cluster
                    const int part = Gp / CS, r0 = (int)crank * part;
                    tma_load_2d_mcast(bs + r0 * KS * 4, &map_hi, ks * KS, grow + r0, &fullB[s], (uint16_t)((1u << CS) - 1u));
                    tma_load_2d_mcast(bs + b_plane_bytes + r0 * KS * 4, &map_corr, ks * KS, grow + r0, &fullB[s], (uint16_t)((1u << CS) - 1u));
                }
                if (++s == n_b) { s = 0; ph ^= 1u; }
            }
        }
    } else if (warp == 1 || (warp == 3 && NB == 2)) {
        // ===== MMA issuers: one elected thread per batch tile (warp 1 -> batch tile 0, warp 3 -> batch tile 1) =====
        if (elect_one()) {
            const int b = (warp == 1) ? 0 : 1;
            const uint32_t idesc = make_idesc_tf32(BM, Gp);
            const uint32_t idesc_c = make_idesc_bf16(BM, Gp);
            const uint32_t d = tmem_base + (uint32_t)(b * Gp);
            const uint64_t desc0 = make_desc(smem_u32(smem), 16, 512, kLayoutSW64);
            int sb = 0, sa = 0; uint32_t pb = 0, pa = 0;
            for (int ks = 0; ks < n_ksteps; ks++) {
                mbar_wait(&fullB[sb], pb);
                mbar_wait(&fullA[sa], pa);
                tc_fence_after();
                if (ks == 0 && warp == 1) KN_STAMP(2);
                const uint32_t ta = tmem_base + a0 + (uint32_t)((sa * NB + b) * 32);
                // B: K-major SW64 (64-byte rows), 8-row groups 512 B apart; stage / plane / k-step only move the
                // 14-bit start-address field (units of 16 B), so the descriptor is one 64-bit add away from desc0.  An
                // 8-k step is 32 B of a row in both planes: 8 tf32 words, or 16 bf16 (8 words) of the corr plane.
                const uint64_t dstage = desc0 + (uint64_t)(((uint32_t)sb * (uint32_t)stage_bytes) >> 4);
#pragma unroll
                for (int kk = 0; kk < KS / 8; kk++) {
                    const uint64_t db_hi = dstage + (uint64_t)(kk * 2);
                    const uint64_t db_corr = db_hi + (uint64_t)(b_plane_bytes >> 4);
                    umma_tf32_ts(d, ta + kk * 8, db_hi, idesc, (ks > 0 || kk > 0) ? 1u : 0u);    // x_hi . w_hi
                    umma_bf16_ts(d, ta + 16 + kk * 8, db_corr, idesc_c, 1u);                     // x_hi . w_lo + x_lo . w_hi
                }
                if (CS == 1) umma_commit(&emptyB[sb]);         // both rings are released when every issuer's MMAs retire
                else umma_commit_mcast(&emptyB[sb], (uint16_t)((1u << CS) - 1u));
                umma_commit(&emptyA[sa]);
                if (++sb == n_b) { sb = 0; pb ^= 1u; }
                if (++sa == n_a) { sa = 0; pa ^= 1u; }
            }
            umma_commit(accum_bar);
            if (warp == 1) KN_STAMP(3);
        }
    } else if (warp >= 4) {
        // ===== A producers: gather X, split into TF32 hi + bf16 corr words, tcgen05.st into the TMEM A ring =====
        // thread = one batch element (TMEM lane); it loads X[cols[k]][n] for the k's of its stage share -- each warp
        // load is one coalesced 128-byte row segment -- and runs PD stages ahead of the TMEM stores (register ring).
        const int q = warp & 3;                                 // TMEM lane quarter of this warp
        const int sel = (warp - 4) >> 2;                        // NB == 2: batch tile; NB == 1: k half of the stage
        constexpr int KW = (NB == 2) ? 16 : 8;                  // k values per thread and stage
        constexpr int PD = 4;                                   // prefetch distance in stages
        const int b_mine = (NB == 2) ? sel : 0;
        const int k0 = (NB == 2) ? 0 : sel * 8;
        const int64_t n = nbase + b_mine * BM + q * 32 + lane;
        const bool n_ok = n < n_vecs;
        // address of X[c][n] = xaddr + c * (ldx * 4): one IMAD.WIDE.U32 + one ld.global.nc per element.  Batch lanes past
        // n_vecs are clamped to the last valid column: their TMEM rows only feed outputs the epilogue never stores.
        const uint64_t xaddr = reinterpret_cast<uint64_t>(X) + (uint64_t)(n_ok ? n : (n_vecs - 1)) * 4ull;
        const uint32_t ldxb = (uint32_t)ldx * 4u;
        float buf[PD][KW];

        auto gather = [&](float (&v)[KW], int ks) {
            const int4 *cp = reinterpret_cast<const int4 *>(s_cols + ks * KS + k0);             // 16-byte aligned
#pragma unroll
            for (int i4 = 0; i4 < KW / 4; i4++) {
                const int4 c = cp[i4];                          // warp-broadcast LDS.128: 4 column indices
                const uint32_t cc[4] = {(uint32_t)c.x, (uint32_t)c.y, (uint32_t)c.z, (uint32_t)c.w};
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    uint64_t a;
                    asm("mad.wide.u32 %0, %1, %2, %3;" : "=l"(a) : "r"(cc[j]), "r"(ldxb), "l"(xaddr));
                    asm volatile("ld.global.nc.f32 %0, [%1];" : "=f"(v[4 * i4 + j]) : "l"(a));
                }
            }
        };
        int psa = 0; uint32_t ppa = 0;                           // producer ring position / phase
        auto publish = [&](const float (&v)[KW]) {
            const int sa = psa;
            uint32_t hi[KW], corr[KW];                          // corr: per 8 k, 4 bf16 x_hi pairs then 4 bf16 x_lo pairs
#pragma unroll
            for (int h = 0; h < KW / 8; h++) split8_tf32_bf16(v + 8 * h, hi + 8 * h, corr + 8 * h, corr + 8 * h + 4);
            mbar_wait(&emptyA[sa], ppa ^ 1u);
            tc_fence_after();
            const uint32_t ta = tmem_base + ((uint32_t)(q * 32) << 16) + a0 + (uint32_t)((sa * NB + b_mine) * 32 + k0);
            tmem_store<KW>(ta, hi);
            tmem_store<KW>(ta + 16, corr);
        };
        // completing a stage (wait for the TMEM stores, then signal the issuers) is deferred until the next
        // gather has been issued, so the store latency overlaps with load issue instead of serialising every stage
        auto finish = [&]() {
            asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
            tc_fence_before();
            mbar_arrive(&fullA[psa]);
            if (++psa == n_a) { psa = 0; ppa ^= 1u; }
        };
#pragma unroll
        for (int d = 0; d < PD; d++)
            if (d < n_ksteps) gather(buf[d], d);
        for (int ks0 = 0; ks0 < n_ksteps; ks0 += PD) {
#pragma unroll
            for (int d = 0; d < PD; d++) {
                const int ks = ks0 + d;
                if (ks < n_ksteps) {
                    publish(buf[d]);
                    if (ks + PD < n_ksteps) gather(buf[d], ks + PD);
                    finish();
                }
            }
        }

        // ===== epilogue: TMEM -> registers -> ReLU -> Y =====
        mbar_wait(accum_bar, 0);
        tc_fence_after();
        if (tid == 128) KN_STAMP(4);
        const int half = (warp - 4) >> 2;                       // two warps per lane quarter: even / odd 16-column chunks
        const int g_valid = min(Gp, G - row0);
        const int32_t *__restrict__ rg = rows + g * (int64_t)G + row0;
#pragma unroll
        for (int b = 0; b < NB; b++) {
            const int64_t ne = nbase + b * BM + q * 32 + lane;
            for (int c0 = half * 16; c0 < Gp; c0 += 32) {
                uint32_t r[16];
                tmem_load16(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(b * Gp + c0), r);
                if (ne < n_vecs)
                    store_rows16<RELU, PEERS>(r, g_valid - c0, [&](int t) { return __ldg(rg + c0 + t); }, Y, ldy, ne, peers);
            }
        }
    }

    if (tid == 128) KN_STAMP(5);
    tc_fence_before();
    __syncthreads();
    if (tid == 0) KN_STAMP(6);
    if (CS > 1) cluster_sync_all();                              // no CTA leaves while a partner may still signal its barriers
    if (warp == 2) tmem_dealloc512(tmem_base);
}

// split of a packed value array (weights), one thread per 8 consecutive k: hi = TF32 words, corr = 4 bf16 pairs of w_lo
// then 4 of w_hi (the B operand of the kind::f16 correction MMA, against the A producers' [x_hi | x_lo])
__global__ void split_tf32_kernel(const float *__restrict__ v, int64_t n8, uint32_t *__restrict__ hi, uint32_t *__restrict__ corr) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n8) {
        const float4 *src = reinterpret_cast<const float4 *>(v) + 2 * i;
        const float4 a = src[0], b = src[1];
        const float x[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
        uint32_t h[8], c[8];
        split8_tf32_bf16(x, h, c + 4, c);
        uint4 *dh = reinterpret_cast<uint4 *>(hi) + 2 * i, *dc = reinterpret_cast<uint4 *>(corr) + 2 * i;
        dh[0] = make_uint4(h[0], h[1], h[2], h[3]); dh[1] = make_uint4(h[4], h[5], h[6], h[7]);
        dc[0] = make_uint4(c[0], c[1], c[2], c[3]); dc[1] = make_uint4(c[4], c[5], c[6], c[7]);
    }
}

typedef CUresult (*PFN_encodeTiled)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                    const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

PFN_encodeTiled get_encode() {
    static PFN_encodeTiled fn = nullptr;
    if (!fn) {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = (PFN_encodeTiled)p;
    }
    return fn;
}

template <int NB, int CS>
int launch_tc(const CUtensorMap *maps, const int32_t *rows, const int32_t *cols, const int32_t *group_k, const int32_t *block_of, int64_t n_groups, int G, int K_pad,
              const float *X, int64_t ldx, float *Y, int64_t ldy, int64_t n_vecs, bool relu, cudaStream_t s)
{
    const int chunks_per_group = (G + 255) / 256;
    const int Gp = tc_gp(G);
    const int stage = 2 * Gp * KS * 4;
    int n_b = (int)((220 * 1024 - (int64_t)K_pad * 4) / stage);   // weight ring in shared memory, next to the column list
    if (n_b > 8) n_b = 8;
    const uint32_t a0 = (uint32_t)(NB * Gp);                     // activation ring in TMEM, after the accumulators
    int n_a = (int)((512 - a0) / (NB * 32));
    if (n_a > 6) n_a = 6;
    KN_REQUIRE(n_b >= 2 && n_a >= 2, "spmm_pg_tc: rings do not fit (Gp=%d NB=%d)", Gp, NB);
    const size_t smem = (size_t)n_b * stage + (size_t)K_pad * 4 + 1024 + 512;
    const int64_t gx = n_groups * chunks_per_group, gy = kn_cdiv(n_vecs, BM * NB);
    KN_REQUIRE(gx * gy <= 0x7fffffffLL, "spmm_pg_tc: grid too large");
    const CUtensorMap *m = maps + (CS > 1 ? 2 : 0);              // maps[2..3]: boxes of Gp/2 rows for the multicast halves
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(gx * gy));
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CS; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    const KnPeers peers = kn_current_peers();
    return dispatch_relu_peers(relu, peers.n > 0, [&](auto R, auto P) {
        const auto kfn = pg_tc_kernel<NB, decltype(R)::value, CS, decltype(P)::value>;
        KN_ONCE_PER_DEVICE { KN_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024)); }
        KN_CUDA(cudaLaunchKernelEx(&cfg, kfn, m[0], m[1], rows, cols, group_k, block_of, G, Gp, K_pad, chunks_per_group, gx, gy, n_b, n_a, a0,
                                   kSuperTiles / NB, X, ldx, Y, ldy, n_vecs, peers));
        return KN_OK;
    });
}

// cluster of 2 along the batch-tile axis whenever the tiles pair up inside a raster super-tile: an even number of batch
// tiles does, as a super-tile holds an even number of them
static_assert((kSuperTiles / 2) % 2 == 0, "kSuperTiles / NB must be even");
template <int NB>
int launch_tc_auto(const CUtensorMap *maps, const int32_t *rows, const int32_t *cols, const int32_t *group_k, const int32_t *block_of, int64_t n_groups, int G, int K_pad,
                   const float *X, int64_t ldx, float *Y, int64_t ldy, int64_t n_vecs, bool relu, cudaStream_t s)
{
    if (kn_cdiv(n_vecs, BM * NB) % 2 == 0) return launch_tc<NB, 2>(maps, rows, cols, group_k, block_of, n_groups, G, K_pad, X, ldx, Y, ldy, n_vecs, relu, s);
    return launch_tc<NB, 1>(maps, rows, cols, group_k, block_of, n_groups, G, K_pad, X, ldx, Y, ldy, n_vecs, relu, s);
}
}  // namespace

KN_API int kn_pg_tc_split(const float *vals, int64_t n, float *vals_hi, float *vals_corr, void *stream) {
    KN_REQUIRE(n >= 0 && n % 8 == 0, "pg_tc_split: length must be a non-negative multiple of 8");
    if (n == 0) return KN_OK;
    KN_REQUIRE(vals && vals_hi && vals_corr, "pg_tc_split: null pointer");
    KN_REQUIRE((((uintptr_t)vals | (uintptr_t)vals_hi | (uintptr_t)vals_corr) & 15) == 0, "pg_tc_split: arrays must be 16-byte aligned");
    split_tf32_kernel<<<(unsigned)kn_cdiv(n / 8, 256), 256, 0, (cudaStream_t)stream>>>(vals, n / 8, reinterpret_cast<uint32_t *>(vals_hi),
                                                                                     reinterpret_cast<uint32_t *>(vals_corr));
    KN_CHECK_LAUNCH();
    return KN_OK;
}

KN_API int kn_pg_tc_tensormaps(const float *vals_hi, const float *vals_corr, int64_t n_rows_total, int32_t G, int32_t K_pad, void *maps_out_host) {
    KN_REQUIRE(vals_hi && vals_corr && maps_out_host, "pg_tc_tensormaps: null pointer");
    KN_REQUIRE(n_rows_total > 0 && G > 0 && K_pad > 0 && K_pad % KS == 0, "pg_tc_tensormaps: bad shape");
    PFN_encodeTiled enc = get_encode();
    if (!enc) { kn_set_error("cuTensorMapEncodeTiled is not available from this driver"); return KN_ERR_UNSUPPORTED; }
    const int Gp = tc_gp(G);
    const float *planes[4] = {vals_hi, vals_corr, vals_hi, vals_corr};
    for (int i = 0; i < 4; i++) {
        CUtensorMap m;                                         // 64-byte aligned local; the caller's buffer need not be
        cuuint64_t dims[2] = {(cuuint64_t)K_pad, (cuuint64_t)n_rows_total};
        cuuint64_t strides[1] = {(cuuint64_t)K_pad * sizeof(float)};
        cuuint32_t box[2] = {(cuuint32_t)KS, (cuuint32_t)(i < 2 ? Gp : Gp / 2)};   // maps 2,3: half boxes for 2-CTA multicast
        cuuint32_t estr[2] = {1, 1};
        CUresult r = enc(&m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void *)planes[i], dims, strides, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) { kn_set_error("cuTensorMapEncodeTiled failed (%d)", (int)r); return KN_ERR_CUDA; }
        memcpy(reinterpret_cast<unsigned char *>(maps_out_host) + i * sizeof(CUtensorMap), &m, sizeof(CUtensorMap));
    }
    return KN_OK;
}

KN_API int kn_spmm_pg_tc_f32(const void *maps_host, const int32_t *rows, const int32_t *cols, const int32_t *group_k, const int32_t *block_of, int64_t n_groups, int32_t G, int32_t K_pad,
                             const float *X, int64_t ldx, float *Y, int64_t ldy, int64_t n_vecs, uint32_t flags, const kn_peers *peers_arg, void *stream) {
    KnPeersScope peers_scope(peers_arg);
    if (!peers_scope.ok) return KN_ERR_INVALID_ARGUMENT;
    KN_REQUIRE(n_groups >= 0 && G > 0 && K_pad > 0 && K_pad % KS == 0, "spmm_pg_tc: bad shape (G=%d K_pad=%d)", G, K_pad);
    KN_REQUIRE(n_vecs >= 0 && ldx >= n_vecs && ldy >= n_vecs, "spmm_pg_tc: bad leading dimension");
    if (n_groups == 0 || n_vecs == 0) return KN_OK;
    KN_REQUIRE(maps_host && rows && cols && X && Y, "spmm_pg_tc: null pointer");
    KN_REQUIRE(n_vecs % 4 == 0 && ldx % 4 == 0 && (((uintptr_t)X) & 15) == 0, "spmm_pg_tc: n_vecs and ldx must be multiples of 4, X 16-byte aligned");
    KN_REQUIRE(ldx * 4 < 0xffffffffLL, "spmm_pg_tc: leading dimension in bytes must fit 32 bits");
    CUtensorMap maps[4];
    memcpy(maps, maps_host, 4 * sizeof(CUtensorMap));
    const bool relu = (flags & KN_SPMM_RELU) != 0;
    // two batch tiles per CTA share every weight stage when accumulators + a >= 2-deep activation ring fit TMEM
    if (2 * tc_gp(G) + 2 * 64 <= 512 && n_vecs > BM)
        return launch_tc_auto<2>(maps, rows, cols, group_k, block_of, n_groups, G, K_pad, X, ldx, Y, ldy, n_vecs, relu, (cudaStream_t)stream);
    return launch_tc_auto<1>(maps, rows, cols, group_k, block_of, n_groups, G, K_pad, X, ldx, Y, ldy, n_vecs, relu, (cudaStream_t)stream);
}

// debug: select the CTA whose phase timestamps are recorded (-1 = none) / read them back (7 x clock64)
KN_API int kn_debug_tc_timing(int32_t cta, int64_t *out_host) {
    if (out_host) {
        long long t[8];
        KN_CUDA(cudaMemcpyFromSymbol(t, g_tc_timing, sizeof(t)));
        for (int i = 0; i < 8; i++) out_host[i] = (int64_t)t[i];
    }
    int c = cta;
    KN_CUDA(cudaMemcpyToSymbol(g_tc_timing_cta, &c, sizeof(int)));
    return KN_OK;
}
