// pgtile_tc.cu -- spatially tiled tensor-core kernel for keyed convolution layers with few output channels (G <= 128).
//
// pgroup_tc.cu runs one output pixel per CTA: for every 16-k stage it pulls 8 KB of gathered activations AND the pixel's
// weight slab (hi + corr planes) from L2.  For G <= 128 that is ~64 B/clk/SM at full tensor rate, ~9.5 KB/clk over the chip,
// against an L2 throughput cap of ~6.3 KB/clk: measured 49 % (G = 64) / 62 % (G = 128) of the tensor ceiling of the former
// 3xTF32 split (3 tf32 MMAs per 8 k), i.e.
// those layers are bound by L2 -> SM traffic, not by the tensor pipe (VGG16 conv1_2 / conv2_x, AllConvNet conv2 / conv3).
//
// Here one CTA owns a TILE of th x tw neighbouring output pixels (2x2 for G <= 96, 1x2 for G <= 128) x 128 batch columns:
//   * the union of the tile's input positions ((th-1)*stride+P) x ((tw-1)*stride+Q) is gathered ONCE per 16-channel chunk:
//     a 3x3 / stride-1 2x2 tile reads 16 positions instead of 4 x 9 = 36 (each gathered stage feeds up to 4 pixels' MMAs);
//   * under permutation-only keys every pixel multiplies the SAME weight matrix, so the P*Q tap slabs of a channel chunk
//     are loaded ONCE per chunk by TMA into a slab ring and reused by every pixel of the tile at its own position
//     (tap of pixel t at union position p = p - t*stride); taps that fall outside the image are simply not issued;
//   * every pixel has its own fp32 accumulator in TMEM.  With stride 1 the pixels of one tile ROW that use a gathered position
//     read CONSECUTIVE taps of one tap row (pixel tx at union column px uses tap dx = px - tx), so with the accumulators of a
//     row laid out in descending tx and the hi (corr) planes of the tap slabs contiguous in shared memory, ONE tcgen05.mma of
//     N = (pixels in the run) x Gp multiplies the stage by all of them (N = 128 .. 256 instead of 64 .. 128);
//   * issuers are elected threads (kn_tc::elect_one -- under `if (lane == 0)` every tcgen05.mma cost 127-143 cycles of an
//     ELECT / R2UR loop, under elect.sync one thread issues at the pipe rate), and an issuer is ONE thread running ~4-6 cycles
//     per dependent scalar instruction, so what counts is instructions per issuer and stage: every tile row has two issuers,
//     one per 8-k half of the 16-k stage, both accumulating into the row's accumulators (zeroed up front: no issuer owns the
//     first write); what an issuer does at a position is a host-built record (kernel parameter), and for the 3x3 / stride-1
//     geometries the whole schedule is folded at compile time (issuer_fast).  A slab is waited for once and released once
//     per chunk and issuer (first / last use), not per use.  Other strides: one issuer and one instruction per (pixel, tap);
//   * gathers: seven warps, cp.async 16 B per lane into a raw shared-memory ring that completes on mbarriers (16 stages =
//     128 KB in flight towards the SM for G = 64); two splitter groups (hi / corr split -> tcgen05.st) on alternate stages;
//   * output rows are transposed through the (by then idle) gather ring and leave as 512-byte cp.async.bulk rows;
//   * A operand (gathered activations, split in registers) in a TMEM ring exactly as in pgroup_tc.cu, and the same split:
//     per 8 k x_hi.w_hi (kind::tf32) + [x_hi | x_lo].[w_lo ; w_hi] (kind::f16 in bf16) into one fp32 accumulator
//     (tc_common.cuh); bias as one extra stage reading the homogeneous row.
// L2 -> SM bytes per (pixel, 16-channel chunk): G = 64: 108 KB -> 50 KB, G = 96: 126 -> 59, G = 128: 216 -> 120.
//
// Weight layout (built by the host): Wt[G][K_pad] TAP-major, k = tap * C + c, bias at k = n_taps * C, zero padded to a
// multiple of 16; hi (TF32) / corr (bf16 pairs) planes + TMA descriptors with boxes of 16 words x Gp rows (kn_pg_tc_split /
// kn_pg_tc_tensormaps).
// Tile tables (kn_conv2d_tiles_index): cols[tile][position][C] = activation row of every (position, channel) under the
// layer's input key (-1 = position outside the image), rows[tile][pixel][G] = output row of every (pixel, channel).
#include "tc_common.cuh"
#include <string.h>

namespace {
using namespace kn_tc;

constexpr int kGatherWarps = 7;
constexpr int kProducerWarp0 = 12;     // first splitter warp: a multiple of 4 (a warp reaches the TMEM lanes of its quarter, warp % 4)
constexpr int kThreads = (kProducerWarp0 + 8) * 32;   // warp 0: TMA (weight slabs)  warps 1-4: MMA issuers  warps 5..: activation gathers (cp.async; warp 7 first allocates TMEM)  warps 12-19: hi/lo splitters + epilogue
constexpr int kGroupThreads = 128;     // the 8 splitter warps work as two groups of 4 (one warp per TMEM lane quarter) on alternate stages
constexpr int kMaxT = 4;               // output pixels per tile (issuer warps 1-4)
constexpr int kGatherWarp0 = 5;        // warps 5 .. 5 + kGatherWarps - 1: activation gathers (stages round-robin)
static_assert(kGatherWarp0 + kGatherWarps <= kProducerWarp0, "gather warps overlap the splitters");
constexpr int kMaxPos = 32;            // union positions per tile
constexpr int kBiasPos = 255;
constexpr int kRawStageBytes = KS * BM * 4;      // one gathered stage: 16 rows x 128 batch columns, fp32

#ifdef KN_TILE_PROF
__device__ long long g_tile_prof[64];
// fine-grained regions cost ~40 cycles each and perturb the loops they sit in: KN_TILE_PROF is a MASK of the slots to record
// (bit s / 10 of the mask enables slots 10 s .. 10 s + 9; -DKN_TILE_PROF=1 records only the phase stamps)
#define PROF_T0(slot) const long long pt0_ = ((KN_TILE_PROF >> ((slot) / 10)) & 1) ? clock64() : 0
#define PROF_ADD(slot) do { if (((KN_TILE_PROF >> ((slot) / 10)) & 1) && blockIdx.x == 5000) atomicAdd((unsigned long long *)&g_tile_prof[slot], (unsigned long long)(clock64() - pt0_)); } while (0)
#define PROF_SET(slot) do { if (blockIdx.x == 5000) g_tile_prof[slot] = clock64(); } while (0)
#else
#define PROF_T0(slot)
#define PROF_ADD(slot)
#define PROF_SET(slot)
#endif

struct TileGeom {
    int C, G, Gp, th, tw, T, stride, P, Q, n_taps, uh, uw, U_pos, n_chunks;
    int n_slots, n_a, n_raw;           // weight-slab ring (shared memory), activation ring (TMEM) and raw gather ring (shared memory) depths
    int n_iss, merged, ksplit;         // MMA issuer threads: ksplit per tile row issuing merged runs (stride 1), or one per pixel
    int bulk_epi, epi_pixels;          // epilogue through shared memory + bulk copies: pixels per pass (0 = per-lane stores)
    uint32_t a0;                       // first TMEM column of the activation ring (after the T accumulators)
    int slab_bytes, plane_bytes;
};

// What every issuer does at every union position (issued in raster order) -- geometry only, the same for every tile, so it is
// built on the host and travels as a kernel parameter (constant bank: a uniform load in the issuers' loop):
//   x: bit 1 this issuer has MMAs here | bit 2 last use of slab (x >> 8 & 255) in the chunk | first accumulator column << 16
//   y: taps read (bit per slab)      z: B descriptor offset (slot = tap)      w: instruction descriptor
struct TileJobs { int4 rec[kMaxT * kMaxPos]; };

// Issuer loop for the common geometries (3x3 taps, stride 1, merged runs, two issuers per tile row), everything that only
// depends on the geometry folded at compile time.  An issuer is ONE thread: at ~4-6 cycles per dependent scalar instruction
// the ~90 instructions per stage of the table-driven loop (record load, bit tests, descriptor arithmetic, ring bookkeeping)
// were 565 cycles per stage against 523 cycles of tensor pipe -- the issuers, not the pipe, set the pace.  Interior tiles
// (every position inside the image) take this path; border tiles the generic loop.
template <int TH, int TW, int GP, int ROW, int KK0>
__device__ __forceinline__ void issuer_fast(int n_chunks, int n_a, uint32_t tmem_base, uint32_t a_base, uint64_t desc0,
                                            uint64_t *fullA, uint64_t *emptyA, uint64_t *fullB, uint64_t *emptyB, int &sa, uint32_t &pa)
{
    constexpr int UW = TW + 2, UH = TH + 2;
    constexpr uint64_t corr_off = (uint64_t)((9u * GP * 64u) >> 4);         // 9 slots (slot = tap) of hi planes, then the corr planes
    for (int cc = 0; cc < n_chunks; cc++) {
        const uint32_t pb = (uint32_t)(cc & 1);
#pragma unroll
        for (int o = 0; o < UH * UW; o++) {
            const int py = o / UW, px = o % UW, dy = py - ROW;
            const int tx_hi = px < TW - 1 ? px : TW - 1, tx_lo = px - 2 > 0 ? px - 2 : 0;
            if (dy >= 0 && dy < 3 && tx_hi >= tx_lo) {
                const int tap0 = dy * 3 + (px - tx_hi), m = tx_hi - tx_lo + 1, acc0 = ROW * TW + (TW - 1 - tx_hi);
                if (px < 3) mbar_wait(&fullB[dy * 3 + px], pb);            // the one slab first read here (pixel 0's tap); the others were read before
                mbar_wait(&fullA[sa], pa);
                tc_fence_after();
                const uint32_t d = tmem_base + (uint32_t)(acc0 * GP);
                const uint32_t ta = a_base + (uint32_t)(sa * 32 + KK0 * 8);
                const uint64_t db_hi = desc0 + (uint64_t)((((uint32_t)tap0 * GP * 64u) >> 4) + KK0 * 2);
                constexpr uint32_t dummy = 0; (void)dummy;
                umma_tf32_ts(d, ta, db_hi, make_idesc_tf32(BM, m * GP), 1u);                 // x_hi . w_hi
                umma_bf16_ts(d, ta + 16, db_hi + corr_off, make_idesc_bf16(BM, m * GP), 1u); // x_hi . w_lo + x_lo . w_hi
                if (tx_hi == TW - 1) umma_commit(&emptyB[tap0]);            // last use of this slab by this issuer in this chunk
                umma_commit(&emptyA[sa]);
            } else {
                mbar_wait(&fullA[sa], pa);
                mbar_arrive(&emptyA[sa]);
            }
            if (++sa == n_a) { sa = 0; pa ^= 1u; }
        }
    }
}

template <bool RELU, bool PEERS, int TH, int TW, int GP>
__global__ void __launch_bounds__(kThreads, 1)
pg_tile_tc_kernel(const __grid_constant__ CUtensorMap map_hi, const __grid_constant__ CUtensorMap map_corr,
                  const int32_t *__restrict__ tile_cols, const int32_t *__restrict__ tile_rows, int32_t bias_col,
                  const TileGeom geo, const __grid_constant__ TileJobs jobs_tab, int64_t n_sp_tiles, int64_t n_btiles, int super_tiles,
                  const float *__restrict__ X, int64_t ldx, float *__restrict__ Y, int64_t ldy, int64_t n_vecs, const __grid_constant__ KnPeers peers)
{
    extern __shared__ unsigned char smem_dyn[];
    unsigned char *smem = reinterpret_cast<unsigned char *>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023) & ~(uintptr_t)1023);
    float *s_raw = reinterpret_cast<float *>(smem + (size_t)geo.n_slots * geo.slab_bytes);          // [n_raw][16 rows][128 batch] gathered fp32
    unsigned char *sp = smem + (size_t)geo.n_slots * geo.slab_bytes + (size_t)geo.n_raw * kRawStageBytes;
    int32_t *s_cols = reinterpret_cast<int32_t *>(sp);                      sp += (size_t)geo.U_pos * geo.C * 4;
    int32_t *s_rows = reinterpret_cast<int32_t *>(sp);                      sp += (size_t)kMaxT * 256 * 4;         // [t][G] output rows of the tile
    uint64_t *fullB = reinterpret_cast<uint64_t *>(sp);
    uint64_t *emptyB = fullB + geo.n_slots;
    uint64_t *fullA = emptyB + geo.n_slots;
    uint64_t *emptyA = fullA + geo.n_a;
    uint64_t *raw_full = emptyA + geo.n_a;
    uint64_t *raw_empty = raw_full + geo.n_raw;
    uint64_t *accum_bar = raw_empty + geo.n_raw;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(accum_bar + 1);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (tid == 0) PROF_SET(0);
    const KnRaster rt = kn_raster(blockIdx.x, n_sp_tiles, n_btiles, super_tiles);
    const int64_t tile = rt.item;
    const int64_t nbase = rt.tile * BM;
    const int T = geo.T, C = geo.C, Gp = geo.Gp, U_pos = geo.U_pos;

    if (warp == 0 && lane == 0) {
        for (int s = 0; s < geo.n_slots; s++) { mbar_init(&fullB[s], 1); mbar_init(&emptyB[s], geo.n_iss); }
        for (int s = 0; s < geo.n_a; s++) { mbar_init(&fullA[s], kGroupThreads); mbar_init(&emptyA[s], geo.n_iss); }
        for (int s = 0; s < geo.n_raw; s++) { mbar_init(&raw_full[s], 32); mbar_init(&raw_empty[s], kGroupThreads); }
        mbar_init(accum_bar, geo.n_iss);
        fence_barrier_init();
    } else if (warp == 7) {
        tmem_alloc512(tmem_slot);
    }
    // the tile's gather table and output rows: ONE global round trip and one barrier before every role starts (the stage list and
    // the issuers' records used to be built here behind a second barrier: 7 k cycles of prologue with the tensor pipe idle)
    const int32_t *__restrict__ tc = tile_cols + tile * (int64_t)U_pos * C;
    for (int i = tid; i < U_pos * C; i += kThreads) s_cols[i] = __ldg(tc + i);
    for (int i = tid; i < T * geo.G; i += kThreads) s_rows[(i / geo.G) * 256 + (i % geo.G)] = __ldg(tile_rows + tile * (int64_t)T * geo.G + i);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    unsigned vmask = 0;                                       // bit p: union position p lies inside the image
    for (int p = 0; p < U_pos; p++) vmask |= (s_cols[p * C] >= 0 ? 1u : 0u) << p;
    const int n_stages = geo.n_chunks * __popc(vmask) + 1;    // in-image (chunk, position) stages + the bias stage
    if (tid == 0) PROF_SET(1);
    const int n_slabs = geo.n_chunks * geo.n_taps + 1;

    if (warp == 0) {
        // ===== TMA producer: weight slabs (chunk, tap) in order, then the bias slab =====
        if (elect_one()) {
            int s = 0; uint32_t ph = 0;
            for (int j = 0; j < n_slabs; j++) {
                const int cc = j / geo.n_taps, tap = j - cc * geo.n_taps;
                const int k0 = (j == n_slabs - 1) ? geo.n_taps * C : tap * C + cc * KS;
                mbar_wait(&emptyB[s], ph ^ 1u);
                unsigned char *bs = smem + (size_t)s * geo.plane_bytes;             // hi planes of all slots, then corr planes: consecutive taps are contiguous
                mbar_arrive_expect_tx(&fullB[s], (uint32_t)geo.slab_bytes);
                tma_load_2d(bs, &map_hi, k0, 0, &fullB[s]);
                tma_load_2d(bs + (size_t)geo.n_slots * geo.plane_bytes, &map_corr, k0, 0, &fullB[s]);
                if (++s == geo.n_slots) { s = 0; ph ^= 1u; }
            }
        }
    } else if (warp >= 1 && warp <= kMaxT) {
        // ===== MMA issuers: one elected thread per tile row (merged runs) or per output pixel =====
        const int w = warp - 1;
        if (w < geo.n_iss && elect_one()) {
            const uint64_t desc0 = make_desc(smem_u32(smem), 16, 512, kLayoutSW64);
            const uint64_t corr_off = (uint64_t)(((uint32_t)geo.n_slots * (uint32_t)geo.plane_bytes) >> 4);
            const int kk0 = w % geo.ksplit;                         // this issuer's 8-k steps of a stage: kk0, kk0 + ksplit, ...
            const uint32_t a_base = tmem_base + geo.a0;
            const int4 *jobs = jobs_tab.rec + w * kMaxPos;
            int sa = 0; uint32_t pa = 0;
            auto issue = [&](uint32_t d, uint64_t dslab, uint32_t idesc) {     // every accumulator was zeroed by the splitters: always accumulate
                const uint32_t ta = a_base + (uint32_t)(sa * 32);
                const uint32_t idesc_c = idesc_tf32_to_bf16(idesc);
                for (int kk = kk0; kk < KS / 8; kk += geo.ksplit) {
                    const uint64_t db_hi = dslab + (uint64_t)(kk * 2);
                    umma_tf32_ts(d, ta + kk * 8, db_hi, idesc, 1u);                // x_hi . w_hi
                    umma_bf16_ts(d, ta + 16 + kk * 8, db_hi + corr_off, idesc_c, 1u);   // x_hi . w_lo + x_lo . w_hi
                }
            };
            bool fast = false;
            if constexpr (TH > 0) {
                if (vmask == (1u << ((TH + 2) * (TW + 2))) - 1u) {      // interior tile
                    fast = true;
                    switch (w) {
                    case 0: issuer_fast<TH, TW, GP, 0, 0>(geo.n_chunks, geo.n_a, tmem_base, a_base, desc0, fullA, emptyA, fullB, emptyB, sa, pa); break;
                    case 1: issuer_fast<TH, TW, GP, 0, 1>(geo.n_chunks, geo.n_a, tmem_base, a_base, desc0, fullA, emptyA, fullB, emptyB, sa, pa); break;
                    case 2: if constexpr (TH > 1) issuer_fast<TH, TW, GP, 1, 0>(geo.n_chunks, geo.n_a, tmem_base, a_base, desc0, fullA, emptyA, fullB, emptyB, sa, pa); break;
                    default: if constexpr (TH > 1) issuer_fast<TH, TW, GP, 1, 1>(geo.n_chunks, geo.n_a, tmem_base, a_base, desc0, fullA, emptyA, fullB, emptyB, sa, pa); break;
                    }
                }
            }
            for (int cc = 0; cc < (fast ? 0 : geo.n_chunks); cc++) {
                uint32_t waited = 0;                                // slabs of this chunk this issuer has already waited for
                const uint32_t pb = (uint32_t)(cc & 1);            // slot = tap: a slab's slot is in its cc-th use
                for (int o = 0; o < U_pos; o++) {
#ifdef KN_TILE_PROF
                    const long long it0_ = clock64();
#endif
                    const int4 r = jobs[o];
                    if ((vmask >> o) & 1u) {
                        if (r.x & 2) {
                            uint32_t need = (uint32_t)r.y & ~waited;
                            while (need) { const int t = __ffs(need) - 1; need &= need - 1u; PROF_T0(10); mbar_wait(&fullB[t], pb); if (w == 0) PROF_ADD(10); }
                            waited |= (uint32_t)r.y;
                        }
                        { PROF_T0(11); mbar_wait(&fullA[sa], pa); if (w == 0) PROF_ADD(11); }
                        tc_fence_after();
                        if (r.x & 2) {
                            { PROF_T0(12); issue(tmem_base + ((uint32_t)r.x >> 16), desc0 + (uint64_t)(uint32_t)r.z, (uint32_t)r.w); if (w == 0) PROF_ADD(12); }
                            PROF_T0(14);
                            if (r.x & 4) umma_commit(&emptyB[(r.x >> 8) & 255]);       // last use of this slab by this issuer in this chunk (waited for above)
                            umma_commit(&emptyA[sa]);
                            if (w == 0) PROF_ADD(14);
                        } else {
                            mbar_arrive(&emptyA[sa]);                                  // a position this issuer's pixels do not read
                        }
                        if (++sa == geo.n_a) { sa = 0; pa ^= 1u; }
#ifdef KN_TILE_PROF
                        if (w == 0 && blockIdx.x == 5000) atomicAdd((unsigned long long *)&g_tile_prof[16], (unsigned long long)(clock64() - it0_));
#endif
                    } else if (r.x & 4) {
                        // position outside the image: the slab's last use does not happen, release it after the earlier ones.  A slab
                        // is never released before its load has landed (border tiles may not read it at all): the ring's phases
                        // stay in step and no bulk copy is in flight when the CTA exits
                        const int t = (r.x >> 8) & 255;
                        if (!((waited >> t) & 1u)) { mbar_wait(&fullB[t], pb); waited |= 1u << t; }
                        umma_commit(&emptyB[t]);
                    }
                }
            }
            {   // bias stage: every pixel of this issuer reads the one bias slab (slot 0 in its n_chunks-th use)
                mbar_wait(&fullB[0], (uint32_t)(geo.n_chunks & 1));
                mbar_wait(&fullA[sa], pa);
                tc_fence_after();
                const int n_acc = geo.merged ? geo.tw : 1;
                for (int a = 0; a < n_acc; a++) issue(tmem_base + (uint32_t)(((w / geo.ksplit) * n_acc + a) * Gp), desc0, make_idesc_tf32(BM, Gp));
                umma_commit(&emptyB[0]);
                umma_commit(&emptyA[sa]);
            }
            umma_commit(accum_bar);
            if (w == 0) PROF_SET(2);
        }
    } else if (warp >= kGatherWarp0 && warp < kGatherWarp0 + kGatherWarps) {
        // ===== gather warps (alternate stages): X rows of every (position, channel chunk) stage into the raw ring, cp.async 16 B per lane =====
        // One warp instruction copies one 512 B row segment; the 16 rows of a stage complete on the stage's mbarrier
        // (cp.async.mbarrier.arrive.noinc from every lane).  Up to n_raw stages (8 KB each) are in flight towards this SM,
        // independent of the splitters' progress.  (Register prefetch -- ld.global into a ring of registers -- ran ONE stage
        // per memory latency, and a lock-step copy / split loop ~1500 cycles per stage: both far below the tensor pipe.)
        const int64_t ncol = nbase + lane * 4;                  // first batch column of this lane's 16-byte chunk
        const bool col_ok = ncol < n_vecs;                      // n_vecs % 4 == 0: a chunk is entirely inside or outside
        const float *__restrict__ xcol = X + (col_ok ? ncol : 0);
        const int bytes = col_ok ? 16 : 0;                      // src-size 0 => 16 bytes of zeros
        const int mine = warp - kGatherWarp0;
        // A warp waits for its slot by parity only, which is sound while the slot's previous lap has been consumed: with g
        // warps taking turns, a warp's previous stage waited for the consumption of stage i - g - n_raw, so g <= n_raw
        // gather warps at most (a 6-stage ring under 7 warps overwrote unconsumed stages and hung: G = 128, C = 512).
        const int n_gw = geo.n_raw < kGatherWarps ? geo.n_raw : kGatherWarps;
        int i = -1, cc = 0, p = -1;                              // stage counter and its (chunk, union position)
        int slot = -1, turn = n_gw - 1; uint32_t rph = 1u;       // the stage's ring slot / the parity its raw_empty is waited with / whose turn it is
        while (mine < n_gw) {
            // next in-image stage, chunk-major; after the last chunk the bias stage (ring position kept incrementally: a runtime
            // division per stage is ~150 cycles of a gather warp's ~460)
            ++i;
            if (++slot == geo.n_raw) { slot = 0; rph ^= 1u; }
            if (++turn == n_gw) turn = 0;
            if (i == n_stages - 1) p = kBiasPos;
            else if (i >= n_stages) break;
            else do { if (++p == U_pos) { p = 0; ++cc; } } while (!((vmask >> p) & 1u));
            if (turn != mine) continue;
            { PROF_T0(30); mbar_wait(&raw_empty[slot], rph); if (tid == kGatherWarp0 * 32) PROF_ADD(30); }
            PROF_T0(31);
            float *dst = s_raw + (size_t)slot * (KS * BM) + lane * 4;
            // the 16 row indices first (4 x LDS.128), then 16 back-to-back copies: an index load in front of every copy
            // serialised the warp at ~75 cycles per copy (1200 cycles per stage, measured) instead of the LSU's ~8
            int32_t cidx[KS];
            if (p == kBiasPos) {
#pragma unroll
                for (int r = 0; r < KS; r++) cidx[r] = bias_col;
            } else {
                const int4 *cp4 = reinterpret_cast<const int4 *>(s_cols + p * C + cc * KS);     // 64-byte aligned: C % 16 == 0
#pragma unroll
                for (int r4 = 0; r4 < KS / 4; r4++) {
                    const int4 c = cp4[r4];
                    cidx[4 * r4 + 0] = c.x; cidx[4 * r4 + 1] = c.y; cidx[4 * r4 + 2] = c.z; cidx[4 * r4 + 3] = c.w;
                }
            }
            const uint32_t d32 = smem_u32(dst);
#pragma unroll
            for (int r = 0; r < KS; r++) {
                const float *src = xcol + (int64_t)cidx[r] * ldx;
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" :: "r"(d32 + (uint32_t)(r * BM * 4)), "l"(src), "r"(bytes));
            }
            asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];\n" :: "r"(smem_u32(&raw_full[slot])) : "memory");
            if (tid == kGatherWarp0 * 32) PROF_ADD(31);
        }
        asm volatile("cp.async.wait_all;\n" ::: "memory");
    } else if (warp >= kProducerWarp0) {
        // ===== splitters: raw stage -> TF32 hi / bf16 corr words -> tcgen05.st into the TMEM ring =====
        // two groups of four warps (one warp per TMEM lane quarter) take alternate stages, so the fixed latencies of one
        // stage's chain (barrier wait, shared-memory reads, TMEM store + wait, arrive) overlap with the other group's stage
        const int q = warp & 3;                                 // TMEM lane quarter
        const int sel = (warp - kProducerWarp0) >> 2;           // splitter group
        const float *src0 = s_raw + q * 32 + lane;
        if (sel == 0) {                                         // zero the accumulators (ordered before the first MMA by fullA[0], which this group completes)
            uint32_t z[16];
#pragma unroll
            for (int j = 0; j < 16; j++) z[j] = 0u;
            for (int c0 = 0; c0 < T * Gp; c0 += 16) tmem_store<16>(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)c0, z);
        }
        int slot = sel - 2, sa = sel - 2; uint32_t rph = 0, aph = 1u;       // ring positions of this group's stages, kept incrementally (n_raw >= 3, n_a >= 2)
        for (int i = sel; i < n_stages; i += 2) {
            slot += 2; if (slot >= geo.n_raw) { slot -= geo.n_raw; rph ^= 1u; }
            sa += 2; if (sa >= geo.n_a) { sa -= geo.n_a; aph ^= 1u; }
            { PROF_T0(20); mbar_wait(&raw_full[slot], rph); if (tid == kProducerWarp0 * 32) PROF_ADD(20); }
            const float *src = src0 + (size_t)slot * (KS * BM);
            uint32_t hi[KS], corr[KS];                          // corr: per 8 k, 4 bf16 x_hi pairs then 4 bf16 x_lo pairs
            { PROF_T0(21);
            float v[KS];
#pragma unroll
            for (int j = 0; j < KS; j++) v[j] = src[j * BM];
#pragma unroll
            for (int h = 0; h < KS / 8; h++) split8_tf32_bf16(v + 8 * h, hi + 8 * h, corr + 8 * h, corr + 8 * h + 4);
            mbar_arrive(&raw_empty[slot]);                      // the values are in registers: the slot can be refilled
            if (tid == kProducerWarp0 * 32) PROF_ADD(21); }
            { PROF_T0(23); mbar_wait(&emptyA[sa], aph); if (tid == kProducerWarp0 * 32) PROF_ADD(23); }
            tc_fence_after();
            PROF_T0(24);
            const uint32_t ta = tmem_base + ((uint32_t)(q * 32) << 16) + geo.a0 + (uint32_t)(sa * 32);
            tmem_store<KS>(ta, hi);
            tmem_store<KS>(ta + 16, corr);
            asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
            tc_fence_before();
            mbar_arrive(&fullA[sa]);
            if (tid == kProducerWarp0 * 32) PROF_ADD(24);
        }
        if (tid == kProducerWarp0 * 32) PROF_SET(3);

        // ===== epilogue: TMEM -> registers -> ReLU -> Y rows of every pixel of the tile =====
        mbar_wait(accum_bar, 0);
        tc_fence_after();
        if (tid == kProducerWarp0 * 32) PROF_SET(4);
        const int half = sel;                                    // two warps per lane quarter: even / odd 16-column chunks
        const int64_t ne = nbase + q * 32 + lane;
        const uint32_t t_lanes = tmem_base + ((uint32_t)(q * 32) << 16);
        // accumulator of pixel t: those of a tile row are in descending tx (merged runs)
        auto acc_of = [&](int t) { return geo.merged ? (t / geo.tw) * geo.tw + (geo.tw - 1 - t % geo.tw) : t; };
        if (!PEERS && geo.bulk_epi) {
            // Output rows through shared memory and bulk copies.  With per-lane stores (below) a warp instruction writes one
            // 128-byte piece of a row and the SM's queue of outstanding stores, not bandwidth, set the pace: 128 KB per CTA took
            // ~10 k cycles (70 per STG, measured), a sixth of the CTA, with nothing else to run on the SM.  Here the accumulators
            // are transposed into [row][128 batch columns] in the (now idle) gather ring, and every row leaves as ONE 512-byte
            // cp.async.bulk; the CTA only waits until shared memory has been read, not until the writes have landed.
            float *stage = s_raw;
            const int e = tid - kProducerWarp0 * 32;             // 0 .. 255
            const int ppp = geo.epi_pixels;                      // pixels per pass (what fits the ring)
            const uint32_t row_bytes = (uint32_t)((n_vecs - nbase < BM ? n_vecs - nbase : BM) * 4);
            for (int t0 = 0; t0 < T; t0 += ppp) {
                const int tn = (T - t0 < ppp) ? T - t0 : ppp;
                asm volatile("bar.sync 1, 256;" ::: "memory");  // the ring is idle (both splitter groups done) / the previous pass has been read
                for (int tl = 0; tl < tn; tl++) {
                    const int acc = acc_of(t0 + tl);
                    for (int c0 = half * 16; c0 < Gp; c0 += 32) {
                        uint32_t r[16];
                        tmem_load16(t_lanes + (uint32_t)(acc * Gp + c0), r);
                        float *dst = stage + (size_t)(tl * geo.G + c0) * BM + q * 32 + lane;
#pragma unroll
                        for (int j = 0; j < 16; j++) {
                            if (c0 + j < geo.G) {
                                float y = __uint_as_float(r[j]);
                                if (RELU) y = fmaxf(y, 0.0f);
                                dst[j * BM] = y;
                            }
                        }
                    }
                }
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");      // generic-proxy writes -> visible to the bulk copies
                asm volatile("bar.sync 1, 256;" ::: "memory");
                for (int i = e; i < tn * geo.G; i += 256) {
                    const int tl = i / geo.G, c = i - tl * geo.G;
                    float *gdst = Y + (int64_t)s_rows[(t0 + tl) * 256 + c] * ldy + nbase;
                    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                                 :: "l"(gdst), "r"(smem_u32(stage + (size_t)i * BM)), "r"(row_bytes) : "memory");
                }
                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
            }
        } else
        for (int t = 0; t < T; t++) {
            const int32_t *rg = s_rows + t * 256;
            const int acc = acc_of(t);
            for (int c0 = half * 16; c0 < Gp; c0 += 32) {
                uint32_t r[16];
                { PROF_T0(40); tmem_load16(t_lanes + (uint32_t)(acc * Gp + c0), r); if (tid == kProducerWarp0 * 32) PROF_ADD(40); }
                PROF_T0(41);
                if (ne < n_vecs) store_rows16<RELU, PEERS>(r, geo.G - c0, [&](int j) { return rg[c0 + j]; }, Y, ldy, ne, peers);
                if (tid == kProducerWarp0 * 32) PROF_ADD(41);
            }
        }
    }

    if (tid == kProducerWarp0 * 32) PROF_SET(5);
    tc_fence_before();
    __syncthreads();
    if (tid == 0) PROF_SET(6);
    if (warp == 7) tmem_dealloc512(tmem_base);
}

// ---- tile tables from the layer geometry -------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
conv_tiles_index_kernel(kn_conv2d_desc d, const int32_t *__restrict__ tile_origin, int64_t n_tiles, int th, int tw,
                        const int32_t *__restrict__ row_of_src, const int32_t *__restrict__ col_map,
                        int32_t *__restrict__ tile_cols, int32_t *__restrict__ tile_rows)
{
    const int Uo = d.U / d.stride, Vo = d.V / d.stride;
    const int uh = (th - 1) * d.stride + d.P, uw = (tw - 1) * d.stride + d.Q;
    const int ph = (d.P - 1) / 2, qh = (d.Q - 1) / 2;
    const int U_pos = uh * uw, T = th * tw;
    for (int64_t tl = blockIdx.x; tl < n_tiles; tl += gridDim.x) {
        const int o = tile_origin[tl];
        const int oy = o / Vo, ox = o - oy * Vo;
        for (int i = threadIdx.x; i < U_pos * d.C; i += blockDim.x) {
            const int p = i / d.C, c = i - p * d.C;
            const int py = p / uw, px = p - py * uw;
            const int iy = oy * d.stride - ph + py, ix = ox * d.stride - qh + px;
            int32_t col = -1;
            if (iy >= 0 && iy < d.U && ix >= 0 && ix < d.V) {
                const int32_t cs = c * d.U * d.V + iy * d.V + ix;
                col = col_map ? __ldg(col_map + cs) : cs;
            }
            tile_cols[tl * (int64_t)U_pos * d.C + i] = col;
        }
        for (int i = threadIdx.x; i < T * d.M; i += blockDim.x) {
            const int t = i / d.M, m = i - t * d.M;
            const int ty = t / tw, tx = t - ty * tw;
            const int64_t s = (int64_t)m * Uo * Vo + (int64_t)(oy + ty) * Vo + (ox + tx);
            tile_rows[tl * (int64_t)T * d.M + i] = row_of_src ? row_of_src[s] : (int32_t)s;
        }
    }
}
}  // namespace

#ifdef KN_TILE_PROF
KN_API int kn_debug_tile_prof(int64_t *out_host, int32_t reset) {
    long long t[64];
    if (reset) { memset(t, 0, sizeof(t)); KN_CUDA(cudaMemcpyToSymbol(g_tile_prof, t, sizeof(t))); return KN_OK; }
    KN_CUDA(cudaMemcpyFromSymbol(t, g_tile_prof, sizeof(t)));
    for (int i = 0; i < 64; i++) out_host[i] = (int64_t)t[i];
    return KN_OK;
}
#endif

KN_API int kn_conv2d_tiles_index(const kn_conv2d_desc *desc, const int32_t *tile_origin, int64_t n_tiles, int32_t th, int32_t tw,
                                 const int32_t *row_of_src, const int32_t *col_map, int32_t *tile_cols, int32_t *tile_rows, void *stream) {
    KN_REQUIRE(desc && desc->C > 0 && desc->M > 0 && desc->stride > 0 && (desc->P % 2) == 1 && (desc->Q % 2) == 1, "conv_tiles: bad descriptor");
    KN_REQUIRE(n_tiles >= 0 && th > 0 && tw > 0, "conv_tiles: bad tile shape");
    if (n_tiles == 0) return KN_OK;
    KN_REQUIRE(tile_origin && tile_cols && tile_rows, "conv_tiles: null pointer");
    const int64_t cap = (int64_t)kn_sm_count() * 8;
    conv_tiles_index_kernel<<<(unsigned)(n_tiles < cap ? n_tiles : cap), 256, 0, (cudaStream_t)stream>>>(*desc, tile_origin, n_tiles, th, tw, row_of_src, col_map, tile_cols, tile_rows);
    KN_CHECK_LAUNCH();
    return KN_OK;
}

KN_API int kn_spmm_tile_tc_f32(const void *maps_host, const int32_t *tile_cols, const int32_t *tile_rows, int32_t bias_col, int64_t n_tiles,
                               int32_t C, int32_t G, int32_t th, int32_t tw, int32_t stride, int32_t P, int32_t Q,
                               const float *X, int64_t ldx, float *Y, int64_t ldy, int64_t n_vecs, uint32_t flags, const kn_peers *peers_arg, void *stream) {
    KnPeersScope peers_scope(peers_arg);
    if (!peers_scope.ok) return KN_ERR_INVALID_ARGUMENT;
    KN_REQUIRE(n_tiles >= 0 && C > 0 && C % KS == 0 && G > 0 && th > 0 && tw > 0 && stride > 0 && P > 0 && Q > 0, "spmm_tile_tc: bad shape (C=%d G=%d)", C, G);
    KN_REQUIRE(n_vecs >= 0 && ldx >= n_vecs && ldy >= n_vecs, "spmm_tile_tc: bad leading dimension");
    if (n_tiles == 0 || n_vecs == 0) return KN_OK;
    KN_REQUIRE(maps_host && tile_cols && tile_rows && X && Y, "spmm_tile_tc: null pointer");
    KN_REQUIRE(n_vecs % 4 == 0 && ldx % 4 == 0 && (((uintptr_t)X) & 15) == 0, "spmm_tile_tc: n_vecs and ldx must be multiples of 4, X 16-byte aligned");
    KN_REQUIRE(ldx * 4 < 0xffffffffLL, "spmm_tile_tc: leading dimension in bytes must fit 32 bits");
    TileGeom g;
    g.C = C; g.G = G; g.Gp = tc_gp(G); g.th = th; g.tw = tw; g.T = th * tw; g.stride = stride; g.P = P; g.Q = Q; g.n_taps = P * Q;
    g.uh = (th - 1) * stride + P; g.uw = (tw - 1) * stride + Q; g.U_pos = g.uh * g.uw; g.n_chunks = C / KS;
    KN_REQUIRE(g.T <= kMaxT && g.U_pos <= kMaxPos && G <= 256, "spmm_tile_tc: tile too large (T=%d positions=%d)", g.T, g.U_pos);
    g.merged = (stride == 1 && tw * g.Gp <= 256) ? 1 : 0;
    g.ksplit = (g.merged && 2 * th <= kMaxT) ? 2 : 1;
    g.n_iss = g.merged ? th * g.ksplit : g.T;
    g.a0 = (uint32_t)(g.T * g.Gp);
    g.n_a = (int)((512 - g.a0) / 32);
    if (g.n_a > 8) g.n_a = 8;
    KN_REQUIRE(g.a0 <= 512 && g.n_a >= 2, "spmm_tile_tc: accumulators of %d pixels x %d rows leave no room for the activation ring", g.T, g.Gp);
    g.plane_bytes = g.Gp * KS * 4;
    g.slab_bytes = 2 * g.plane_bytes;
    const size_t fixed = (size_t)g.U_pos * C * 4 + (size_t)kMaxT * 256 * 4 + 1024 /*align*/ + 1024 /*barriers*/;
    const int64_t avail = 226 * 1024 - (int64_t)fixed;
    // shared memory: the weight slabs of exactly one channel chunk -- slot = tap, so the issuers' descriptors do not depend on the
    // chunk; a slab is released at its last use inside the chunk, so the next chunk's slabs stream in behind the issuers -- and
    // the raw gather ring (bytes in flight towards this SM)
    const int n_slots = g.n_taps;
    int n_raw = (int)((avail - (int64_t)n_slots * g.slab_bytes) / kRawStageBytes);
    if (n_raw > 16) n_raw = 16;
    KN_REQUIRE(n_raw >= 3, "spmm_tile_tc: the weight slabs of one channel chunk do not fit shared memory (Gp=%d taps=%d)", g.Gp, g.n_taps);
    KN_REQUIRE((size_t)(2 * n_slots + 2 * g.n_a + 2 * n_raw + 2) * 8 <= 1024, "spmm_tile_tc: too many barriers");
    g.n_slots = n_slots;
    g.n_raw = n_raw;
    g.epi_pixels = (int)(((int64_t)n_raw * kRawStageBytes) / ((int64_t)G * BM * 4));
    if (g.epi_pixels > g.T) g.epi_pixels = g.T;
    g.bulk_epi = (g.epi_pixels >= 1 && (((uintptr_t)Y) & 15) == 0 && ldy % 4 == 0) ? 1 : 0;
    const size_t smem = (size_t)n_slots * g.slab_bytes + (size_t)n_raw * kRawStageBytes + fixed;
    const int64_t n_btiles = kn_cdiv(n_vecs, BM);
    KN_REQUIRE(n_tiles * n_btiles <= 0x7fffffffLL, "spmm_tile_tc: grid too large");
    TileJobs jobs;
    memset(&jobs, 0, sizeof(jobs));
    for (int w = 0; w < g.n_iss; w++) {
        for (int p = 0; p < g.U_pos; p++) {
            const int py = p / g.uw, px = p - py * g.uw;
            int tap0 = -1, m = 0, acc0 = 0, rel = 0;
            if (g.merged) {
                // issuers of tile row `row` (stride 1): the run of pixels tx_hi .. tx_lo (descending) reads taps dx = px - tx (ascending);
                // a slab's last use in a chunk is by the row's last pixel
                const int row = w / g.ksplit;
                const int dy = py - row;
                const int tx_hi = px < g.tw - 1 ? px : g.tw - 1, tx_lo = px - g.Q + 1 > 0 ? px - g.Q + 1 : 0;
                if (dy >= 0 && dy < g.P && tx_hi >= tx_lo) {
                    tap0 = dy * g.Q + (px - tx_hi); m = tx_hi - tx_lo + 1; acc0 = row * g.tw + (g.tw - 1 - tx_hi); rel = (tx_hi == g.tw - 1) ? 1 : 0;
                }
            } else {
                const int ty = w / g.tw, tx = w - ty * g.tw;
                const int dy = py - ty * g.stride, dx = px - tx * g.stride;
                if (dy >= 0 && dy < g.P && dx >= 0 && dx < g.Q) { tap0 = dy * g.Q + dx; m = 1; acc0 = w; rel = 1; }
            }
            if (tap0 < 0) continue;
            int4 &rec = jobs.rec[w * kMaxPos + p];
            rec.x = 2 | (rel << 2) | (tap0 << 8) | ((acc0 * g.Gp) << 16);
            rec.y = (int)(((1u << m) - 1u) << tap0);
            rec.z = (int)(((uint32_t)tap0 * (uint32_t)g.plane_bytes) >> 4);          // slab ring of exactly n_taps slots: slot = tap
            rec.w = (int)make_idesc_tf32(BM, m * g.Gp);
        }
    }
    CUtensorMap maps[4];
    memcpy(maps, maps_host, 4 * sizeof(CUtensorMap));
    const KnPeers peers = kn_current_peers();
    const bool relu = (flags & KN_SPMM_RELU) != 0;
    const dim3 grid((unsigned)(n_tiles * n_btiles));
    cudaStream_t s = (cudaStream_t)stream;
    // geometry-specialised issuers (issuer_fast) for 3x3 / stride-1 layers with the tile shapes the host picks
    const bool spec_ok = g.merged && g.ksplit == 2 && P == 3 && Q == 3 && stride == 1 && g.n_slots == 9;
    const int spec = !spec_ok ? 0 : (th == 2 && tw == 2 && g.Gp == 64) ? 1 : (th == 2 && tw == 2 && g.Gp == 96) ? 2 : (th == 1 && tw == 2 && g.Gp == 128) ? 3 : 0;
    return dispatch_relu_peers(relu, peers.n > 0, [&](auto R, auto PP) {
        constexpr bool r = decltype(R)::value, pp = decltype(PP)::value;
        const decltype(&pg_tile_tc_kernel<r, pp, 0, 0, 0>) kfns[4] = {pg_tile_tc_kernel<r, pp, 0, 0, 0>, pg_tile_tc_kernel<r, pp, 2, 2, 64>,
                                                                      pg_tile_tc_kernel<r, pp, 2, 2, 96>, pg_tile_tc_kernel<r, pp, 1, 2, 128>};
        KN_ONCE_PER_DEVICE {
            for (auto kfn : kfns) KN_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        }
        kfns[spec]<<<grid, kThreads, smem, s>>>(maps[0], maps[1], tile_cols, tile_rows, bias_col, g, jobs, n_tiles, n_btiles, kSuperTiles,
                                                X, ldx, Y, ldy, n_vecs, peers);
        KN_CHECK_LAUNCH();
        return KN_OK;
    });
}
