// tc_common.cuh -- what the tcgen05 kernels (pgroup_tc.cu, pgtile_tc.cu) share: their stage / tile constants, PTX wrappers
// (mbarriers, TMA loads, UMMA descriptors, tcgen05.mma / .ld / .st / .commit, TMEM allocation), the per-lane output store and
// the launch dispatch.  sm_100a only.
#pragma once
#include "common.cuh"
#include <cuda.h>
#include <type_traits>

namespace kn_tc {

constexpr int KS = 16;                 // k per stage, = the TMA box width (words) of the weight planes (kn_pg_tc_tensormaps)
constexpr int BM = 128;                // batch columns per UMMA (M): one per TMEM lane
// rasterisation super-tile (kn_raster): 8 x 128 = 1024 batch columns, small enough that the X rows shared by neighbouring
// groups (3x3 windows re-read every row 9 times, one image row of groups apart) are still L2-resident when they are re-read
// (sweep 4..32: 4/8 best by ~1 %)
constexpr int kSuperTiles = 8;
// weight rows per UMMA (N) and per TMA box: G rounded up to the UMMA's N granularity of 16, at most 256 (a taller group
// runs in 256-row chunks)
__host__ __device__ constexpr int tc_gp(int G) { return G > 256 ? 256 : (G + 15) / 16 * 16; }

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}" :: "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n\t}" :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t"      // suspend-time hint: sleep in hardware, do not spin
        "@p bra DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "DONE:\n\t}" :: "r"(smem_u32(bar)), "r"(parity), "r"(0x989680u) : "memory");
}
// One lane of a converged warp (elect.sync).  The issuer / TMA-producer code runs under THIS predicate, not under
// `lane == 0`: tcgen05.mma, tcgen05.commit and the bulk-tensor copy are uniform-datapath instructions, and inside a branch
// the compiler only knows to be divergent it wraps every one of them in an ELECT / 6 x R2UR / BRA.U.ANY loop -- measured
// 127-143 cycles per tcgen05.mma per thread whatever its shape.  Under elect.sync it emits plain uniform code and one thread
// issues 128 x N x 8 tf32 MMAs at the pipe rate (42 cycles for N = 64, 74 for N = 128, 138 for N = 256; scratch/umma_rate.cu).
__device__ __forceinline__ bool elect_one() {
    uint32_t p;
    asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.b32 %0, 1, 0, P;\n\t}" : "=r"(p));
    return p != 0;
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tma_load_2d(void *dst, const CUtensorMap *map, int c0, int c1, uint64_t *bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 :: "r"(smem_u32(dst)), "l"(map), "r"(c0), "r"(c1), "r"(smem_u32(bar)) : "memory");
}

__device__ __forceinline__ void tma_load_2d_mcast(void *dst, const CUtensorMap *map, int c0, int c1, uint64_t *bar, uint16_t cta_mask) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%2, %3}], [%4], %5;"
                 :: "r"(smem_u32(dst)), "l"(map), "r"(c0), "r"(c1), "r"(smem_u32(bar)), "h"(cta_mask) : "memory");
}
__device__ __forceinline__ void umma_commit_mcast(uint64_t *bar, uint16_t cta_mask) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 :: "r"(smem_u32(bar)), "h"(cta_mask) : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t *bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(smem_u32(bar)) : "memory");
}

// shared-memory matrix descriptors (cute::UMMA::SmemDescriptor, version 1 = Blackwell)
//   bits [0,14) start>>4 | [16,30) LBO>>4 | [32,46) SBO>>4 | [46,48) version | [61,64) layout type
__device__ __forceinline__ uint64_t make_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout_type) {
    return (uint64_t)((smem_addr & 0x3FFFF) >> 4) | ((uint64_t)(lbo_bytes >> 4) << 16) | ((uint64_t)(sbo_bytes >> 4) << 32) |
           ((uint64_t)1 << 46) | ((uint64_t)layout_type << 61);
}
constexpr uint32_t kLayoutSW64 = 4;      // (SWIZZLE_128B_BASE32B = 1 is the only MN-major layout for 32-bit operands; not used: A lives in TMEM)

// instruction descriptors (cute::UMMA::InstrDescriptor): D=f32, A (TMEM) and B K-major.  The A / B format field is the only
// difference between the two kinds: tf32 (2) under kind::tf32, bf16 (1) under kind::f16.
__host__ __device__ constexpr uint32_t make_idesc_fmt(int M, int N, uint32_t ab_format) {
    return (1u << 4) | (ab_format << 7) | (ab_format << 10) | (0u << 15) | (0u << 16) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__host__ __device__ constexpr uint32_t make_idesc_tf32(int M, int N) { return make_idesc_fmt(M, N, 2u); }
__host__ __device__ constexpr uint32_t make_idesc_bf16(int M, int N) { return make_idesc_fmt(M, N, 1u); }
// the kind::f16 (bf16) descriptor of the same shape as a kind::tf32 one
__host__ __device__ constexpr uint32_t idesc_tf32_to_bf16(uint32_t idesc_tf32) {
    return idesc_tf32 ^ (make_idesc_tf32(0, 0) ^ make_idesc_bf16(0, 0));
}

// A operand from tensor memory: D[tmem] (+)= A[tmem] . B[smem desc]
__device__ __forceinline__ void umma_tf32_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}"
        :: "r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// the same with bf16 operands (K = 16 per instruction, two elements per 32-bit TMEM column / 4-byte word of B); it may
// accumulate into an accumulator that kind::tf32 instructions also write: both keep D in fp32
__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
        :: "r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}

// The split of the tensor-core kernels (2 MMAs per 8 k):  x.w ~= x_hi.w_hi  (kind::tf32, K = 8)
//                                                                + [x_hi | x_lo] . [w_lo ; w_hi]  (kind::f16 in bf16, K = 16)
// hi = v rounded to nearest TF32, lo = v - hi (exact in fp32, |lo| <= 2^-11 |v|).  The correction terms are ~2^-11 of the
// product, so bf16's 8-bit significand leaves them ~2^-18 of it; bf16 has fp32's exponent range (no scaling, where fp16
// would underflow on x_lo).  Per product the error is below 1.04 * 2^-17 |x||w|: two cross terms of <= 2^-11 |x||w| whose
// operands are rounded to bf16 (2^-8 each), plus the dropped lo.lo (<= 2^-22).  The former 3xTF32 split was ~3 * 2^-20;
// both are far inside the rtol 1e-4 parity bar (tests/test_split_numerics.py models them).
__device__ __forceinline__ uint32_t tf32_rna(float v) {
    uint32_t h;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(h) : "f"(v));
    return h & 0xFFFFE000u;                 // the tf32 value as an fp32 bit pattern
}
__device__ __forceinline__ uint32_t bf16x2_rn(float k_even, float k_odd) {        // the lower half holds the lower k
    uint32_t r;
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(k_odd), "f"(k_even));
    return r;
}
// 8 consecutive k of one row: hi[8] = TF32 words, bhi[4] / blo[4] = bf16 pairs of hi / lo (k = 2j in the lower half of word j)
__device__ __forceinline__ void split8_tf32_bf16(const float *v, uint32_t *hi, uint32_t *bhi, uint32_t *blo) {
    float h[8], l[8];
#pragma unroll
    for (int i = 0; i < 8; i++) {
        hi[i] = tf32_rna(v[i]);
        h[i] = __uint_as_float(hi[i]);
        l[i] = v[i] - h[i];
    }
#pragma unroll
    for (int j = 0; j < 4; j++) {
        bhi[j] = bf16x2_rn(h[2 * j], h[2 * j + 1]);
        blo[j] = bf16x2_rn(l[2 * j], l[2 * j + 1]);
    }
}

template <int NW>
__device__ __forceinline__ void tmem_store(uint32_t taddr, const uint32_t (&r)[NW]) {
    if constexpr (NW == 16) {
        asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
                     :: "r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
                        "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]) : "memory");
    } else {
        asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
                     :: "r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]) : "memory");
    }
}
// 16 consecutive columns of the warp's 32 TMEM lanes (lane i of the warp gets TMEM lane (taddr >> 16) + i), waited for
__device__ __forceinline__ void tmem_load16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                   "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                 : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// All 512 TMEM columns for the CTA (the kernels run one CTA per SM); one whole warp calls both.  The base address lands in
// *slot (shared memory) and is read after the next __syncthreads, between tc_fence_before / tc_fence_after.
__device__ __forceinline__ void tmem_alloc512(uint32_t *slot) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" :: "r"(smem_u32(slot)));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
}
// after tc_fence_before + __syncthreads: no tcgen05 operation of the CTA is outstanding
__device__ __forceinline__ void tmem_dealloc512(uint32_t base) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" :: "r"(base));
}

// Per-lane epilogue of 16 accumulator columns of batch column ne (< n_vecs): r[t] (fp32 bits, ReLU applied here) goes to row
// row_of(t) of Y for t < n_rows; the other columns have no row (row_of is not called for them).  PEERS (fused all-gather): to
// that row of every destination whose bit is set in the row's need mask -- row ids and masks are loaded first (a load placed
// between the stores would be serialised behind them), then one pass of stores per destination.  PEERS is a template
// parameter because its code costs the plain epilogue ~10 %.  The plain path keeps each row-id load under the same guard as
// its store: loading all 16 first made the compiler branch around every store instead of predicating it (pg_tc's conv
// layers 1-2 % slower on a B200).
template <bool RELU, bool PEERS, typename RowOf>
__device__ __forceinline__ void store_rows16(uint32_t (&r)[16], int n_rows, RowOf row_of, float *__restrict__ Y, int64_t ldy, int64_t ne,
                                             const KnPeers &peers) {
    if constexpr (!PEERS) {
#pragma unroll
        for (int t = 0; t < 16; t++) {
            if (t < n_rows) {
                float y = __uint_as_float(r[t]);
                if (RELU) y = fmaxf(y, 0.0f);
                Y[(int64_t)row_of(t) * ldy + ne] = y;
            }
        }
    } else {
        int32_t yrow[16];
        unsigned pmask[16];
#pragma unroll
        for (int t = 0; t < 16; t++) yrow[t] = (t < n_rows) ? row_of(t) : -1;
#pragma unroll
        for (int t = 0; t < 16; t++) pmask[t] = (yrow[t] >= 0) ? kn_peer_mask(peers, yrow[t]) : 0u;
#pragma unroll
        for (int t = 0; t < 16; t++) {
            float y = __uint_as_float(r[t]);
            if (RELU) y = fmaxf(y, 0.0f);
            r[t] = __float_as_uint(y);
        }
        for (int p = 0; p < peers.n; p++) {
            float *__restrict__ yb = peers.y[p];
#pragma unroll
            for (int t = 0; t < 16; t++)
                if ((pmask[t] >> p) & 1u) yb[(int64_t)yrow[t] * ldy + ne] = __uint_as_float(r[t]);
        }
    }
}

// Host: calls launch(std::bool_constant<RELU>, std::bool_constant<PEERS>) for the run-time pair and returns its result, so a
// kernel's launch code names its instantiation once.
template <typename F>
int dispatch_relu_peers(bool relu, bool peers, F &&launch) {
    if (peers) return relu ? launch(std::true_type{}, std::true_type{}) : launch(std::false_type{}, std::true_type{});
    return relu ? launch(std::true_type{}, std::false_type{}) : launch(std::false_type{}, std::false_type{});
}


}  // namespace kn_tc
