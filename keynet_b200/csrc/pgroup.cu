// pgroup.cu -- pattern-grouped execution format for keyed layer matrices and its fp32 SIMT kernel.
//
// Rows of a keyed Toeplitz matrix that belong to the same output pixel (all M output channels)
// touch exactly the same columns -- also after permutation / gain keys, which only relabel rows
// and columns.  Grouping rows by identical column set turns the matrix into
//
//     group g:   rows[g][0..G)          output rows (scattered by the output key)
//                cols[g][0..K_pad)      the shared column list (gather list into X)
//                vals[g][0..G)[0..K_pad) dense value block, zero padded
//
// and the SpMM into one small GEMM per group with a GATHERED B operand:
//     Y[rows[g], :] = vals[g] (G x K) . X[cols[g], :] (K x N)
// This is the B200 form of the reference's unique-tile storage (TiledMatrix / Conv2dTiledMatrix,
// keynet/sparse.py:517-835: "unique spatial tile x dense (Cout,Cin) channel block"), but it is
// discovered from the compiled CSR itself (row-pattern hashing), so it also applies where the
// reference's tiling does not (global permutation keys, keynet/system.py:360).
// Column indices are read once per group instead of once per stored value (4 instead of 8 bytes per
// nnz), every gathered X row is reused by G output rows from shared memory, and the value block
// is reused across the whole batch tile: the kernel is bound by the fp32 FMA pipe, not by L1/L2
// gathers like the row-per-warp CSR kernel.
//
// Kernel: CTA = 256 threads = 8 warps, tile = (8*RW rows) x (128 batch columns), K chunks of 32
// staged through a 3-stage cp.async ring (A: value rows, B: gathered X rows).  Warp w owns rows
// [w*RW, (w+1)*RW), lane l owns 4 consecutive batch columns: RW*4 accumulators, A operands are
// warp-broadcast LDS.128, B operands conflict-free LDS.128, 16*RW FFMA per (RW+4) LDS.
#include "common.cuh"

namespace {

constexpr int kThreads = 256;
constexpr int KT = 32;       // k chunk
constexpr int TN = 128;      // batch columns per CTA
constexpr int kStages = 3;

__device__ __forceinline__ uint64_t mix64(uint64_t x) {    // splitmix64 finaliser
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}

// order-independent 64-bit hash of a row's column set (+ its length); one warp per row
__global__ void __launch_bounds__(kThreads)
row_pattern_hash_kernel(const int64_t *__restrict__ indptr, const int32_t *__restrict__ indices, int64_t n_rows, uint64_t *__restrict__ hash) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int64_t r = (int64_t)blockIdx.x * (kThreads / 32) + warp; r < n_rows; r += (int64_t)gridDim.x * (kThreads / 32)) {
        const int64_t beg = indptr[r], end = indptr[r + 1];
        uint64_t h = 0;
        for (int64_t e = beg + lane; e < end; e += 32) h += mix64((uint64_t)(uint32_t)indices[e]);
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) h += __shfl_xor_sync(0xffffffffu, h, off);
        if (lane == 0) hash[r] = mix64(h ^ ((uint64_t)(end - beg) << 40));
    }
}

// mismatch[i] = 1 iff row rows[i] and row leaders[i] do not have identical column lists
__global__ void __launch_bounds__(kThreads)
pg_verify_kernel(const int64_t *__restrict__ indptr, const int32_t *__restrict__ indices,
                 const int64_t *__restrict__ rows, const int64_t *__restrict__ leaders, int64_t n, int32_t *__restrict__ mismatch) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int64_t i = (int64_t)blockIdx.x * (kThreads / 32) + warp; i < n; i += (int64_t)gridDim.x * (kThreads / 32)) {
        const int64_t r = rows[i], l = leaders[i];
        const int64_t rb = indptr[r], lb = indptr[l], len = indptr[r + 1] - rb;
        int bad = (len != indptr[l + 1] - lb) ? 1 : 0;
        if (!bad && r != l)
            for (int64_t e = lane; e < len; e += 32) bad |= (indices[rb + e] != indices[lb + e]) ? 1 : 0;
        bad = __any_sync(0xffffffffu, bad);
        if (lane == 0) mismatch[i] = bad;
    }
}

// pack one class: cols[g][K_pad], vals[g][G][K_pad]; padding columns repeat the group's first column with value 0
__global__ void __launch_bounds__(kThreads)
pg_pack_kernel(const int64_t *__restrict__ indptr, const int32_t *__restrict__ indices, const float *__restrict__ data,
               const int64_t *__restrict__ rows, int64_t n_groups, int G, int K_pad,
               int32_t *__restrict__ cols, float *__restrict__ vals) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t n_rows = n_groups * G;
    for (int64_t i = (int64_t)blockIdx.x * (kThreads / 32) + warp; i < n_rows; i += (int64_t)gridDim.x * (kThreads / 32)) {
        const int64_t g = i / G;
        const int64_t r = rows[i];
        const int64_t beg = indptr[r];
        const int len = (int)(indptr[r + 1] - beg);
        float *__restrict__ v = vals + i * (int64_t)K_pad;
        for (int k = lane; k < K_pad; k += 32) v[k] = (k < len) ? data[beg + k] : 0.0f;
        if (i == g * G) {                                  // the group's first row writes the column list
            int32_t *__restrict__ c = cols + g * (int64_t)K_pad;
            const int32_t c0 = len > 0 ? indices[beg] : 0;
            for (int k = lane; k < K_pad; k += 32) c[k] = (k < len) ? indices[beg + k] : c0;
        }
    }
}

__device__ __forceinline__ void cp_async16(void *smem_dst, const void *gmem_src, bool valid) {
    const unsigned dst = (unsigned)__cvta_generic_to_shared(smem_dst);
    const int bytes = valid ? 16 : 0;                     // src-size 0 => 16 bytes of zeros
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" :: "r"(dst), "l"(gmem_src), "r"(bytes));
}
__device__ __forceinline__ void cp_async4(void *smem_dst, const void *gmem_src, bool valid) {
    const unsigned dst = (unsigned)__cvta_generic_to_shared(smem_dst);
    const int bytes = valid ? 4 : 0;                      // src-size 0 => 4 bytes of zeros
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;\n" :: "r"(dst), "l"(gmem_src), "r"(bytes));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" :: "n"(N)); }

// Narrow batches (1 <= n_vecs <= 32, run_start != null; kn_spmm_pg_narrow_f32): a 128-column tile would hold n_vecs useful
// columns, so its columns become (group, batch column) pairs, j = p * NB + n with NB = 1 << nb_shift >= n_vecs.  A work item
// is then a RUN -- run_groups[run_start[i] .. run_start[i+1]), at most 128 / NB groups sharing one value block and one
// group_k -- so the staged value rows serve every group of the run.  The B stage gathers X[cols[g_p][k]][n] with 4-byte
// cp.async (zero for n >= n_vecs and for missing groups: any ldx and alignment); the FMA loop is the same as for wide
// batches, so every output element is the same fp32 chain (bit-identical to a wide launch over a zero-padded X).
constexpr int kNarrowMaxRW = 4;   // narrow batches use row tiles of 8, 16 or 32 rows: a thin grid needs CTAs more than long tiles

template <int RW, bool RELU>
__global__ void __launch_bounds__(kThreads, 2)
pg_simt_kernel(const int32_t *__restrict__ rows, const int32_t *__restrict__ cols, const float *__restrict__ vals,
               const int32_t *__restrict__ group_k, const int32_t *__restrict__ block_of, int64_t n_groups, int G, int K_pad, int tiles_per_group, int64_t n_items, int64_t n_tiles,
               const float *__restrict__ X, int64_t ldx, float *__restrict__ Y, int64_t ldy, int64_t n_vecs, const __grid_constant__ KnPeers peers,
               const int32_t *__restrict__ run_groups, const int32_t *__restrict__ run_start, int nb_shift)
{
    constexpr int TM = 8 * RW;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float (*sA)[TM][KT] = reinterpret_cast<float (*)[TM][KT]>(smem_raw);
    float (*sB)[KT][TN] = reinterpret_cast<float (*)[KT][TN]>(smem_raw + sizeof(float) * kStages * TM * KT);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const KnRaster rt = kn_raster(blockIdx.x, n_items, n_tiles, 16);      // super-tile = 16 x 128 batch columns
    const int64_t item = rt.item / tiles_per_group;                       // group, or run of groups (narrow)
    const int rowtile = (int)(rt.item - item * tiles_per_group);
    const int64_t nbase = rt.tile * TN;
    const bool narrow = RW <= kNarrowMaxRW && run_start != nullptr;    // compiled out of the taller row tiles
    const int r0 = narrow ? __ldg(run_start + item) : 0;
    const int n_here = narrow ? __ldg(run_start + item + 1) - r0 : 1;   // groups of the run (<= 128 >> nb_shift)
    const int64_t g = narrow ? (int64_t)__ldg(run_groups + r0) : item;
    // groups of one class share K_pad (storage) but loop only over their own K (edge / corner pixels have fewer taps)
    const int n_chunks = group_k ? (__ldg(group_k + g) + KT - 1) / KT : K_pad / KT;

    const int64_t blk = block_of ? (int64_t)__ldg(block_of + g) : g;       // unique value block of this group
    const float *__restrict__ vbase = vals + (blk * G + (int64_t)rowtile * TM) * K_pad;
    const int32_t *__restrict__ cbase = cols + g * (int64_t)K_pad;
    const int rows_here = min(TM, G - rowtile * TM);
    // narrow: this thread's B-stage column (group p of the run, batch column n), fixed over the k loop
    const int jb = tid & (TN - 1), pb = jb >> nb_shift, nb = jb & ((1 << nb_shift) - 1);
    const bool jok = narrow && pb < n_here && nb < n_vecs;
    const int32_t *__restrict__ cb = narrow ? cols + (int64_t)__ldg(run_groups + r0 + (jok ? pb : 0)) * K_pad : cbase;
    const float *__restrict__ xb = X + (jok ? nb : 0);

    auto load_stage = [&](int s, int kc) {
        // A: TM rows x 8 chunks of 16 B
#pragma unroll
        for (int i = 0; i < (TM * 8 + kThreads - 1) / kThreads; i++) {
            const int idx = tid + i * kThreads;
            if (idx < TM * 8) {
                const int r = idx >> 3, ch = idx & 7;
                const bool ok = r < rows_here;
                cp_async16(&sA[s][r][ch * 4], vbase + (ok ? ((int64_t)r * K_pad + kc * KT + ch * 4) : 0), ok);
            }
        }
        if (narrow) {
            // B: per thread one tile column, 16 of the 32 gathered rows, 4 bytes each
#pragma unroll
            for (int i = 0; i < (KT * TN) / kThreads; i++) {
                const int kr = (tid >> 7) + i * (kThreads / TN);
                cp_async4(&sB[s][kr][jb], xb + (int64_t)__ldg(cb + kc * KT + kr) * ldx, jok);
            }
            return;
        }
        // B: 32 gathered X rows x 32 chunks of 16 B (one warp per row: 512 contiguous bytes)
#pragma unroll
        for (int i = 0; i < (KT * (TN / 4)) / kThreads; i++) {
            const int idx = tid + i * kThreads;
            const int kr = idx >> 5, ch = idx & 31;
            const int32_t c = __ldg(cbase + kc * KT + kr);
            const int64_t n = nbase + ch * 4;
            const bool ok = n < n_vecs;
            cp_async16(&sB[s][kr][ch * 4], X + (int64_t)c * ldx + (ok ? n : 0), ok);
        }
    };

    float acc[RW][4];
#pragma unroll
    for (int i = 0; i < RW; i++) { acc[i][0] = acc[i][1] = acc[i][2] = acc[i][3] = 0.0f; }

#pragma unroll
    for (int s = 0; s < kStages - 1; s++) {
        if (s < n_chunks) load_stage(s, s);
        cp_async_commit();
    }
    for (int kc = 0; kc < n_chunks; kc++) {
        cp_async_wait<kStages - 2>();
        __syncthreads();
        {   // prefetch chunk kc + kStages - 1 into the stage that was consumed in iteration kc - 1
            const int nk = kc + kStages - 1;
            if (nk < n_chunks) load_stage(nk % kStages, nk);
            cp_async_commit();
        }
        const int s = kc % kStages;
#pragma unroll
        for (int k4 = 0; k4 < KT; k4 += 4) {
            const float4 b0 = *reinterpret_cast<const float4 *>(&sB[s][k4 + 0][lane * 4]);
            const float4 b1 = *reinterpret_cast<const float4 *>(&sB[s][k4 + 1][lane * 4]);
            const float4 b2 = *reinterpret_cast<const float4 *>(&sB[s][k4 + 2][lane * 4]);
            const float4 b3 = *reinterpret_cast<const float4 *>(&sB[s][k4 + 3][lane * 4]);
#pragma unroll
            for (int i = 0; i < RW; i++) {
                const float4 a = *reinterpret_cast<const float4 *>(&sA[s][warp * RW + i][k4]);   // warp-broadcast
                acc[i][0] = fmaf(a.x, b0.x, acc[i][0]); acc[i][1] = fmaf(a.x, b0.y, acc[i][1]); acc[i][2] = fmaf(a.x, b0.z, acc[i][2]); acc[i][3] = fmaf(a.x, b0.w, acc[i][3]);
                acc[i][0] = fmaf(a.y, b1.x, acc[i][0]); acc[i][1] = fmaf(a.y, b1.y, acc[i][1]); acc[i][2] = fmaf(a.y, b1.z, acc[i][2]); acc[i][3] = fmaf(a.y, b1.w, acc[i][3]);
                acc[i][0] = fmaf(a.z, b2.x, acc[i][0]); acc[i][1] = fmaf(a.z, b2.y, acc[i][1]); acc[i][2] = fmaf(a.z, b2.z, acc[i][2]); acc[i][3] = fmaf(a.z, b2.w, acc[i][3]);
                acc[i][0] = fmaf(a.w, b3.x, acc[i][0]); acc[i][1] = fmaf(a.w, b3.y, acc[i][1]); acc[i][2] = fmaf(a.w, b3.z, acc[i][2]); acc[i][3] = fmaf(a.w, b3.w, acc[i][3]);
            }
        }
    }
    cp_async_wait<0>();

    if (narrow) {                                                    // scalar stores of the (group, column) pairs
#pragma unroll
        for (int c = 0; c < 4; c++) {
            const int j = lane * 4 + c, p = j >> nb_shift, n = j & ((1 << nb_shift) - 1);
            if (p < n_here && n < n_vecs) {
                const int64_t rbase = (int64_t)__ldg(run_groups + r0 + p) * G + (int64_t)rowtile * TM;
#pragma unroll
                for (int i = 0; i < RW; i++) {
                    const int r = warp * RW + i;
                    if (r < rows_here) Y[(int64_t)__ldg(rows + rbase + r) * ldy + n] = RELU ? fmaxf(acc[i][c], 0.0f) : acc[i][c];
                }
            }
        }
        return;
    }
    const int64_t n0 = nbase + lane * 4;
    if (n0 < n_vecs) {
#pragma unroll
        for (int i = 0; i < RW; i++) {
            const int r = warp * RW + i;
            if (r < rows_here) {
                const int64_t yrow = rows[g * G + (int64_t)rowtile * TM + r];
                float4 o = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
                if (RELU) { o.x = fmaxf(o.x, 0.0f); o.y = fmaxf(o.y, 0.0f); o.z = fmaxf(o.z, 0.0f); o.w = fmaxf(o.w, 0.0f); }
                if (peers.n == 0) *reinterpret_cast<float4 *>(Y + yrow * ldy + n0) = o;
                else {
                    const unsigned pmask = kn_peer_mask(peers, yrow);
                    KN_FOR_EACH_DEST(peers, Y, pmask, yb) *reinterpret_cast<float4 *>(yb + yrow * ldy + n0) = o;
                }
            }
        }
    }
}

// ---- small groups (G <= 16, K <= 128; LeNet-sized layers): one warp per (group, batch super-tile) -------------
// The warp stages its group's column list and value block (transposed to [k][row]) in shared memory once, then
// walks the 128-column batch tiles of its super-tile: per k one coalesced LDG.128 of the gathered X row segment
// feeds 4*G FFMA (values come as warp-broadcast LDS.128), exact K (no padding), G rows x 512 B written per tile.
template <int GM, bool RELU>
__global__ void __launch_bounds__(kThreads, 2)
pg_small_kernel(const int32_t *__restrict__ rows, const int32_t *__restrict__ cols, const float *__restrict__ vals,
                const int32_t *__restrict__ group_k, const int32_t *__restrict__ block_of, int64_t n_groups, int G, int K_pad, int64_t n_supers, int tiles_per_super,
                const float *__restrict__ X, int64_t ldx, float *__restrict__ Y, int64_t ldy, int64_t n_vecs, const __grid_constant__ KnPeers peers)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int per_warp = K_pad * (GM + 1);                                   // floats: vals [K_pad][GM] + cols [K_pad]
    float *s_val = reinterpret_cast<float *>(smem_raw) + (size_t)warp * per_warp;
    int32_t *s_col = reinterpret_cast<int32_t *>(s_val + (size_t)K_pad * GM);
    const int64_t item = (int64_t)blockIdx.x * (kThreads / 32) + warp;       // groups fastest inside a super-tile
    if (item >= n_groups * n_supers) return;
    const int64_t sup = item / n_groups, g = item - sup * n_groups;
    const int K = group_k ? __ldg(group_k + g) : K_pad;
    const int64_t blk = block_of ? (int64_t)__ldg(block_of + g) : g;

    // K rounded up to the prefetch block with zero values / a valid column: the k loop carries no predicates
    constexpr int PD = (GM <= 8) ? 8 : 4;                                    // gathered X rows in flight per lane: 2 x PD LDG.128
    const int Kr = (K + 2 * PD - 1) / (2 * PD) * (2 * PD);                   // <= K_pad (a multiple of 32)
    for (int i = lane; i < Kr; i += 32) s_col[i] = __ldg(cols + g * (int64_t)K_pad + (i < K ? i : 0));
    for (int i = lane; i < Kr * GM; i += 32) {
        const int k = i / GM, r = i - k * GM;
        s_val[i] = (r < G && k < K) ? __ldg(vals + (blk * G + r) * (int64_t)K_pad + k) : 0.0f;
    }
    __syncwarp();

    for (int t = 0; t < tiles_per_super; t++) {
        const int64_t n0 = (sup * tiles_per_super + t) * TN + lane * 4;
        if (n0 - lane * 4 >= n_vecs) break;                                  // warp-uniform
        const bool ok = n0 < n_vecs;
        const float *__restrict__ xb = X + (ok ? n0 : 0);
        float acc[GM][4];
#pragma unroll
        for (int r = 0; r < GM; r++) { acc[r][0] = acc[r][1] = acc[r][2] = acc[r][3] = 0.0f; }
        // one coalesced LDG.128 per k feeds 4*GM FFMA; with a single load in flight the loop is bound by L2 latency, so
        // the gathers run a double-buffered register ring 2 x PD rows ahead of the FMAs
        auto gather = [&](int k) { return __ldg(reinterpret_cast<const float4 *>(xb + (int64_t)s_col[k] * ldx)); };
        auto fma_row = [&](const float4 x, int k) {
#pragma unroll
            for (int r4 = 0; r4 < GM; r4 += 4) {
                const float4 a = *reinterpret_cast<const float4 *>(&s_val[k * GM + r4]);
                acc[r4 + 0][0] = fmaf(a.x, x.x, acc[r4 + 0][0]); acc[r4 + 0][1] = fmaf(a.x, x.y, acc[r4 + 0][1]); acc[r4 + 0][2] = fmaf(a.x, x.z, acc[r4 + 0][2]); acc[r4 + 0][3] = fmaf(a.x, x.w, acc[r4 + 0][3]);
                acc[r4 + 1][0] = fmaf(a.y, x.x, acc[r4 + 1][0]); acc[r4 + 1][1] = fmaf(a.y, x.y, acc[r4 + 1][1]); acc[r4 + 1][2] = fmaf(a.y, x.z, acc[r4 + 1][2]); acc[r4 + 1][3] = fmaf(a.y, x.w, acc[r4 + 1][3]);
                acc[r4 + 2][0] = fmaf(a.z, x.x, acc[r4 + 2][0]); acc[r4 + 2][1] = fmaf(a.z, x.y, acc[r4 + 2][1]); acc[r4 + 2][2] = fmaf(a.z, x.z, acc[r4 + 2][2]); acc[r4 + 2][3] = fmaf(a.z, x.w, acc[r4 + 2][3]);
                acc[r4 + 3][0] = fmaf(a.w, x.x, acc[r4 + 3][0]); acc[r4 + 3][1] = fmaf(a.w, x.y, acc[r4 + 3][1]); acc[r4 + 3][2] = fmaf(a.w, x.z, acc[r4 + 3][2]); acc[r4 + 3][3] = fmaf(a.w, x.w, acc[r4 + 3][3]);
            }
        };
        float4 xa[PD], xc[PD];
#pragma unroll
        for (int i = 0; i < PD; i++) xa[i] = gather(i);
        for (int k0 = 0; k0 < Kr; k0 += 2 * PD) {
#pragma unroll
            for (int i = 0; i < PD; i++) xc[i] = gather(k0 + PD + i);
#pragma unroll
            for (int i = 0; i < PD; i++) fma_row(xa[i], k0 + i);
            if (k0 + 2 * PD < Kr) {
#pragma unroll
                for (int i = 0; i < PD; i++) xa[i] = gather(k0 + 2 * PD + i);
            }
#pragma unroll
            for (int i = 0; i < PD; i++) fma_row(xc[i], k0 + PD + i);
        }
        if (ok) {
#pragma unroll
            for (int r4 = 0; r4 < GM; r4 += 4) {                              // row ids / need masks of 4 rows, then their stores
                int32_t yrows[4];
                unsigned pmask[4];
#pragma unroll
                for (int i = 0; i < 4; i++) yrows[i] = (r4 + i < G) ? __ldg(rows + g * G + r4 + i) : 0;
                if (peers.n != 0) {
#pragma unroll
                    for (int i = 0; i < 4; i++) pmask[i] = kn_peer_mask(peers, yrows[i]);
                }
#pragma unroll
                for (int i = 0; i < 4; i++) {
                    const int r = r4 + i;
                    if (r < G) {
                        float4 o = make_float4(acc[r][0], acc[r][1], acc[r][2], acc[r][3]);
                        if (RELU) { o.x = fmaxf(o.x, 0.0f); o.y = fmaxf(o.y, 0.0f); o.z = fmaxf(o.z, 0.0f); o.w = fmaxf(o.w, 0.0f); }
                        const int64_t yoff = (int64_t)yrows[i] * ldy + n0;
                        if (peers.n == 0) *reinterpret_cast<float4 *>(Y + yoff) = o;
                        else KN_FOR_EACH_DEST(peers, Y, pmask[i], yb) *reinterpret_cast<float4 *>(yb + yoff) = o;
                    }
                }
            }
        }
    }
}

// split-K epilogue: Y[rows[i]][:] = relu?( sum_s part[s*G + i][:] ).  A layer with one huge pattern group (a dense fully
// connected layer: VGG16 fc6 is 4096 x 25 089) has too few (row chunk, batch tile) work items to fill 148 SMs, so its K range
// is cut into S slices that run as S independent groups writing partial rows; this pass adds them (and is where the fused
// ReLU and the peer stores of the row-sharded path happen).
template <bool RELU>
__global__ void __launch_bounds__(kThreads)
splitk_reduce_kernel(const float *__restrict__ part, int S, int G, const int32_t *__restrict__ rows, float *__restrict__ Y, int64_t ldy, int64_t n_vecs,
                     const __grid_constant__ KnPeers peers)
{
    const int64_t n4 = n_vecs / 4;
    const int64_t total = (int64_t)G * n4;
    for (int64_t t = (int64_t)blockIdx.x * kThreads + threadIdx.x; t < total; t += (int64_t)gridDim.x * kThreads) {
        const int64_t i = t / n4, c = (t - i * n4) * 4;
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int s = 0; s < S; s++) {
            const float4 v = *reinterpret_cast<const float4 *>(part + ((int64_t)s * G + i) * n_vecs + c);
            acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
        }
        if (RELU) { acc.x = fmaxf(acc.x, 0.0f); acc.y = fmaxf(acc.y, 0.0f); acc.z = fmaxf(acc.z, 0.0f); acc.w = fmaxf(acc.w, 0.0f); }
        const int64_t yrow = rows[i];
        const unsigned pmask = kn_peer_mask(peers, yrow);
        KN_FOR_EACH_DEST(peers, Y, pmask, yb) *reinterpret_cast<float4 *>(yb + yrow * ldy + c) = acc;
    }
}

template <int GM>
int launch_small(const int32_t *rows, const int32_t *cols, const float *vals, const int32_t *group_k, const int32_t *block_of, int64_t n_groups, int G, int K_pad,
                 const float *X, int64_t ldx, float *Y, int64_t ldy, int64_t n_vecs, bool relu, cudaStream_t s)
{
    // up to 2048 batch columns per warp work item (the group's values are staged once per item), fewer when that would
    // leave the grid with only a few waves of CTAs (tail effect: LeNet conv2 has 196 groups)
    int tiles_per_super = 16;
    const int64_t n_tiles = kn_cdiv(n_vecs, TN);
    while (tiles_per_super > 2 && n_groups * kn_cdiv(n_tiles, tiles_per_super) < (int64_t)kn_sm_count() * 2 * 8 * (kThreads / 32)) tiles_per_super /= 2;
    const int64_t n_supers = kn_cdiv(n_tiles, tiles_per_super);
    const int64_t n_items = n_groups * n_supers, gx = kn_cdiv(n_items, kThreads / 32);
    KN_REQUIRE(gx <= 0x7fffffffLL, "spmm_pg(small): grid too large");
    const size_t smem = (size_t)(kThreads / 32) * K_pad * (GM + 1) * sizeof(float);
    KN_ONCE_PER_DEVICE {
        KN_CUDA(cudaFuncSetAttribute(pg_small_kernel<GM, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
        KN_CUDA(cudaFuncSetAttribute(pg_small_kernel<GM, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
    }
    if (relu) pg_small_kernel<GM, true><<<(unsigned)gx, kThreads, smem, s>>>(rows, cols, vals, group_k, block_of, n_groups, G, K_pad, n_supers, tiles_per_super, X, ldx, Y, ldy, n_vecs, kn_current_peers());
    else      pg_small_kernel<GM, false><<<(unsigned)gx, kThreads, smem, s>>>(rows, cols, vals, group_k, block_of, n_groups, G, K_pad, n_supers, tiles_per_super, X, ldx, Y, ldy, n_vecs, kn_current_peers());
    KN_CHECK_LAUNCH();
    return KN_OK;
}

// run_start != null: narrow batches over the n_runs runs of the run table, NB = 1 << nb_shift (see pg_simt_kernel)
template <int RW>
int launch_pg(const int32_t *rows, const int32_t *cols, const float *vals, const int32_t *group_k, const int32_t *block_of, int64_t n_groups, int G, int K_pad,
              const float *X, int64_t ldx, float *Y, int64_t ldy, int64_t n_vecs, bool relu, cudaStream_t s,
              const int32_t *run_groups = nullptr, const int32_t *run_start = nullptr, int64_t n_runs = 0, int nb_shift = 0)
{
    constexpr int TM = 8 * RW;
    const size_t smem = sizeof(float) * kStages * (TM * KT + KT * TN);
    const int tiles_per_group = (G + TM - 1) / TM;
    const int64_t gx = (run_start ? n_runs : n_groups) * tiles_per_group, gy = run_start ? 1 : kn_cdiv(n_vecs, TN);
    KN_REQUIRE(gx * gy <= 0x7fffffffLL, "spmm_pg: grid too large");
    KN_ONCE_PER_DEVICE {
        KN_CUDA(cudaFuncSetAttribute(pg_simt_kernel<RW, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        KN_CUDA(cudaFuncSetAttribute(pg_simt_kernel<RW, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    }
    dim3 grid((unsigned)(gx * gy));
    if (relu) pg_simt_kernel<RW, true><<<grid, kThreads, smem, s>>>(rows, cols, vals, group_k, block_of, n_groups, G, K_pad, tiles_per_group, gx, gy, X, ldx, Y, ldy, n_vecs, kn_current_peers(),
                                                                    run_groups, run_start, nb_shift);
    else      pg_simt_kernel<RW, false><<<grid, kThreads, smem, s>>>(rows, cols, vals, group_k, block_of, n_groups, G, K_pad, tiles_per_group, gx, gy, X, ldx, Y, ldy, n_vecs, kn_current_peers(),
                                                                     run_groups, run_start, nb_shift);
    KN_CHECK_LAUNCH();
    return KN_OK;
}

int row_grid(int64_t n_rows) {
    const int64_t want = kn_cdiv(n_rows, kThreads / 32);
    const int64_t cap = (int64_t)kn_sm_count() * 8;
    return (int)(want < cap ? (want > 0 ? want : 1) : cap);
}
}  // namespace

KN_API int kn_csr_row_pattern_hash(const int64_t *indptr, const int32_t *indices, int64_t n_rows, uint64_t *hash, void *stream) {
    KN_REQUIRE(n_rows >= 0, "pattern_hash: negative row count");
    if (n_rows == 0) return KN_OK;
    KN_REQUIRE(indptr && hash, "pattern_hash: null pointer");
    row_pattern_hash_kernel<<<row_grid(n_rows), kThreads, 0, (cudaStream_t)stream>>>(indptr, indices, n_rows, hash);
    KN_CHECK_LAUNCH();
    return KN_OK;
}

KN_API int kn_pg_verify(const int64_t *indptr, const int32_t *indices, const int64_t *rows, const int64_t *leaders, int64_t n,
                        int32_t *mismatch, void *stream) {
    KN_REQUIRE(n >= 0, "pg_verify: negative count");
    if (n == 0) return KN_OK;
    KN_REQUIRE(indptr && rows && leaders && mismatch, "pg_verify: null pointer");
    pg_verify_kernel<<<row_grid(n), kThreads, 0, (cudaStream_t)stream>>>(indptr, indices, rows, leaders, n, mismatch);
    KN_CHECK_LAUNCH();
    return KN_OK;
}

KN_API int kn_pg_pack(const int64_t *indptr, const int32_t *indices, const float *data, const int64_t *rows,
                      int64_t n_groups, int32_t G, int32_t K_pad, int32_t *cols, float *vals, void *stream) {
    KN_REQUIRE(n_groups >= 0 && G > 0 && K_pad > 0 && K_pad % KT == 0, "pg_pack: bad shape (G=%d K_pad=%d)", G, K_pad);
    if (n_groups == 0) return KN_OK;
    KN_REQUIRE(indptr && indices && data && rows && cols && vals, "pg_pack: null pointer");
    pg_pack_kernel<<<row_grid(n_groups * G), kThreads, 0, (cudaStream_t)stream>>>(indptr, indices, data, rows, n_groups, G, K_pad, cols, vals);
    KN_CHECK_LAUNCH();
    return KN_OK;
}

KN_API int kn_splitk_reduce_f32(const float *part, int32_t S, int32_t G, const int32_t *rows, float *Y, int64_t ldy, int64_t n_vecs, uint32_t flags, const kn_peers *peers_arg, void *stream) {
    KnPeersScope peers_scope(peers_arg);
    if (!peers_scope.ok) return KN_ERR_INVALID_ARGUMENT;
    KN_REQUIRE(S > 0 && G > 0 && n_vecs >= 0 && ldy >= n_vecs, "splitk_reduce: bad shape (S=%d G=%d)", S, G);
    if (n_vecs == 0) return KN_OK;
    KN_REQUIRE(part && rows && Y, "splitk_reduce: null pointer");
    KN_REQUIRE(n_vecs % 4 == 0 && ldy % 4 == 0 && (((uintptr_t)part | (uintptr_t)Y) & 15) == 0, "splitk_reduce: n_vecs, ldy must be multiples of 4 and buffers 16-byte aligned");
    const int64_t total = (int64_t)G * (n_vecs / 4);
    const int64_t want = kn_cdiv(total, kThreads), cap = (int64_t)kn_sm_count() * 8;
    const unsigned grid = (unsigned)(want < cap ? want : cap);
    if (flags & KN_SPMM_RELU) splitk_reduce_kernel<true><<<grid, kThreads, 0, (cudaStream_t)stream>>>(part, S, G, rows, Y, ldy, n_vecs, kn_current_peers());
    else                      splitk_reduce_kernel<false><<<grid, kThreads, 0, (cudaStream_t)stream>>>(part, S, G, rows, Y, ldy, n_vecs, kn_current_peers());
    KN_CHECK_LAUNCH();
    return KN_OK;
}

KN_API int kn_spmm_pg_f32(const int32_t *rows, const int32_t *cols, const float *vals, const int32_t *group_k, const int32_t *block_of, int64_t n_groups, int32_t G, int32_t K_pad,
                          const float *X, int64_t ldx, float *Y, int64_t ldy, int64_t n_vecs, uint32_t flags, const kn_peers *peers_arg, void *stream) {
    KnPeersScope peers_scope(peers_arg);
    if (!peers_scope.ok) return KN_ERR_INVALID_ARGUMENT;
    KN_REQUIRE(n_groups >= 0 && G > 0 && K_pad > 0 && K_pad % KT == 0, "spmm_pg: bad shape (G=%d K_pad=%d)", G, K_pad);
    KN_REQUIRE(n_vecs >= 0 && ldx >= n_vecs && ldy >= n_vecs, "spmm_pg: bad leading dimension");
    if (n_groups == 0 || n_vecs == 0) return KN_OK;
    KN_REQUIRE(rows && cols && vals && X && Y, "spmm_pg: null pointer");
    KN_REQUIRE(n_vecs % 4 == 0 && ldx % 4 == 0 && ldy % 4 == 0 && (((uintptr_t)X | (uintptr_t)Y) & 15) == 0,
               "spmm_pg: n_vecs, ldx, ldy must be multiples of 4 and X, Y 16-byte aligned");
    cudaStream_t s = (cudaStream_t)stream;
    const bool relu = (flags & KN_SPMM_RELU) != 0;
    if (G <= 8 && K_pad <= 128)  return launch_small<8>(rows, cols, vals, group_k, block_of, n_groups, G, K_pad, X, ldx, Y, ldy, n_vecs, relu, s);
    if (G <= 16 && K_pad <= 128) return launch_small<16>(rows, cols, vals, group_k, block_of, n_groups, G, K_pad, X, ldx, Y, ldy, n_vecs, relu, s);
    if (G <= 8)  return launch_pg<1>(rows, cols, vals, group_k, block_of, n_groups, G, K_pad, X, ldx, Y, ldy, n_vecs, relu, s);
    if (G <= 16) return launch_pg<2>(rows, cols, vals, group_k, block_of, n_groups, G, K_pad, X, ldx, Y, ldy, n_vecs, relu, s);
    if (G <= 32) return launch_pg<4>(rows, cols, vals, group_k, block_of, n_groups, G, K_pad, X, ldx, Y, ldy, n_vecs, relu, s);
    if (G <= 64) return launch_pg<8>(rows, cols, vals, group_k, block_of, n_groups, G, K_pad, X, ldx, Y, ldy, n_vecs, relu, s);
    // pick the row tile (96 or 128) that wastes fewer padded rows
    const int waste96 = ((G + 95) / 96) * 96 - G, waste128 = ((G + 127) / 128) * 128 - G;
    if (waste96 < waste128) return launch_pg<12>(rows, cols, vals, group_k, block_of, n_groups, G, K_pad, X, ldx, Y, ldy, n_vecs, relu, s);
    return launch_pg<16>(rows, cols, vals, group_k, block_of, n_groups, G, K_pad, X, ldx, Y, ldy, n_vecs, relu, s);
}

KN_API int kn_spmm_pg_narrow_f32(const int32_t *rows, const int32_t *cols, const float *vals, const int32_t *group_k, const int32_t *block_of, int64_t n_groups, int32_t G, int32_t K_pad,
                                 const int32_t *run_groups, const int32_t *run_start, int64_t n_runs, int32_t row_form,
                                 const float *X, int64_t ldx, float *Y, int64_t ldy, int64_t n_vecs, uint32_t flags, const kn_peers *peers, void *stream) {
    KN_REQUIRE(peers == nullptr, "spmm_pg_narrow: no output peers (the fused row-sharded path pads its batch to the grouped kernels)");
    KN_REQUIRE(n_vecs >= 1 && n_vecs <= 32, "spmm_pg_narrow: n_vecs must be in 1..32 (got %lld)", (long long)n_vecs);
    KN_REQUIRE(ldx >= n_vecs && ldy >= n_vecs, "spmm_pg_narrow: bad leading dimension");
    KN_REQUIRE(n_groups >= 0 && G > 0 && K_pad > 0 && K_pad % KT == 0, "spmm_pg_narrow: bad shape (G=%d K_pad=%d)", G, K_pad);
    KN_REQUIRE(row_form == 0 || (row_form == 1 && n_vecs <= 8), "spmm_pg_narrow: the row form (row_form = 1) serves n_vecs <= 8 (row_form=%d)", row_form);
    if (n_groups == 0) return KN_OK;
    KN_REQUIRE(run_groups && run_start && n_runs > 0 && n_runs <= n_groups, "spmm_pg_narrow: empty run table (%lld runs for %lld groups)", (long long)n_runs, (long long)n_groups);
    KN_REQUIRE(rows && cols && vals && X && Y, "spmm_pg_narrow: null pointer");
    KnPeersScope peers_scope(nullptr);
    cudaStream_t s = (cudaStream_t)stream;
    const bool relu = (flags & KN_SPMM_RELU) != 0;
    if (row_form) {
        KnGroupRows gr;
        (gr.rows = rows, gr.cols = cols, gr.group_k = group_k, gr.block_of = block_of, gr.vals = vals, gr.G = G, gr.K_pad = K_pad);
        return kn_spmm_group_rows(gr, n_groups * G, X, ldx, Y, ldy, (int)n_vecs, relu, s);
    }
    int nb_shift = 0;
    while ((1 << nb_shift) < n_vecs) nb_shift++;
    static_assert(kNarrowMaxRW == 4, "the dispatch below stops at pg_simt<4>");
    if (G <= 8)  return launch_pg<1>(rows, cols, vals, group_k, block_of, n_groups, G, K_pad, X, ldx, Y, ldy, n_vecs, relu, s, run_groups, run_start, n_runs, nb_shift);
    if (G <= 16) return launch_pg<2>(rows, cols, vals, group_k, block_of, n_groups, G, K_pad, X, ldx, Y, ldy, n_vecs, relu, s, run_groups, run_start, n_runs, nb_shift);
    return launch_pg<4>(rows, cols, vals, group_k, block_of, n_groups, G, K_pad, X, ldx, Y, ldy, n_vecs, relu, s, run_groups, run_start, n_runs, nb_shift);
}
