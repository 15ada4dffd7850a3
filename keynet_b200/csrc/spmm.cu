// spmm.cu -- CSR x dense-batch product with fused ReLU (kernel K1 of SURVEY.md 2.2).
//
//   Y[R][N] = W_hat[R][C] . X[C][N]        fp32, X/Y row-major (features x batch)
//
// Replaces SparseMatrix.torchdot (reference keynet/sparse.py:488-492 -> scipy csr_matvecs).
//
// Two layouts, picked by batch width N:
//   * rowwarp<V>  (N > 8): one warp per output row; the 32 lanes span 32*V consecutive batch
//     columns, so every gathered X row segment is one coalesced 128*V-byte read and every lane
//     owns V accumulators.  The row's (col,val) pairs are read 32 at a time with coalesced
//     loads, parked in shared memory and broadcast back with one LDS.64 per entry.  Each output
//     element is accumulated sequentially in stored order, like the reference.
//     grid = (row blocks, batch chunks) with row blocks fastest, so the CTAs resident at any
//     moment work on the SAME batch chunk: that chunk's slab of X (C x 128V bytes) is what has
//     to live in L2, not all of X.
//   * lanes_nnz<NB> (N <= 8): one warp per row, lanes stride over the row's entries (coalesced
//     index/value reads), NB accumulators per lane, warp-shuffle tree reduction at the end.  It also takes its rows from a
//     pattern-group class (KnGroupRows, common.cuh): the row form of narrow batches on layers without a CSR.
#include "common.cuh"
#include <stdlib.h>

namespace {

constexpr int kWarps = 8;   // 256 threads per CTA

template <int V> struct VecT;
template <> struct VecT<1> { using type = float; };
template <> struct VecT<2> { using type = float2; };
template <> struct VecT<4> { using type = float4; };

template <int V>
__device__ __forceinline__ void fma_vec(float (&acc)[V], float w, const float *__restrict__ xp) {
    if constexpr (V == 4) {
        const float4 x = __ldg(reinterpret_cast<const float4 *>(xp));
        acc[0] = fmaf(w, x.x, acc[0]); acc[1] = fmaf(w, x.y, acc[1]);
        acc[2] = fmaf(w, x.z, acc[2]); acc[3] = fmaf(w, x.w, acc[3]);
    } else if constexpr (V == 2) {
        const float2 x = __ldg(reinterpret_cast<const float2 *>(xp));
        acc[0] = fmaf(w, x.x, acc[0]); acc[1] = fmaf(w, x.y, acc[1]);
    } else {
        acc[0] = fmaf(w, __ldg(xp), acc[0]);
    }
}

template <int V, bool RELU>
__global__ void __launch_bounds__(kWarps * 32)
spmm_rowwarp_kernel(const int64_t *__restrict__ indptr, const int32_t *__restrict__ indices,
                    const float *__restrict__ data, int64_t n_rows,
                    const float *__restrict__ X, int64_t ldx, float *__restrict__ Y, int64_t ldy, int64_t n_vecs,
                    const int32_t *__restrict__ out_rows, const __grid_constant__ KnPeers peers)
{
    __shared__ int2 s_ent[kWarps][32];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * kWarps + warp;
    if (row >= n_rows) return;                                   // warp-uniform
    const int64_t n0 = ((int64_t)blockIdx.y * 32 + lane) * V;
    const bool active = n0 < n_vecs;                             // host guarantees n_vecs % V == 0
    const int64_t beg = indptr[row], end = indptr[row + 1];
    const float *__restrict__ xbase = X + (active ? n0 : 0);

    float acc[V];
#pragma unroll
    for (int i = 0; i < V; i++) acc[i] = 0.0f;

    for (int64_t base = beg; base < end; base += 32) {
        const int64_t e = base + lane;
        int c = 0; float w = 0.0f;
        if (e < end) { c = kn_ldg_stream_i32(indices + e); w = kn_ldg_stream_f32(data + e); }
        s_ent[warp][lane] = make_int2(c, __float_as_int(w));
        __syncwarp();
        const int cnt = (int)((end - base) < 32 ? (end - base) : 32);
        if (active) {
            int t = 0;
            for (; t + 4 <= cnt; t += 4) {
                const int2 p0 = s_ent[warp][t], p1 = s_ent[warp][t + 1], p2 = s_ent[warp][t + 2], p3 = s_ent[warp][t + 3];
                if constexpr (V == 4) {
                    // issue the four gathers before the FMAs (memory-level parallelism)
                    const float4 x0 = __ldg(reinterpret_cast<const float4 *>(xbase + (int64_t)p0.x * ldx));
                    const float4 x1 = __ldg(reinterpret_cast<const float4 *>(xbase + (int64_t)p1.x * ldx));
                    const float4 x2 = __ldg(reinterpret_cast<const float4 *>(xbase + (int64_t)p2.x * ldx));
                    const float4 x3 = __ldg(reinterpret_cast<const float4 *>(xbase + (int64_t)p3.x * ldx));
                    const float w0 = __int_as_float(p0.y), w1 = __int_as_float(p1.y), w2 = __int_as_float(p2.y), w3 = __int_as_float(p3.y);
                    acc[0] = fmaf(w0, x0.x, acc[0]); acc[1] = fmaf(w0, x0.y, acc[1]); acc[2] = fmaf(w0, x0.z, acc[2]); acc[3] = fmaf(w0, x0.w, acc[3]);
                    acc[0] = fmaf(w1, x1.x, acc[0]); acc[1] = fmaf(w1, x1.y, acc[1]); acc[2] = fmaf(w1, x1.z, acc[2]); acc[3] = fmaf(w1, x1.w, acc[3]);
                    acc[0] = fmaf(w2, x2.x, acc[0]); acc[1] = fmaf(w2, x2.y, acc[1]); acc[2] = fmaf(w2, x2.z, acc[2]); acc[3] = fmaf(w2, x2.w, acc[3]);
                    acc[0] = fmaf(w3, x3.x, acc[0]); acc[1] = fmaf(w3, x3.y, acc[1]); acc[2] = fmaf(w3, x3.z, acc[2]); acc[3] = fmaf(w3, x3.w, acc[3]);
                } else {
                    fma_vec<V>(acc, __int_as_float(p0.y), xbase + (int64_t)p0.x * ldx);
                    fma_vec<V>(acc, __int_as_float(p1.y), xbase + (int64_t)p1.x * ldx);
                    fma_vec<V>(acc, __int_as_float(p2.y), xbase + (int64_t)p2.x * ldx);
                    fma_vec<V>(acc, __int_as_float(p3.y), xbase + (int64_t)p3.x * ldx);
                }
            }
            for (; t < cnt; t++) {
                const int2 p = s_ent[warp][t];
                fma_vec<V>(acc, __int_as_float(p.y), xbase + (int64_t)p.x * ldx);
            }
        }
        __syncwarp();
    }
    if (active) {
        if (RELU) {
#pragma unroll
            for (int i = 0; i < V; i++) acc[i] = fmaxf(acc[i], 0.0f);
        }
        const int64_t yrow = out_rows ? (int64_t)out_rows[row] : row;
        const int64_t yoff = yrow * ldy + n0;
        KN_FOR_EACH_DEST(peers, Y, kn_peer_mask(peers, yrow), yb) {                         // fused all-gather: the row goes to every peer's buffer
            float *yp = yb + yoff;
            if constexpr (V == 4) *reinterpret_cast<float4 *>(yp) = make_float4(acc[0], acc[1], acc[2], acc[3]);
            else if constexpr (V == 2) *reinterpret_cast<float2 *>(yp) = make_float2(acc[0], acc[1]);
            else yp[0] = acc[0];
        }
    }
}

// Wide variant for large batches: the warp covers WS consecutive 128-column segments (WS x 512 B contiguous per gathered
// X row).  A 512-byte piece per row keeps too few bytes in flight per warp for short rows (a permutation key has ONE entry
// per row: three dependent loads to move 512 B) and opens a new DRAM page per piece; 2 KB per row quadruples the bytes in
// flight and reads whole pages.
template <int WS, bool RELU>
__global__ void __launch_bounds__(kWarps * 32, (WS <= 2) ? 6 : 4)
spmm_rowwarp_wide_kernel(const int64_t *__restrict__ indptr, const int32_t *__restrict__ indices,
                         const float *__restrict__ data, int64_t n_rows,
                         const float *__restrict__ X, int64_t ldx, float *__restrict__ Y, int64_t ldy, int64_t n_vecs,
                         const int32_t *__restrict__ out_rows, const __grid_constant__ KnPeers peers)
{
    __shared__ int2 s_ent[kWarps][32];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * kWarps + warp;
    if (row >= n_rows) return;                                   // warp-uniform
    const int64_t n0 = (int64_t)blockIdx.y * (WS * 128) + lane * 4;
    const int64_t beg = indptr[row], end = indptr[row + 1];
    bool act[WS];
#pragma unroll
    for (int s = 0; s < WS; s++) act[s] = n0 + s * 128 < n_vecs;
    float acc[WS][4];
#pragma unroll
    for (int s = 0; s < WS; s++) { acc[s][0] = acc[s][1] = acc[s][2] = acc[s][3] = 0.0f; }

    for (int64_t base = beg; base < end; base += 32) {
        const int64_t e = base + lane;
        int c = 0; float w = 0.0f;
        if (e < end) { c = kn_ldg_stream_i32(indices + e); w = kn_ldg_stream_f32(data + e); }
        s_ent[warp][lane] = make_int2(c, __float_as_int(w));
        __syncwarp();
        const int cnt = (int)((end - base) < 32 ? (end - base) : 32);
        int t = 0;
        for (; t + 2 <= cnt; t += 2) {                                         // 2 x WS gathers in flight per lane
            const int2 p0 = s_ent[warp][t], p1 = s_ent[warp][t + 1];
            const float *__restrict__ x0p = X + (int64_t)p0.x * ldx + n0, *__restrict__ x1p = X + (int64_t)p1.x * ldx + n0;
            float4 x0[WS], x1[WS];
#pragma unroll
            for (int s = 0; s < WS; s++) x0[s] = act[s] ? __ldg(reinterpret_cast<const float4 *>(x0p + s * 128)) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int s = 0; s < WS; s++) x1[s] = act[s] ? __ldg(reinterpret_cast<const float4 *>(x1p + s * 128)) : make_float4(0.f, 0.f, 0.f, 0.f);
            const float w0 = __int_as_float(p0.y), w1 = __int_as_float(p1.y);
#pragma unroll
            for (int s = 0; s < WS; s++) {
                acc[s][0] = fmaf(w0, x0[s].x, acc[s][0]); acc[s][1] = fmaf(w0, x0[s].y, acc[s][1]); acc[s][2] = fmaf(w0, x0[s].z, acc[s][2]); acc[s][3] = fmaf(w0, x0[s].w, acc[s][3]);
            }
#pragma unroll
            for (int s = 0; s < WS; s++) {
                acc[s][0] = fmaf(w1, x1[s].x, acc[s][0]); acc[s][1] = fmaf(w1, x1[s].y, acc[s][1]); acc[s][2] = fmaf(w1, x1[s].z, acc[s][2]); acc[s][3] = fmaf(w1, x1[s].w, acc[s][3]);
            }
        }
        if (t < cnt) {
            const int2 p0 = s_ent[warp][t];
            const float *__restrict__ x0p = X + (int64_t)p0.x * ldx + n0;
            const float w0 = __int_as_float(p0.y);
#pragma unroll
            for (int s = 0; s < WS; s++) {
                const float4 x = act[s] ? __ldg(reinterpret_cast<const float4 *>(x0p + s * 128)) : make_float4(0.f, 0.f, 0.f, 0.f);
                acc[s][0] = fmaf(w0, x.x, acc[s][0]); acc[s][1] = fmaf(w0, x.y, acc[s][1]); acc[s][2] = fmaf(w0, x.z, acc[s][2]); acc[s][3] = fmaf(w0, x.w, acc[s][3]);
            }
        }
        __syncwarp();
    }
    const int64_t yrow = out_rows ? (int64_t)out_rows[row] : row;
    const unsigned pmask = kn_peer_mask(peers, yrow);
#pragma unroll
    for (int s = 0; s < WS; s++) {
        if (act[s]) {
            float4 o = make_float4(acc[s][0], acc[s][1], acc[s][2], acc[s][3]);
            if (RELU) { o.x = fmaxf(o.x, 0.0f); o.y = fmaxf(o.y, 0.0f); o.z = fmaxf(o.z, 0.0f); o.w = fmaxf(o.w, 0.0f); }
            KN_FOR_EACH_DEST(peers, Y, pmask, yb) *reinterpret_cast<float4 *>(yb + yrow * ldy + n0 + s * 128) = o;
        }
    }
}

template <int NB, bool RELU>
__global__ void __launch_bounds__(kWarps * 32)
spmm_lanes_nnz_kernel(const int64_t *__restrict__ indptr, const int32_t *__restrict__ indices,
                      const float *__restrict__ data, int64_t n_rows,
                      const float *__restrict__ X, int64_t ldx, float *__restrict__ Y, int64_t ldy, int n_vecs,
                      const int32_t *__restrict__ out_rows, const __grid_constant__ KnPeers peers, const KnGroupRows gr)
{
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * kWarps + warp;
    if (row >= n_rows) return;
    int64_t beg, end, yrow;
    if (gr.cols == nullptr) {
        beg = indptr[row]; end = indptr[row + 1];
        yrow = out_rows ? (int64_t)out_rows[row] : row;
    } else {                                       // row row % G of pattern group row / G: its entries start at offset 0
        const int64_t g = row / gr.G, blk = gr.block_of ? (int64_t)__ldg(gr.block_of + g) : g;
        indices = gr.cols + g * gr.K_pad;
        data = gr.vals + (blk * gr.G + (row - g * gr.G)) * gr.K_pad;
        beg = 0; end = gr.group_k ? __ldg(gr.group_k + g) : gr.K_pad;
        yrow = __ldg(gr.rows + row);
    }
    const unsigned pmask = kn_peer_mask(peers, yrow);
    float acc[NB];
#pragma unroll
    for (int n = 0; n < NB; n++) acc[n] = 0.0f;
    for (int64_t e = beg + lane; e < end; e += 32) {
        const int c = kn_ldg_stream_i32(indices + e);
        const float w = kn_ldg_stream_f32(data + e);
        const float *__restrict__ xp = X + (int64_t)c * ldx;
#pragma unroll
        for (int n = 0; n < NB; n++)
            if (n < n_vecs) acc[n] = fmaf(w, __ldg(xp + n), acc[n]);
    }
#pragma unroll
    for (int n = 0; n < NB; n++) {
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) acc[n] += __shfl_xor_sync(0xffffffffu, acc[n], off);
    }
#pragma unroll
    for (int n = 0; n < NB; n++)
        if (lane == n && n < n_vecs) {
            const float o = RELU ? fmaxf(acc[n], 0.0f) : acc[n];
            KN_FOR_EACH_DEST(peers, Y, pmask, yb) yb[yrow * ldy + n] = o;
        }
}

template <int V>
int launch_rowwarp(const int64_t *indptr, const int32_t *indices, const float *data, int64_t n_rows,
                   const float *X, int64_t ldx, float *Y, int64_t ldy, int64_t n_vecs, bool relu, const int32_t *out_rows, cudaStream_t s)
{
    const int64_t gx = kn_cdiv(n_rows, kWarps), gy = kn_cdiv(n_vecs, 32 * V);
    KN_REQUIRE(gx <= 0x7fffffffLL && gy <= 65535, "spmm: grid too large (rows=%lld, n_vecs=%lld)", (long long)n_rows, (long long)n_vecs);
    dim3 grid((unsigned)gx, (unsigned)gy);
    if (relu) spmm_rowwarp_kernel<V, true><<<grid, kWarps * 32, 0, s>>>(indptr, indices, data, n_rows, X, ldx, Y, ldy, n_vecs, out_rows, kn_current_peers());
    else      spmm_rowwarp_kernel<V, false><<<grid, kWarps * 32, 0, s>>>(indptr, indices, data, n_rows, X, ldx, Y, ldy, n_vecs, out_rows, kn_current_peers());
    KN_CHECK_LAUNCH();
    return KN_OK;
}

template <int WS>
int launch_rowwarp_wide(const int64_t *indptr, const int32_t *indices, const float *data, int64_t n_rows,
                        const float *X, int64_t ldx, float *Y, int64_t ldy, int64_t n_vecs, bool relu, const int32_t *out_rows, cudaStream_t s)
{
    const int64_t gx = kn_cdiv(n_rows, kWarps), gy = kn_cdiv(n_vecs, 128 * WS);
    KN_REQUIRE(gx <= 0x7fffffffLL && gy <= 65535, "spmm: grid too large (rows=%lld, n_vecs=%lld)", (long long)n_rows, (long long)n_vecs);
    dim3 grid((unsigned)gx, (unsigned)gy);
    if (relu) spmm_rowwarp_wide_kernel<WS, true><<<grid, kWarps * 32, 0, s>>>(indptr, indices, data, n_rows, X, ldx, Y, ldy, n_vecs, out_rows, kn_current_peers());
    else      spmm_rowwarp_wide_kernel<WS, false><<<grid, kWarps * 32, 0, s>>>(indptr, indices, data, n_rows, X, ldx, Y, ldy, n_vecs, out_rows, kn_current_peers());
    KN_CHECK_LAUNCH();
    return KN_OK;
}

template <int NB>
int launch_lanes(const int64_t *indptr, const int32_t *indices, const float *data, int64_t n_rows,
                 const float *X, int64_t ldx, float *Y, int64_t ldy, int n_vecs, bool relu, const int32_t *out_rows, cudaStream_t s,
                 const KnGroupRows &gr = KnGroupRows())
{
    const int64_t gx = kn_cdiv(n_rows, kWarps);
    KN_REQUIRE(gx <= 0x7fffffffLL, "spmm: too many rows (%lld)", (long long)n_rows);
    if (relu) spmm_lanes_nnz_kernel<NB, true><<<(unsigned)gx, kWarps * 32, 0, s>>>(indptr, indices, data, n_rows, X, ldx, Y, ldy, n_vecs, out_rows, kn_current_peers(), gr);
    else      spmm_lanes_nnz_kernel<NB, false><<<(unsigned)gx, kWarps * 32, 0, s>>>(indptr, indices, data, n_rows, X, ldx, Y, ldy, n_vecs, out_rows, kn_current_peers(), gr);
    KN_CHECK_LAUNCH();
    return KN_OK;
}

}  // namespace

int kn_spmm_group_rows(const KnGroupRows &gr, int64_t n_rows, const float *X, int64_t ldx, float *Y, int64_t ldy, int n_vecs, bool relu, cudaStream_t s)
{
    if (n_vecs == 1) return launch_lanes<1>(nullptr, nullptr, nullptr, n_rows, X, ldx, Y, ldy, n_vecs, relu, nullptr, s, gr);
    if (n_vecs == 2) return launch_lanes<2>(nullptr, nullptr, nullptr, n_rows, X, ldx, Y, ldy, n_vecs, relu, nullptr, s, gr);
    if (n_vecs <= 4) return launch_lanes<4>(nullptr, nullptr, nullptr, n_rows, X, ldx, Y, ldy, n_vecs, relu, nullptr, s, gr);
    return launch_lanes<8>(nullptr, nullptr, nullptr, n_rows, X, ldx, Y, ldy, n_vecs, relu, nullptr, s, gr);
}

static int spmm_csr_impl(const int64_t *indptr, const int32_t *indices, const float *data,
                         int64_t n_rows, int64_t n_cols, const int32_t *out_rows,
                         const float *X, int64_t ldx, float *Y, int64_t ldy, int64_t n_vecs,
                         uint32_t flags, void *stream)
{
    KN_REQUIRE(n_rows >= 0 && n_cols >= 0 && n_vecs >= 0, "spmm: negative dimension");
    KN_REQUIRE(ldx >= n_vecs && ldy >= n_vecs, "spmm: leading dimension smaller than n_vecs (ldx=%lld ldy=%lld n_vecs=%lld)",
               (long long)ldx, (long long)ldy, (long long)n_vecs);
    if (n_rows == 0 || n_vecs == 0) return KN_OK;
    KN_REQUIRE(indptr && X && Y, "spmm: null pointer");
    KN_REQUIRE(X != Y, "spmm: X and Y must not alias");
    cudaStream_t s = (cudaStream_t)stream;
    const bool relu = (flags & KN_SPMM_RELU) != 0;
    if (n_vecs <= 8) {
        const int nv = (int)n_vecs;
        if (nv == 1) return launch_lanes<1>(indptr, indices, data, n_rows, X, ldx, Y, ldy, nv, relu, out_rows, s);
        if (nv == 2) return launch_lanes<2>(indptr, indices, data, n_rows, X, ldx, Y, ldy, nv, relu, out_rows, s);
        if (nv <= 4) return launch_lanes<4>(indptr, indices, data, n_rows, X, ldx, Y, ldy, nv, relu, out_rows, s);
        return launch_lanes<8>(indptr, indices, data, n_rows, X, ldx, Y, ldy, nv, relu, out_rows, s);
    }
    const uintptr_t align = (uintptr_t)X | (uintptr_t)Y;
    static const int wide = getenv("KN_CSR_WIDE") ? atoi(getenv("KN_CSR_WIDE")) : 2;
    if (n_vecs % 4 == 0 && ldx % 4 == 0 && ldy % 4 == 0 && (align & 15) == 0 && n_vecs >= 2048 && wide > 1) {
        // enough batch columns to fill the machine with 512-column warps (kn_cdiv(n_rows, 8) x n_vecs / 512 CTAs)
        if (wide == 2) return launch_rowwarp_wide<2>(indptr, indices, data, n_rows, X, ldx, Y, ldy, n_vecs, relu, out_rows, s);
        return launch_rowwarp_wide<4>(indptr, indices, data, n_rows, X, ldx, Y, ldy, n_vecs, relu, out_rows, s);
    }
    if (n_vecs % 4 == 0 && ldx % 4 == 0 && ldy % 4 == 0 && (align & 15) == 0 && n_vecs >= 128)
        return launch_rowwarp<4>(indptr, indices, data, n_rows, X, ldx, Y, ldy, n_vecs, relu, out_rows, s);
    if (n_vecs % 2 == 0 && ldx % 2 == 0 && ldy % 2 == 0 && (align & 7) == 0 && n_vecs >= 64)
        return launch_rowwarp<2>(indptr, indices, data, n_rows, X, ldx, Y, ldy, n_vecs, relu, out_rows, s);
    return launch_rowwarp<1>(indptr, indices, data, n_rows, X, ldx, Y, ldy, n_vecs, relu, out_rows, s);
}

KN_API int kn_spmm_csr_f32(const int64_t *indptr, const int32_t *indices, const float *data,
                           int64_t n_rows, int64_t n_cols,
                           const float *X, int64_t ldx, float *Y, int64_t ldy, int64_t n_vecs,
                           uint32_t flags, const kn_peers *peers_arg, void *stream)
{
    KnPeersScope peers_scope(peers_arg);
    if (!peers_scope.ok) return KN_ERR_INVALID_ARGUMENT;
    return spmm_csr_impl(indptr, indices, data, n_rows, n_cols, nullptr, X, ldx, Y, ldy, n_vecs, flags, stream);
}

KN_API int kn_spmm_csr_rows_f32(const int64_t *indptr, const int32_t *indices, const float *data,
                                int64_t n_rows, int64_t n_cols, const int32_t *out_rows,
                                const float *X, int64_t ldx, float *Y, int64_t ldy, int64_t n_vecs,
                                uint32_t flags, const kn_peers *peers_arg, void *stream)
{
    KnPeersScope peers_scope(peers_arg);
    if (!peers_scope.ok) return KN_ERR_INVALID_ARGUMENT;
    return spmm_csr_impl(indptr, indices, data, n_rows, n_cols, out_rows, X, ldx, Y, ldy, n_vecs, flags, stream);
}
