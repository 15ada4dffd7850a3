// common.cuh -- shared helpers for libkeynet_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include "../../include/keynet_b200.h"

#define KN_API extern "C" __attribute__((visibility("default")))

// thread-local last-error text, set by every failing entry point (abi.cu)
void kn_set_error(const char *fmt, ...);

#define KN_REQUIRE(cond, ...)                                   \
    do {                                                        \
        if (!(cond)) {                                          \
            kn_set_error(__VA_ARGS__);                          \
            return KN_ERR_INVALID_ARGUMENT;                     \
        }                                                       \
    } while (0)

#define KN_CUDA(call)                                                                   \
    do {                                                                                \
        cudaError_t e_ = (call);                                                        \
        if (e_ != cudaSuccess) {                                                        \
            kn_set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
            return KN_ERR_CUDA;                                                         \
        }                                                                               \
    } while (0)

#define KN_CHECK_LAUNCH() KN_CUDA(cudaGetLastError())

// cudaFuncSetAttribute belongs to the function ON ONE DEVICE: a process that drives several GPUs must set it on each.
// KN_ONCE_PER_DEVICE { ... } runs its body the first time the enclosing call site (one per template instantiation) is
// reached with a given current device.
struct KnOncePerDevice {
    bool done[64] = {false};
    bool first() {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return true;
        if (done[dev]) return false;
        done[dev] = true;
        return true;
    }
};
#define KN_ONCE_PER_DEVICE static KnOncePerDevice kn_once_; if (kn_once_.first())

static inline int64_t kn_cdiv(int64_t a, int64_t b) { return (a + b - 1) / b; }

// Output replication for the fused SpMM + all-gather (K5): when n > 0 every epilogue stores its rows to all n buffers
// (its own and the peers' NVLink-mapped ones, same layout everywhere) instead of the single Y it was given.
// row_mask (optional, device memory, one byte per output row of Y): bit p set = peer p reads this row in the next layer;
// rows nobody else needs never cross NVLink (the all-gather becomes a halo exchange).  null = every row to every peer.
struct KnPeers { int n; float *y[8]; const unsigned char *row_mask; };
// Kernels take it as `const __grid_constant__ KnPeers`, so the pointer list is read straight from the constant bank
// (a plain by-value struct indexed at run time would be copied to local memory and slow every epilogue).
// The mask is loaded by kn_peer_mask() BEFORE the store loop (a load placed between stores is serialised behind them: the
// compiler must assume the stores alias it, and each row then pays a full L2 round trip).
__device__ __forceinline__ unsigned kn_peer_mask(const KnPeers &peers, int64_t row) {
    return (peers.n > 0 && peers.row_mask != nullptr) ? (unsigned)__ldg(peers.row_mask + row) : 0xffu;
}
#define KN_FOR_EACH_DEST(peers, Y, mask, dst)                                                 \
    for (unsigned p_ = 0, np_ = ((peers).n > 0 ? (peers).n : 1); p_ < np_; p_++)              \
        if (((mask) >> p_) & 1u)                                                              \
            if (float *dst = ((peers).n > 0 ? (peers).y[p_] : (Y)); true)
// Every kn_spmm_* entry point takes the destinations as an explicit argument (const kn_peers *, include/keynet_b200.h) and
// opens a KnPeersScope for the duration of the call; its launch helpers read the validated device-side form back with
// kn_current_peers().  Nothing survives the call: there is no state shared between calls or threads.
KnPeers kn_current_peers();
struct KnPeersScope {
    KnPeers saved;
    bool ok;
    explicit KnPeersScope(const kn_peers *p);
    ~KnPeersScope();
};

// Rows of one pattern-group class (csrc/pgroup.cu) as the CSR kernel's row source: row i of the product is row i % G of
// group i / G, its entries the group's first group_k[g] columns cols[g][k] with values vals[block_of[g]][i % G][k], written to
// Y[rows[i]].  The row form of narrow batches (kn_spmm_pg_narrow_f32): one warp per row, lanes over the row's columns.
struct KnGroupRows {
    const int32_t *rows = nullptr, *cols = nullptr, *group_k = nullptr, *block_of = nullptr;
    const float *vals = nullptr;
    int G = 0, K_pad = 0;
};
// n_rows = n_groups * G rows, 1 <= n_vecs <= 8 (csrc/spmm.cu); plain stores, no peers
int kn_spmm_group_rows(const KnGroupRows &gr, int64_t n_rows, const float *X, int64_t ldx, float *Y, int64_t ldy, int n_vecs, bool relu, cudaStream_t s);

// number of SMs of the current device (cached); B200 = 148
int kn_sm_count();

// streaming (read-once) 128-bit load that does not allocate in L1
__device__ __forceinline__ int4 kn_ldg_stream_int4(const int4 *p) {
    int4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.s32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}
__device__ __forceinline__ int kn_ldg_stream_i32(const int *p) {
    int r;
    asm volatile("ld.global.nc.L1::no_allocate.s32 %0, [%1];" : "=r"(r) : "l"(p));
    return r;
}
__device__ __forceinline__ float kn_ldg_stream_f32(const float *p) {
    float r;
    asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(r) : "l"(p));
    return r;
}

// CTA rasterisation shared by the grouped kernels: a 1-D grid enumerates (work item, batch tile) pairs so that
// the batch tiles of one work item (pattern group / row tile) run back to back inside a super-tile of `S` batch
// tiles -- its weight block is fetched from HBM once per super-tile and then served from L2 -- while the X rows
// touched by neighbouring work items of the same super-tile (S*tile columns wide) stay L2-resident as well.
struct KnRaster { int64_t item; int64_t tile; };
__device__ __forceinline__ KnRaster kn_raster(int64_t linear, int64_t n_items, int64_t n_tiles, int64_t S) {
    const int64_t full = n_tiles / S, rem = n_tiles - full * S, per_super = S * n_items;
    KnRaster r;
    if (linear < full * per_super) {
        const int64_t sup = linear / per_super, w = linear - sup * per_super;
        r.item = w / S; r.tile = sup * S + (w - r.item * S);
    } else {
        const int64_t w = linear - full * per_super;
        r.item = w / rem; r.tile = full * S + (w - r.item * rem);
    }
    return r;
}

// normalised bitonic sort of n (key,val) pairs by key, ascending; works for any n >= 0
template <typename KeyPtr, typename ValPtr>
__device__ __forceinline__ void bitonic_sort_pairs(KeyPtr keys, ValPtr vals, int n) {
    if (n < 2) return;
    int np2 = 1;
    while (np2 < n) np2 <<= 1;
    for (int k = 2; k <= np2; k <<= 1) {
        // first step of the stage: partner is the mirror inside the k-block
        for (int i = threadIdx.x; i < np2 / 2; i += blockDim.x) {
            const int blk = i / (k / 2), off = i - blk * (k / 2);
            const int a = blk * k + off, b = blk * k + (k - 1 - off);
            if (b < n) {
                const int32_t ka = keys[a], kb = keys[b];
                if (ka > kb) { keys[a] = kb; keys[b] = ka; const float t = vals[a]; vals[a] = vals[b]; vals[b] = t; }
            }
        }
        __syncthreads();
        for (int j = k / 4; j > 0; j >>= 1) {
            for (int i = threadIdx.x; i < np2 / 2; i += blockDim.x) {
                const int a = 2 * j * (i / j) + (i % j), b = a + j;
                if (b < n) {
                    const int32_t ka = keys[a], kb = keys[b];
                    if (ka > kb) { keys[a] = kb; keys[b] = ka; const float t = vals[a]; vals[a] = vals[b]; vals[b] = t; }
                }
            }
            __syncthreads();
        }
    }
}

