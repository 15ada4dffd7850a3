/*
 * keynet_b200.h -- C ABI of libkeynet_b200.so: the B200 (sm_100a) implementation of the
 * keyed-layer forward path of visym/keynet.
 *
 * The reference has no FFI: its operator boundary is the Python `SparseMatrix` protocol
 * (keynet/sparse.py:419-514) plus the key-compile call site `A.dot(W).dot(Ainv)`
 * (keynet/layer.py:35,46,59,70) and the Toeplitz builders (keynet/sparse.py:122-212).  Each
 * entry point below names the reference interface it replaces.  The ctypes binding a
 * maintainer would add to the reference is shown in INTEGRATION.md.
 *
 * Conventions
 *   - every pointer is caller-owned DEVICE memory unless the name ends in `_host`;
 *   - CSR: `indptr` int64 [n_rows+1] (absolute offsets into indices/data, so a row shard is
 *     just `indptr + row_begin`), `indices` int32, `data` float32;
 *   - dense operands are row-major: X is [n_cols][ldx], Y is [n_rows][ldy], n_vecs <= ld;
 *     this is the reference's `W.torchdot(x.t())` operand (features x batch);
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream); every call
 *     is asynchronous on that stream and re-entrant;
 *   - return value: 0 on success, negative kn_status on failure; never throws.  The message
 *     for the calling thread's last failure is kn_last_error().
 *   - two-phase builders: `*_count` writes per-row entry counts, the caller scans them with
 *     kn_exclusive_scan_i64, allocates indices/data, then calls `*_fill`.
 */
#ifndef KEYNET_B200_H
#define KEYNET_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KN_ABI_VERSION 2

typedef enum {
    KN_OK = 0,
    KN_ERR_INVALID_ARGUMENT = -1,
    KN_ERR_CUDA = -2,
    KN_ERR_UNSUPPORTED = -3
} kn_status;

/* flags for kn_spmm_csr_f32 */
#define KN_SPMM_RELU 1u        /* fuse max(y,0): the unkeyed nn.ReLU appended at keynet/system.py:92 */

int kn_abi_version(void);
const char *kn_last_error(void);

/* Device facts used to size grids (returns KN_ERR_CUDA if no device). */
int kn_device_info(int *sm_count, int *cc_major, int *cc_minor, int64_t *total_mem_bytes);

/* ---- fused SpMM + all-gather (kernel K5) --------------------------------------------------------------
 * Every kn_spmm_* entry point (and kn_splitk_reduce_f32) takes `const kn_peers *peers`.  NULL (or n = 0): each output row
 * is stored to the Y argument.  Otherwise each output row is stored to ALL n buffers y[i] instead -- y[i] = device address
 * on rank i of the same Y argument (NVLink peer mappings, e.g. torch symmetric memory; the own rank is one of them): a
 * row-sharded layer writes its slot of every rank's gathered activation buffer from the epilogue, so no separate
 * all-gather runs.  row_mask (optional, DEVICE memory, one byte per output row of Y): bit i set = rank i reads that row in
 * its next layer; only those copies are stored, so a conv layer sharded by pixels sends its halo rows to the neighbouring
 * shard and nothing else -- the all-gather of keynet's row-sharded layers (BASELINE north_star) degenerates to a halo
 * exchange.  The argument is read during the call only: no state is kept between calls or threads. */
typedef struct kn_peers {
    int32_t n;                  /* destinations, 0..8 */
    int32_t reserved;
    uint64_t y[8];              /* device addresses */
    const uint8_t *row_mask;    /* device memory or NULL */
} kn_peers;

/* Neighbourhood synchronisation between the layers of the fused row-sharded forward: flags_host[i] = device address on rank
 * i of an int32[8] flag array in NVLink-mapped memory.  epoch_counter: device int32 of the calling rank, advanced by one per
 * call (all ranks make the same sequence of calls; keeping the epoch on the device makes the launch replayable in a CUDA
 * graph).  The calling rank stores the new epoch into flags[q][my_rank] of every rank q in signal_mask (after a system-scope
 * fence: its earlier peer stores are visible first) and then waits until flags[my_rank][p] >= epoch for every p in wait_mask.  Replaces a barrier over all ranks: a conv layer sharded by
 * pixels only depends on its two neighbours.  timeout_flag (device int, nullable) is set if a peer never arrives. */
int kn_peer_sync(const uint64_t *flags_host, int32_t world, int32_t my_rank, uint32_t signal_mask, uint32_t wait_mask, int32_t *epoch_counter,
                 int32_t *timeout_flag, void *stream);

/* ---- SpMM:  Y[n_rows][n_vecs] = W . X  (+ optional ReLU) --------------------------------
 * Replaces SparseMatrix.torchdot (keynet/sparse.py:488-492 -> scipy csr_matvecs), called from
 * KeyedLayer.forward / .decrypt (keynet/layer.py:92,99) and KeyedSensor.encrypt (system.py:254).
 * fp32 accumulate; each output element sums its row's entries in stored order. */
int kn_spmm_csr_f32(const int64_t *indptr, const int32_t *indices, const float *data,
                    int64_t n_rows, int64_t n_cols,
                    const float *X, int64_t ldx, float *Y, int64_t ldy, int64_t n_vecs,
                    uint32_t flags, const kn_peers *peers, void *stream);

/* Same product for a subset of rows: output row i is written to Y[out_rows[i]] (out_rows NULL = identity).
 * Used for the rows of a layer matrix that are not covered by pattern groups (below). */
int kn_spmm_csr_rows_f32(const int64_t *indptr, const int32_t *indices, const float *data,
                         int64_t n_rows, int64_t n_cols, const int32_t *out_rows,
                         const float *X, int64_t ldx, float *Y, int64_t ldy, int64_t n_vecs,
                         uint32_t flags, const kn_peers *peers, void *stream);

/* ---- general key compile: C = A . B on CSR (csrc/spgemm.cu) ------------------------------------------------
 * Replaces the two scipy csr_matmat calls of `A.dot(W).dot(Ainv)` (keynet/layer.py:35,59,70) for keys with several
 * entries per row: Givens-rotation orthogonal and doubly stochastic blocks (keynet/sparse.py:288-353), their
 * block-diagonal repeats (keynet/system.py:398-410).  Three steps, the caller scans in between (kn_exclusive_scan_i64):
 *   kn_spgemm_bound  ub[r] = number of products a_rj * b_jc of row r                       -> scan -> tmp_ptr
 *   kn_spgemm_rows   products of row r expanded into tmp[tmp_ptr[r] ..), sorted by column, duplicates added in fp32,
 *                    exact zeros dropped (scipy never stores one), compacted; row_nnz[r] = kept     -> scan -> out_indptr
 *   kn_csr_compact   tmp slices -> out CSR (canonical: ascending columns) */
int kn_spgemm_bound(const int64_t *a_indptr, const int32_t *a_indices, int64_t n_rows, const int64_t *b_indptr, int64_t *ub, void *stream);
int kn_spgemm_rows(const int64_t *a_indptr, const int32_t *a_indices, const float *a_data, int64_t n_rows,
                   const int64_t *b_indptr, const int32_t *b_indices, const float *b_data,
                   const int64_t *tmp_ptr, int32_t *tmp_indices, float *tmp_data, int64_t *row_nnz, void *stream);
int kn_csr_compact(const int64_t *tmp_ptr, const int32_t *tmp_indices, const float *tmp_data, int64_t n_rows,
                   const int64_t *out_indptr, int32_t *out_indices, float *out_data, void *stream);

/* ---- pattern-grouped execution format (csrc/pgroup.cu) ------------------------------------------
 * B200 form of the reference's unique-tile storage (TiledMatrix / Conv2dTiledMatrix,
 * keynet/sparse.py:517-835): rows with an identical column set form a group whose values are a dense
 * G x K block; the product becomes one small GEMM per group with a gathered B operand.
 *   kn_csr_row_pattern_hash  64-bit hash of every row's column set (grouping key)
 *   kn_pg_verify             mismatch[i]=1 iff rows[i] and leaders[i] differ in their column lists
 *   kn_pg_pack               rows[n_groups][G] -> cols[n_groups][K_pad], vals[n_groups][G][K_pad] (zero padded)
 *   kn_spmm_pg_f32           Y[rows[g][:], :] = vals[g] . X[cols[g][:], :]  (+ReLU); fp32 FMA, K_pad % 32 == 0,
 *                            n_vecs/ldx/ldy multiples of 4; group_k[g] (nullable) = number of leading columns of group g
 *                            that are real (the rest of K_pad is zero padding and is skipped); block_of[g] (nullable) =
 *                            index of the group's value block in `vals` when identical blocks are stored once (unique tiles) */
int kn_csr_row_pattern_hash(const int64_t *indptr, const int32_t *indices, int64_t n_rows, uint64_t *hash, void *stream);
int kn_pg_verify(const int64_t *indptr, const int32_t *indices, const int64_t *rows, const int64_t *leaders, int64_t n,
                 int32_t *mismatch, void *stream);
int kn_pg_pack(const int64_t *indptr, const int32_t *indices, const float *data, const int64_t *rows,
               int64_t n_groups, int32_t G, int32_t K_pad, int32_t *cols, float *vals, void *stream);
int kn_spmm_pg_f32(const int32_t *rows, const int32_t *cols, const float *vals, const int32_t *group_k, const int32_t *block_of, int64_t n_groups, int32_t G, int32_t K_pad,
                   const float *X, int64_t ldx, float *Y, int64_t ldy, int64_t n_vecs, uint32_t flags, const kn_peers *peers, void *stream);

/* Split-K epilogue for a layer that is ONE huge group (dense fully connected layers): the K range is cut into S slices
 * that run as S groups of kn_spmm_pg_tc_f32 / kn_spmm_pg_f32 writing partial rows part[s*G + i][n_vecs]; this adds them:
 * Y[rows[i]][:] = relu?(sum_s part[s*G + i][:]) (and performs the peer stores of the row-sharded path). */
int kn_splitk_reduce_f32(const float *part, int32_t S, int32_t G, const int32_t *rows, float *Y, int64_t ldy, int64_t n_vecs, uint32_t flags, const kn_peers *peers, void *stream);

/* Narrow batches (csrc/pgroup.cu): same contract as kn_spmm_pg_f32 for 1 <= n_vecs <= 32, with any ldx / ldy >= n_vecs and
 * any 4-byte alignment of X and Y (no padding of the batch to 32 columns).
 *   run_groups[n_groups], run_start[n_runs+1]  run table: the class's groups listed run by run; a run is at most
 *                            128 / NB groups (NB = n_vecs rounded up to a power of two) that share one value block
 *                            (block_of) and one group_k.  Required whenever n_groups > 0.
 *   row_form = 0             shared-block form (pg_simt over runs): the tile's 128 columns are (group, batch column) pairs
 *                            of one run, the run's value rows are staged once and serve all its groups; per output element
 *                            the same fp32 FMA chain as kn_spmm_pg_f32's pg_simt kernel (bit-identical results).
 *   row_form = 1             row form (n_vecs <= 8; CSR kernel spmm_lanes_nnz over the class's rows): one warp per row,
 *                            lanes over the group's first group_k columns, fixed shuffle reduction (deterministic).
 * peers must be NULL: the fused row-sharded path pads its batch to the grouped kernels itself. */
int kn_spmm_pg_narrow_f32(const int32_t *rows, const int32_t *cols, const float *vals, const int32_t *group_k, const int32_t *block_of, int64_t n_groups, int32_t G, int32_t K_pad,
                          const int32_t *run_groups, const int32_t *run_start, int64_t n_runs, int32_t row_form,
                          const float *X, int64_t ldx, float *Y, int64_t ldy, int64_t n_vecs, uint32_t flags, const kn_peers *peers, void *stream);

/* Clustered variant for short reductions (csrc/pgcluster.cu; G <= 256, walked 16 rows at a time above 16): the groups of a tile of neighbouring output pixels
 * form a cluster with ONE union column list that is staged in shared memory once per (cluster, 128 batch columns), so a
 * 3x3 convolution reads every X row from L2 about once instead of 9 times.
 *   cl_gptr[n_clusters+1]   group range of every cluster (groups are stored cluster by cluster)
 *   cl_uptr[n_clusters+1]   range of every cluster in ucols; at most KN_CG_MAX_UNION columns per cluster
 *   ucols                   union column lists
 *   lidx[n_groups][K_pad]   BYTE offset (local column index x 512) of every column of the group in the staged tile
 *   valsT[n_blocks][K_pad][GM]  value blocks k-major, GM = G rounded up to even (G <= 16) or to a multiple of 16 (zero padded)
 * rows / group_k / block_of as in kn_spmm_pg_f32.  u_max / g_max = largest union / group count of a cluster: the CTA stages
 * u_max x 512 B of X plus g_max x K_pad x 4 B of lidx, together at most KN_CG_MAX_UNION x 512 B. */
#define KN_CG_MAX_UNION 224
int kn_spmm_cg_f32(const int32_t *cl_gptr, const int32_t *cl_uptr, const int32_t *ucols, const int32_t *rows, const int32_t *lidx, const float *valsT,
                   const int32_t *group_k, const int32_t *block_of, int64_t n_clusters, int32_t G, int32_t K_pad, int32_t u_max, int32_t g_max,
                   const float *X, int64_t ldx, float *Y, int64_t ldy, int64_t n_vecs, uint32_t flags, const kn_peers *peers, void *stream);

/* Tensor-core variant (csrc/pgroup_tc.cu): tcgen05.mma with an error-compensated split, per 8 k
 *   x_hi.w_hi (kind::tf32)  +  [x_hi | x_lo] . [w_lo ; w_hi] (kind::f16 with bf16 operands, K = 16),
 * both into one fp32 accumulator in TMEM (hi = v rounded to nearest TF32, lo = v - hi; error per product < 2^-16.9 |x||w|),
 * weight blocks by TMA, gathered activations written into the UMMA layout by producer warps.
 *   kn_pg_tc_split: vals[n] (n % 8 == 0, 16-byte aligned arrays) -> vals_hi[n]: hi as fp32 bit patterns, and vals_corr[n]:
 *   per 8 consecutive values v[8j .. 8j+7], 8 words = 4 bf16 pairs of lo, then 4 bf16 pairs of hi (word i of each four
 *   holds v[8j+2i] in its lower 16 bits and v[8j+2i+1] in its upper 16 bits).  Rows of length K_pad % 16 == 0 keep
 *   every group of 8 inside a row.
 *   kn_pg_tc_tensormaps: writes four CUtensorMap (4 x 128 bytes, HOST memory) describing the hi / corr planes
 *   [n_rows_total][K_pad] of 4-byte words (full boxes, and half boxes for the 2-CTA multicast launch).
 *   kn_spmm_pg_tc_f32: same contract as kn_spmm_pg_f32 (results agree with fp32 FMA to ~1e-6 relative). */
#define KN_TENSORMAP_BYTES 128
int kn_pg_tc_split(const float *vals, int64_t n, float *vals_hi, float *vals_corr, void *stream);
int kn_pg_tc_tensormaps(const float *vals_hi, const float *vals_corr, int64_t n_rows_total, int32_t G, int32_t K_pad, void *maps_out_host);
int kn_spmm_pg_tc_f32(const void *maps_host, const int32_t *rows, const int32_t *cols, const int32_t *group_k, const int32_t *block_of, int64_t n_groups, int32_t G, int32_t K_pad,
                      const float *X, int64_t ldx, float *Y, int64_t ldy, int64_t n_vecs, uint32_t flags, const kn_peers *peers, void *stream);

/* debug aid: record clock64 phase stamps (entry, prologue, first stage, last MMA issue, accumulators ready, epilogue
 * stored, teardown) of CTA `cta` of the next kn_spmm_pg_tc_f32 launches (-1 = off); out_host (nullable) receives 8 values. */
int kn_debug_tc_timing(int32_t cta, int64_t *out_host);

/* ---- prefix sum: out[0]=0, out[i+1]=out[i]+in[i]; out has n+1 entries (in may alias out+1) */
int kn_exclusive_scan_i64(const int64_t *in, int64_t *out, int64_t n, void *stream);

/* ---- Toeplitz construction ---------------------------------------------------------------
 * Replaces sparse_toeplitz_conv2d / sparse_toeplitz_avgpool2d (keynet/sparse.py:122-212): the
 * homogeneous CSR matrix of a 'same'-padded cross-correlation,
 *   row (m,ku,kv) = m*Uo*Vo + ku*Vo + kv,  col (c,y,x) = c*U*V + y*V + x,  bias in column C*U*V,
 *   last row = e_last.  Rows are emitted with ascending columns and explicit zeros kept.
 * `weight`/`bias` must already carry the reference's offset rounding fl32(fl32(w+off)-off)
 * (sparse.py:184-187,193-196) -- it is applied by the host wrapper.
 * depthwise != 0: weight is [C][P][Q] and only channel c==m is emitted (avg-pool; the
 * reference's C*C zero blocks are dropped by the key compile that always follows, layer.py:59).
 * row_ids (nullable): emit only these source rows, in this order -- this is where the output
 * permutation key and the row shard are applied; NULL = rows 0..n_rows-1. */
typedef struct {
    int32_t C, U, V;        /* input  channels, height, width */
    int32_t M;              /* output channels */
    int32_t P, Q;           /* kernel height, width (odd) */
    int32_t stride;
    int32_t depthwise;      /* 0: full conv, 1: channel-diagonal (avgpool) */
    int32_t has_bias;       /* 1: homogeneous form with bias column and last row */
} kn_conv2d_desc;

int kn_toeplitz_conv2d_count(const kn_conv2d_desc *desc_host, const int64_t *row_ids, int64_t n_rows,
                             int64_t *row_nnz, void *stream);
int kn_toeplitz_conv2d_fill(const kn_conv2d_desc *desc_host, const float *weight, const float *bias,
                            const int64_t *row_ids, int64_t n_rows,
                            const int64_t *indptr, int32_t *indices, float *data, void *stream);

/* Homogeneous matrix of nn.Linear, [[W, b],[0, 1]] with exact zeros dropped
 * (keynet/torch.py:80-89 + keynet/layer.py:69).  weight is [n_out][n_in] row-major. */
int kn_linear_count(const float *weight, const float *bias, int64_t n_out, int64_t n_in,
                    const int64_t *row_ids, int64_t n_rows, int64_t *row_nnz, void *stream);
int kn_linear_fill(const float *weight, const float *bias, int64_t n_out, int64_t n_in,
                   const int64_t *row_ids, int64_t n_rows,
                   const int64_t *indptr, int32_t *indices, float *data, void *stream);

/* ---- key compile for monomial keys (permutation and/or diagonal gain) ----------------------
 * Replaces `A.dot(W).dot(Ainv)` (keynet/layer.py:35,59,70 -> two scipy csr_matmat) when A and
 * Ainv have one entry per row.  The row gather by A is done upstream (row_ids of the builders /
 * kn_csr_gather_rows); this call applies, per stored entry (r, c, v):
 *     c' = col_map[c]                         (Ainv[c, c'] is the entry of row c)
 *     v' = fl32( fl32(row_scale[r]*v) * col_scale[c] )     (left product first, as the reference)
 *     dropped if v' == 0                      (scipy SpGEMM drops exact zeros)
 * and writes rows with ascending c' (canonical form).  col_map / row_scale / col_scale may be
 * NULL (identity / 1.0).  No FMA contraction, no flush-to-zero: values are bit-exact with scipy.
 * row_bias / col_bias (nullable): bias columns of affine photometric keys [[D, b],[0, 1]] (keynet/sparse.py:99-119) on the
 * left / right: the row's last-column entry becomes fl(a_r*w_last) + row_bias[r] + sum_c fl(fl(a_r*w_c) * col_bias[c]) (a row
 * reduction: equal to the reference to fp32 rounding; all other entries and all indices stay bit-exact).
 * keep_zeros != 0 keeps exact zeros (the structural matrix the pattern groups are built from, so that a tiny weight
 * rounded to 0 by the reference's offset trick does not split a pixel's rows into different column patterns). */
int kn_keycompile_count(const int64_t *indptr, const int32_t *indices, const float *data, int64_t n_rows,
                        const float *row_scale, const float *col_scale, const float *row_bias, const float *col_bias, int64_t n_cols_in,
                        int32_t keep_zeros, int64_t *row_nnz, void *stream);
int kn_keycompile_fill(const int64_t *indptr, const int32_t *indices, const float *data, int64_t n_rows, int64_t n_cols,
                       const int32_t *col_map, const float *row_scale, const float *col_scale,
                       const float *row_bias, const float *col_bias, int64_t n_cols_in, int32_t keep_zeros,
                       const int64_t *out_indptr, int32_t *out_indices, float *out_data, void *stream);

/* ---- fused key compile of a conv / linear layer (csrc/keyedconv.cu) ------------------------------------------------
 * W_hat = A . toeplitz(conv2d) . Ainv for monomial keys WITHOUT materialising the un-keyed Toeplitz matrix: replaces
 * keynet/sparse.py:163-203 (sparse_toeplitz_conv2d) + the two SpGEMMs of keynet/layer.py:35 (and, as a 1x1 convolution
 * on a 1x1 image, keynet/torch.py:80-89 + keynet/layer.py:69-70 for nn.Linear) in one pass with one column sort per
 * output pixel -- all M rows of a pixel share their column set.
 *   pix[n_groups]        output pixels to compile (ku*Vo + kv), NULL = all Uo*Vo pixels in raster order
 *   row_of_src[R_src+1]  compiled row of every Toeplitz row s = m*Uo*Vo + pixel (last entry: the homogeneous row); < 0 =
 *                        not held by this shard; NULL = identity (no output key, not sharded)
 *   col_map[K_src+1]     new column of every source column (input key / gathered layout); NULL = identity
 *   row_scale (per compiled row), col_scale (per source column): gains of A and Ainv; NULL = 1
 * Values: fl32(fl32(row_scale*w)*col_scale), exact zeros dropped unless keep_zeros; columns ascending.  Weights must be
 * the offset-rounded ones (keynet/sparse.py:184-187).  Two phase: count -> kn_exclusive_scan_i64 -> fill.
 * Returns KN_ERR_UNSUPPORTED when C*P*Q+1 exceeds the shared-memory sort (8192): use the two-kernel path then. */
int kn_keyed_conv2d_count(const kn_conv2d_desc *desc, const float *weight, const float *bias, const int32_t *pix, int64_t n_groups,
                          const int32_t *row_of_src, const float *row_scale, const float *col_scale, int32_t keep_zeros,
                          int64_t *row_nnz, void *stream);
int kn_keyed_conv2d_fill(const kn_conv2d_desc *desc, const float *weight, const float *bias, const int32_t *pix, int64_t n_groups,
                         const int32_t *row_of_src, const int32_t *col_map, const float *row_scale, const float *col_scale, int32_t keep_zeros,
                         const int64_t *out_indptr, int32_t *out_indices, float *out_data, void *stream);
/* The pattern-group execution format (below) of the same keyed layer straight from the geometry, no CSR involved:
 *   kn_conv2d_groups_index   rows[g][M], cols[g][K_pad] (Toeplitz tap order, padding repeats the first column), group_k[g]
 *   kn_conv2d_groups_values  vals[b][M][K_pad] for the pixels block_pix[b]: one block per pixel with gain keys, one block per
 *                            border class (which taps are in bounds) with permutation-only keys -- the unique tiles of
 *                            keynet/sparse.py:553-568,690-779 by construction. */
int kn_conv2d_groups_index(const kn_conv2d_desc *desc, const int32_t *pix, int64_t n_groups, const int32_t *row_of_src, const int32_t *col_map,
                           int32_t K_pad, int32_t *rows, int32_t *cols, int32_t *group_k, void *stream);
int kn_conv2d_groups_values(const kn_conv2d_desc *desc, const float *weight, const float *bias, const int32_t *block_pix, int64_t n_blocks,
                            const int32_t *row_of_src, const float *row_scale, const float *col_scale, int32_t K_pad, float *vals, void *stream);

/* ---- spatially tiled tensor-core product for keyed conv layers with G <= 128 output channels (csrc/pgtile_tc.cu) -----
 * Same product as kn_spmm_pg_tc_f32 (SparseMatrix.torchdot, keynet/sparse.py:488-492, of a Toeplitz conv layer of
 * keynet/sparse.py:163-203 under permutation-only keys), organised by TILES of th x tw neighbouring output pixels: the
 * union of a tile's input positions is gathered once per 16-channel chunk and the P*Q weight slabs of the chunk are
 * loaded once and shared by all pixels of the tile -- those layers are bound by L2 -> SM traffic, not by the tensor pipe.
 *   kn_conv2d_tiles_index  tile tables: tile_cols[tile][(th-1)*stride+P][(tw-1)*stride+Q][C] activation row of every
 *                          (input position, channel) under the input key (col_map), -1 outside the image;
 *                          tile_rows[tile][th*tw][M] output row of every (pixel, channel).  tile_origin[tile] = top-left
 *                          output pixel (ku*Vo + kv) of the tile.
 *   kn_spmm_tile_tc_f32    maps_host: TMA descriptors (kn_pg_tc_tensormaps) of the TAP-major weight matrix Wt[G][K_pad],
 *                          k = tap*C + c, bias at k = P*Q*C, zero padded to a multiple of 16; bias_col = activation row
 *                          of the homogeneous coordinate.  C % 16 == 0, th*tw <= 6, union positions <= 32. */
int kn_conv2d_tiles_index(const kn_conv2d_desc *desc, const int32_t *tile_origin, int64_t n_tiles, int32_t th, int32_t tw,
                          const int32_t *row_of_src, const int32_t *col_map, int32_t *tile_cols, int32_t *tile_rows, void *stream);
int kn_spmm_tile_tc_f32(const void *maps_host, const int32_t *tile_cols, const int32_t *tile_rows, int32_t bias_col, int64_t n_tiles,
                        int32_t C, int32_t G, int32_t th, int32_t tw, int32_t stride, int32_t P, int32_t Q,
                        const float *X, int64_t ldx, float *Y, int64_t ldy, int64_t n_vecs, uint32_t flags, const kn_peers *peers, void *stream);

/* ---- fused keyed conv (+ReLU) -> keyed average pooling for small layers (csrc/convpool.cu) ---------------------------
 * Y = W_pool . relu(W_conv . X) for two consecutive keyed layers (keynet/layer.py:32-35 conv, :48-59 avgpool, ReLU of
 * keynet/system.py:92) under permutation-only keys, with the intermediate (all conv outputs of an image) in shared memory
 * instead of HBM.  weight / bias: the conv's offset-rounded coefficients; pool_w: the pooling coefficient as the reference
 * stores it (offset-rounded 1/k^2, keynet/sparse.py:206-212; windows centred, zero padded, divisor k*k);
 * xrow[C*U*V + 1]: activation row of every conv input (c, y, x) under the conv's input key, last = homogeneous row;
 * yrow[M*Up*Vp + 1]: output row of every pooled (m, py, px) under the pool's output key, last = homogeneous row. */
int kn_convpool_f32(const kn_conv2d_desc *desc, const float *weight, const float *bias, const int32_t *xrow,
                    int32_t pool_k, int32_t pool_stride, float pool_w, const int32_t *yrow,
                    const float *X, int64_t ldx, float *Y, int64_t ldy, int64_t n_vecs, void *stream);

/* Gather rows of a CSR matrix: out row i = in row row_ids[i] (SparseMatrix key A applied on the left
 * for explicit matrices, e.g. sensor keys / ReLU keys, keynet/layer.py:46). */
int kn_csr_gather_rows_count(const int64_t *indptr, const int64_t *row_ids, int64_t n_rows, int64_t *row_nnz, void *stream);
int kn_csr_gather_rows_fill(const int64_t *indptr, const int32_t *indices, const float *data,
                            const int64_t *row_ids, int64_t n_rows,
                            const int64_t *out_indptr, int32_t *out_indices, float *out_data, void *stream);

/* ---- activation layout helpers -------------------------------------------------------------
 * affine_to_linear (keynet/torch.py:65-68) fused with the transpose the reference does at
 * layer.py:92: images [n_vecs][dim] row-major -> X [dim+1][ldx] with a trailing row of ones. */
int kn_affine_to_linear_t(const float *images, int64_t n_vecs, int64_t dim, float *X, int64_t ldx, void *stream);
/* KeyedSensor.encrypt (keynet/system.py:250-255) in one pass for a monomial image key A (one entry per row: permutation x
 * gain, optionally a bias column): Y = A . affine_to_linear(images)^T written directly, Y[row_of_col[d]][n] =
 * scale_of_col[d] * images[n][d] (+ row_bias[row], NULL = none); d = dim is the homogeneous 1.  Saves the pass that
 * kn_affine_to_linear_t + kn_spmm_csr_f32 spend writing and re-reading the un-keyed X. */
int kn_encrypt_monomial_t(const float *images, int64_t n_vecs, int64_t dim, const int32_t *row_of_col, const float *scale_of_col,
                          const float *row_bias, float *Y, int64_t ldy, void *stream);
/* inverse: X [dim+1][ldx] -> out [n_vecs][dim]; *bad_count_dev (int32, device) receives the number of
 * vectors whose homogeneous coordinate is not within atol of 1 (linear_to_affine raises on it, torch.py:74). */
int kn_linear_to_affine_t(const float *X, int64_t ldx, int64_t n_vecs, int64_t dim, float *out,
                          float atol, int32_t *bad_count_dev, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* KEYNET_B200_H */
