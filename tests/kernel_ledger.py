"""Every `__global__` entry of libkeynet_b200.so, as plain data shared by tests/test_kernel_ledger.py (the set compiled into
the library must equal this ledger) and tests/test_gpu_kernel_matrix.py (every SpMM instantiation must run and match an
exact reference).

Names are in one normalised spelling: no namespace, no return type, no parameter list, template arguments as the
compiler's values (`true` / `false` for bools, plain integers) with no spaces, e.g. `pg_tile_tc_kernel<false,true,1,2,128>`.
`normalise()` maps both spellings this project meets onto it: the profiler's
(`void (anonymous namespace)::pg_tc_kernel<2, true, 2, false>(CUtensorMap_st, ...)`) and cu++filt's
(`void <unnamed>::pg_tc_kernel<(int)2, (bool)1, (int)2, (bool)0>(CUtensorMap_st, ...)`).
"""
import re


# The instantiations that compute Y = W . X (the keyed forward), one per line.
SPMM_KERNELS = [
    # spmm.cu (CSR): lanes_nnz<NB, RELU> for N <= 8, rowwarp<V, RELU> and rowwarp_wide<WS, RELU> above
    'spmm_lanes_nnz_kernel<1,false>',
    'spmm_lanes_nnz_kernel<1,true>',
    'spmm_lanes_nnz_kernel<2,false>',
    'spmm_lanes_nnz_kernel<2,true>',
    'spmm_lanes_nnz_kernel<4,false>',
    'spmm_lanes_nnz_kernel<4,true>',
    'spmm_lanes_nnz_kernel<8,false>',
    'spmm_lanes_nnz_kernel<8,true>',
    'spmm_rowwarp_kernel<1,false>',
    'spmm_rowwarp_kernel<1,true>',
    'spmm_rowwarp_kernel<2,false>',
    'spmm_rowwarp_kernel<2,true>',
    'spmm_rowwarp_kernel<4,false>',
    'spmm_rowwarp_kernel<4,true>',
    'spmm_rowwarp_wide_kernel<2,false>',
    'spmm_rowwarp_wide_kernel<2,true>',
    'spmm_rowwarp_wide_kernel<4,false>',
    'spmm_rowwarp_wide_kernel<4,true>',
    # pgroup.cu (fp32 FMA pattern groups): pg_small<GM, RELU>, pg_simt<RW, RELU>, and the split-K epilogue
    'pg_small_kernel<8,false>',
    'pg_small_kernel<8,true>',
    'pg_small_kernel<16,false>',
    'pg_small_kernel<16,true>',
    'pg_simt_kernel<1,false>',
    'pg_simt_kernel<1,true>',
    'pg_simt_kernel<2,false>',
    'pg_simt_kernel<2,true>',
    'pg_simt_kernel<4,false>',
    'pg_simt_kernel<4,true>',
    'pg_simt_kernel<8,false>',
    'pg_simt_kernel<8,true>',
    'pg_simt_kernel<12,false>',
    'pg_simt_kernel<12,true>',
    'pg_simt_kernel<16,false>',
    'pg_simt_kernel<16,true>',
    'splitk_reduce_kernel<false>',
    'splitk_reduce_kernel<true>',
    # pgcluster.cu (clustered small groups): <GM, RELU>
    'pg_cluster_kernel<2,false>',
    'pg_cluster_kernel<2,true>',
    'pg_cluster_kernel<4,false>',
    'pg_cluster_kernel<4,true>',
    'pg_cluster_kernel<6,false>',
    'pg_cluster_kernel<6,true>',
    'pg_cluster_kernel<8,false>',
    'pg_cluster_kernel<8,true>',
    'pg_cluster_kernel<10,false>',
    'pg_cluster_kernel<10,true>',
    'pg_cluster_kernel<12,false>',
    'pg_cluster_kernel<12,true>',
    'pg_cluster_kernel<14,false>',
    'pg_cluster_kernel<14,true>',
    'pg_cluster_kernel<16,false>',
    'pg_cluster_kernel<16,true>',
    # pgroup_tc.cu: <NB (batch tiles per CTA), RELU, CS (cluster size), PEERS>
    'pg_tc_kernel<1,false,1,false>',
    'pg_tc_kernel<1,false,1,true>',
    'pg_tc_kernel<1,false,2,false>',
    'pg_tc_kernel<1,false,2,true>',
    'pg_tc_kernel<1,true,1,false>',
    'pg_tc_kernel<1,true,1,true>',
    'pg_tc_kernel<1,true,2,false>',
    'pg_tc_kernel<1,true,2,true>',
    'pg_tc_kernel<2,false,1,false>',
    'pg_tc_kernel<2,false,1,true>',
    'pg_tc_kernel<2,false,2,false>',
    'pg_tc_kernel<2,false,2,true>',
    'pg_tc_kernel<2,true,1,false>',
    'pg_tc_kernel<2,true,1,true>',
    'pg_tc_kernel<2,true,2,false>',
    'pg_tc_kernel<2,true,2,true>',
    # pgtile_tc.cu: <RELU, PEERS, TH, TW, GP>; <0,0,0> is the generic issuer, the others the interior-tile issuers
    'pg_tile_tc_kernel<false,false,0,0,0>',
    'pg_tile_tc_kernel<false,false,1,2,128>',
    'pg_tile_tc_kernel<false,false,2,2,64>',
    'pg_tile_tc_kernel<false,false,2,2,96>',
    'pg_tile_tc_kernel<false,true,0,0,0>',
    'pg_tile_tc_kernel<false,true,1,2,128>',
    'pg_tile_tc_kernel<false,true,2,2,64>',
    'pg_tile_tc_kernel<false,true,2,2,96>',
    'pg_tile_tc_kernel<true,false,0,0,0>',
    'pg_tile_tc_kernel<true,false,1,2,128>',
    'pg_tile_tc_kernel<true,false,2,2,64>',
    'pg_tile_tc_kernel<true,false,2,2,96>',
    'pg_tile_tc_kernel<true,true,0,0,0>',
    'pg_tile_tc_kernel<true,true,1,2,128>',
    'pg_tile_tc_kernel<true,true,2,2,64>',
    'pg_tile_tc_kernel<true,true,2,2,96>',
]

# Every other entry, with the test module that exercises it.
OTHER_KERNELS = {
    'affine_to_linear_t_kernel': 'test_gpu_parity.py',
    'encrypt_monomial_t_kernel': 'test_gpu_engine.py',
    'linear_to_affine_t_kernel': 'test_gpu_engine.py',
    'conv_class_lists_kernel': 'test_gpu_keyedconv.py',
    'conv_class_zeros_kernel': 'test_gpu_keyedconv.py',
    'conv_groups_index_kernel': 'test_gpu_keyedconv.py',
    'conv_groups_values_kernel': 'test_gpu_keyedconv.py',
    'keyed_conv_count_class_kernel': 'test_gpu_keyedconv.py',
    'keyed_conv_count_kernel': 'test_gpu_keyedconv.py',
    'keyed_conv_fill_kernel<true>': 'test_gpu_keyedconv.py',
    'keyed_conv_lists_kernel': 'test_gpu_keyedconv.py',
    'keyed_conv_rows_kernel': 'test_gpu_keyedconv.py',
    'toeplitz_count_kernel': 'test_gpu_keyedconv.py',
    'toeplitz_fill_kernel': 'test_gpu_keyedconv.py',
    'linear_count_kernel': 'test_gpu_keyedconv.py',
    'linear_fill_kernel': 'test_gpu_keyedconv.py',
    'keycompile_count_kernel': 'test_gpu_keyedconv.py',
    'keycompile_fill_kernel': 'test_gpu_keyedconv.py',
    'keycompile_fill_short_kernel': 'test_gpu_keyedconv.py',
    'keycompile_count_bias_kernel': 'test_gpu_parity.py',
    'gather_rows_count_kernel': 'test_gpu_keyedconv.py',
    'gather_rows_fill_kernel': 'test_gpu_keyedconv.py',
    'conv_tiles_index_kernel': 'test_gpu_tiles.py',
    'csr_compact_kernel': 'test_gpu_general_keys.py',
    'spgemm_bound_kernel': 'test_gpu_general_keys.py',
    'spgemm_rows_kernel': 'test_gpu_general_keys.py',
    'row_pattern_hash_kernel': 'test_gpu_parity.py',
    'pg_verify_kernel': 'test_gpu_parity.py',
    'pg_pack_kernel': 'test_gpu_parity.py',
    'scan_tile_sums_kernel': 'test_gpu_parity.py',
    'tile_scan_kernel': 'test_gpu_parity.py',
    'tile_sum_kernel': 'test_gpu_parity.py',
    'split_tf32_kernel': 'test_gpu_mixed_split.py',
    'peer_sync_kernel': 'test_gpu_dist.py',
    'convpool_kernel<4,4>': 'test_gpu_fusion.py',
    'convpool_kernel<4,6>': 'test_gpu_fusion.py',
    'convpool_kernel<8,4>': 'test_gpu_fusion.py',
    'convpool_kernel<8,6>': 'test_gpu_fusion.py',
}

_NS = re.compile(r'\(anonymous namespace\)::|<unnamed>::|_GLOBAL__N_\w*::')


def normalise(name):
    """One kernel name (demangled by cu++filt or as torch.profiler reports it) in the ledger's spelling."""
    s = _NS.sub('', name.strip())
    if s.startswith('void '):
        s = s[5:]
    # cut the parameter list: the first '(' outside the template argument list
    depth = 0
    for (i, ch) in enumerate(s):
        if ch == '<':
            depth += 1
        elif ch == '>':
            depth -= 1
        elif ch == '(' and depth == 0:
            s = s[:i]
            break
    s = s.replace('(bool)1', 'true').replace('(bool)0', 'false')
    s = re.sub(r'\((?:int|unsigned int|long|unsigned)\)', '', s)
    return s.replace(' ', '')


def family(name):
    """Kernel name without template arguments (`pg_tc_kernel`), of a normalised name."""
    return name.split('<', 1)[0]


SPMM_FAMILIES = sorted(set(family(k) for k in SPMM_KERNELS))
