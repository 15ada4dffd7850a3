"""ctypes binding of libkeynet_b200.so (C ABI declared in include/keynet_b200.h).

There is NO fallback: if the shared library is missing or a call fails, this module raises.
Build the library with `python -c "import __graft_entry__ as g; g.build()"` (nvcc, sm_100a).
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('KEYNET_B200_LIB', os.path.join(_HERE, 'lib', 'libkeynet_b200.so'))

KN_SPMM_RELU = 1
KN_ERR_UNSUPPORTED = -3

# every symbol include/keynet_b200.h declares (tests/test_abi.py checks the two lists agree)
SYMBOLS = [
    'kn_abi_version', 'kn_last_error', 'kn_device_info', 'kn_peer_sync',
    'kn_spmm_csr_f32', 'kn_spmm_csr_rows_f32', 'kn_exclusive_scan_i64',
    'kn_csr_row_pattern_hash', 'kn_pg_verify', 'kn_pg_pack', 'kn_spmm_pg_f32', 'kn_spmm_cg_f32',
    'kn_pg_tc_split', 'kn_pg_tc_tensormaps', 'kn_spmm_pg_tc_f32', 'kn_debug_tc_timing',
    'kn_toeplitz_conv2d_count', 'kn_toeplitz_conv2d_fill', 'kn_linear_count', 'kn_linear_fill',
    'kn_keycompile_count', 'kn_keycompile_fill', 'kn_csr_gather_rows_count', 'kn_csr_gather_rows_fill',
    'kn_affine_to_linear_t', 'kn_linear_to_affine_t',
    'kn_conv2d_tiles_index', 'kn_spmm_tile_tc_f32', 'kn_convpool_f32',
    'kn_keyed_conv2d_count', 'kn_keyed_conv2d_fill', 'kn_conv2d_groups_index', 'kn_conv2d_groups_values',
    'kn_spgemm_bound', 'kn_spgemm_rows', 'kn_csr_compact', 'kn_encrypt_monomial_t', 'kn_splitk_reduce_f32',
    'kn_spmm_pg_narrow_f32',
]


class kn_conv2d_desc(ctypes.Structure):
    _fields_ = [('C', ctypes.c_int32), ('U', ctypes.c_int32), ('V', ctypes.c_int32), ('M', ctypes.c_int32),
                ('P', ctypes.c_int32), ('Q', ctypes.c_int32), ('stride', ctypes.c_int32),
                ('depthwise', ctypes.c_int32), ('has_bias', ctypes.c_int32)]


class kn_peers(ctypes.Structure):
    """include/keynet_b200.h: destinations of a fused SpMM + all-gather."""
    _fields_ = [('n', ctypes.c_int32), ('reserved', ctypes.c_int32), ('y', ctypes.c_uint64 * 8), ('row_mask', ctypes.c_void_p)]


class Peers(object):
    """Output destinations of one kn_spmm_* call: ptrs[i] = device address on rank i of the slot the call's Y argument
    denotes (NVLink peer mappings); row_mask: uint8 CUDA tensor, one byte per output row, bit i = rank i reads the row
    (None = every row to every rank).  Passed explicitly to every call; nothing is kept in the library."""

    def __init__(self, ptrs, row_mask=None):
        assert 0 < len(ptrs) <= 8
        if row_mask is not None:
            assert row_mask.is_cuda and row_mask.dtype.itemsize == 1 and row_mask.is_contiguous()
        self.row_mask = row_mask                          # keeps the tensor alive
        self.c = kn_peers()
        self.c.n = len(ptrs)
        for (i, p) in enumerate(ptrs):
            self.c.y[i] = int(p)
        self.c.row_mask = None if row_mask is None else row_mask.data_ptr()


def peers_arg(peers):
    return None if peers is None else ctypes.byref(peers.c)


class NativeError(RuntimeError):
    pass


_lib = None


def lib():
    """Load (once) and return the shared library; raises NativeError if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NativeError('libkeynet_b200.so not found at %s -- build it with __graft_entry__.build(); '
                          'keynet_b200 has no CPU fallback' % LIB_PATH)
    L = ctypes.CDLL(LIB_PATH)
    vp, i64, i32, u32, f32 = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int, ctypes.c_uint32, ctypes.c_float
    pp = ctypes.POINTER(kn_peers)
    L.kn_abi_version.restype = i32
    L.kn_abi_version.argtypes = []
    L.kn_last_error.restype = ctypes.c_char_p
    L.kn_last_error.argtypes = []
    L.kn_device_info.restype = i32
    L.kn_device_info.argtypes = [ctypes.POINTER(ctypes.c_int)] * 3 + [ctypes.POINTER(ctypes.c_int64)]
    sig = {
        'kn_peer_sync': [vp, ctypes.c_int32, ctypes.c_int32, u32, u32, vp, vp, vp],
        'kn_spmm_csr_f32': [vp, vp, vp, i64, i64, vp, i64, vp, i64, i64, u32, pp, vp],
        'kn_spmm_csr_rows_f32': [vp, vp, vp, i64, i64, vp, vp, i64, vp, i64, i64, u32, pp, vp],
        'kn_csr_row_pattern_hash': [vp, vp, i64, vp, vp],
        'kn_pg_verify': [vp, vp, vp, vp, i64, vp, vp],
        'kn_pg_pack': [vp, vp, vp, vp, i64, ctypes.c_int32, ctypes.c_int32, vp, vp, vp],
        'kn_spmm_pg_f32': [vp, vp, vp, vp, vp, i64, ctypes.c_int32, ctypes.c_int32, vp, i64, vp, i64, i64, u32, pp, vp],
        'kn_spmm_pg_narrow_f32': [vp, vp, vp, vp, vp, i64, ctypes.c_int32, ctypes.c_int32, vp, vp, i64, ctypes.c_int32, vp, i64, vp, i64, i64, u32, pp, vp],
        'kn_spmm_cg_f32': [vp, vp, vp, vp, vp, vp, vp, vp, i64, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, vp, i64, vp, i64, i64, u32, pp, vp],
        'kn_debug_tc_timing': [ctypes.c_int32, vp],
        'kn_encrypt_monomial_t': [vp, i64, i64, vp, vp, vp, vp, i64, vp],
        'kn_splitk_reduce_f32': [vp, ctypes.c_int32, ctypes.c_int32, vp, vp, i64, i64, u32, pp, vp],
        'kn_spgemm_bound': [vp, vp, i64, vp, vp, vp],
        'kn_spgemm_rows': [vp, vp, vp, i64, vp, vp, vp, vp, vp, vp, vp, vp],
        'kn_csr_compact': [vp, vp, vp, i64, vp, vp, vp, vp],
        'kn_pg_tc_split': [vp, i64, vp, vp, vp],
        'kn_pg_tc_tensormaps': [vp, vp, i64, ctypes.c_int32, ctypes.c_int32, vp],
        'kn_spmm_pg_tc_f32': [vp, vp, vp, vp, vp, i64, ctypes.c_int32, ctypes.c_int32, vp, i64, vp, i64, i64, u32, pp, vp],
        'kn_exclusive_scan_i64': [vp, vp, i64, vp],
        'kn_toeplitz_conv2d_count': [ctypes.POINTER(kn_conv2d_desc), vp, i64, vp, vp],
        'kn_toeplitz_conv2d_fill': [ctypes.POINTER(kn_conv2d_desc), vp, vp, vp, i64, vp, vp, vp, vp],
        'kn_linear_count': [vp, vp, i64, i64, vp, i64, vp, vp],
        'kn_linear_fill': [vp, vp, i64, i64, vp, i64, vp, vp, vp, vp],
        'kn_keycompile_count': [vp, vp, vp, i64, vp, vp, vp, vp, i64, ctypes.c_int32, vp, vp],
        'kn_keycompile_fill': [vp, vp, vp, i64, i64, vp, vp, vp, vp, vp, i64, ctypes.c_int32, vp, vp, vp, vp],
        'kn_keyed_conv2d_count': [ctypes.POINTER(kn_conv2d_desc), vp, vp, vp, i64, vp, vp, vp, ctypes.c_int32, vp, vp],
        'kn_keyed_conv2d_fill': [ctypes.POINTER(kn_conv2d_desc), vp, vp, vp, i64, vp, vp, vp, vp, ctypes.c_int32, vp, vp, vp, vp],
        'kn_conv2d_groups_index': [ctypes.POINTER(kn_conv2d_desc), vp, i64, vp, vp, ctypes.c_int32, vp, vp, vp, vp],
        'kn_conv2d_groups_values': [ctypes.POINTER(kn_conv2d_desc), vp, vp, vp, i64, vp, vp, vp, ctypes.c_int32, vp, vp],
        'kn_conv2d_tiles_index': [ctypes.POINTER(kn_conv2d_desc), vp, i64, ctypes.c_int32, ctypes.c_int32, vp, vp, vp, vp, vp],
        'kn_spmm_tile_tc_f32': [vp, vp, vp, ctypes.c_int32, i64] + [ctypes.c_int32] * 7 + [vp, i64, vp, i64, i64, u32, pp, vp],
        'kn_convpool_f32': [ctypes.POINTER(kn_conv2d_desc), vp, vp, vp, ctypes.c_int32, ctypes.c_int32, f32, vp, vp, i64, vp, i64, i64, vp],
        'kn_csr_gather_rows_count': [vp, vp, i64, vp, vp],
        'kn_csr_gather_rows_fill': [vp, vp, vp, vp, i64, vp, vp, vp, vp],
        'kn_affine_to_linear_t': [vp, i64, i64, vp, i64, vp],
        'kn_linear_to_affine_t': [vp, i64, i64, i64, vp, f32, vp, vp],
    }
    for (name, argtypes) in sig.items():
        fn = getattr(L, name)
        fn.restype = i32
        fn.argtypes = argtypes
    _lib = L
    return L


def check(rc):
    if rc != 0:
        raise NativeError('libkeynet_b200 call failed (%d): %s' % (rc, lib().kn_last_error().decode('utf-8', 'replace')))


def ptr(t):
    """Device pointer of a torch tensor (None -> NULL)."""
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def stream_ptr():
    import torch
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def require_cuda():
    import torch
    if not torch.cuda.is_available():
        raise NativeError('keynet_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback')
