"""The kernels compiled into libkeynet_b200.so are exactly the ledger's (tests/kernel_ledger.py): a new template instantiation
cannot land without a ledger line, and tests/test_gpu_kernel_matrix.py then fails until a case runs it.  Runs without a GPU:
cuobjdump and cu++filt read the sm_100a cubins that nvcc cross-compiled."""
import os
import subprocess

from tests import kernel_ledger as kl


def _tool(name):
    nvcc = os.environ.get('NVCC', '/usr/local/cuda/bin/nvcc')
    path = os.path.join(os.path.dirname(nvcc), name)
    assert os.path.exists(path), '%s not found next to nvcc (%s)' % (name, nvcc)
    return path


def _compiled_entries():
    from keynet_b200 import build as kb
    lib = kb.build()
    out = subprocess.run([_tool('cuobjdump'), '-symbols', lib], check=True, capture_output=True, text=True).stdout
    mangled = [line.split()[-1] for line in out.splitlines() if 'STO_ENTRY' in line]
    assert mangled, 'cuobjdump listed no kernel entries in %s' % lib
    demangled = subprocess.run([_tool('cu++filt')], input='\n'.join(mangled) + '\n', check=True, capture_output=True, text=True).stdout.split('\n')
    names = [kl.normalise(d) for d in demangled[:len(mangled)]]
    return set(n for n in names if not n.startswith('$__internal'))


def test_normalise_both_spellings():
    prof = 'void (anonymous namespace)::pg_tc_kernel<2, true, 2, false>(CUtensorMap_st, CUtensorMap_st, int const*, long)'
    filt = 'void <unnamed>::pg_tc_kernel<(int)2, (bool)1, (int)2, (bool)0>(CUtensorMap_st, CUtensorMap_st, const int *, long)'
    assert kl.normalise(prof) == kl.normalise(filt) == 'pg_tc_kernel<2,true,2,false>'
    assert kl.normalise('(anonymous namespace)::tile_sum_kernel(long const*, long, long*)') == 'tile_sum_kernel'
    assert kl.normalise('<unnamed>::tile_sum_kernel(const long *, long, long *)') == 'tile_sum_kernel'


def test_ledger_shape():
    assert len(kl.SPMM_KERNELS) == len(set(kl.SPMM_KERNELS)) == 84
    assert not set(kl.SPMM_KERNELS) & set(kl.OTHER_KERNELS)
    here = os.path.dirname(os.path.abspath(__file__))
    missing = sorted(set(f for f in kl.OTHER_KERNELS.values() if not os.path.exists(os.path.join(here, f))))
    assert not missing, 'test modules named in OTHER_KERNELS do not exist: %s' % missing


def test_library_kernels_equal_ledger():
    compiled = _compiled_entries()
    ledger = set(kl.SPMM_KERNELS) | set(kl.OTHER_KERNELS)
    unlisted = sorted(compiled - ledger)
    absent = sorted(ledger - compiled)
    assert not unlisted and not absent, ('kernels compiled but missing from tests/kernel_ledger.py: %s; '
                                         'ledger entries not compiled: %s' % (unlisted, absent))
