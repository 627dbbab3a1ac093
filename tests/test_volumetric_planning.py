"""
CPU-side checks of the 3-D (volumetric) kernel choice: float32 'valid' problems with three shift axes run on the plane
mode of the tensor-memory kernels (DESIGN.md §3.10) where they plan; everything else stays on the generic kernels.
"""
import ctypes

import pytest

from tnmf_b200 import _lib

OPS = (_lib.OP_RECONSTRUCT, _lib.OP_GRADIENT_H, _lib.OP_GRADIENT_W)
TC3 = ['recon_os3_kernel', 'hupd_ts3_kernel', 'gradw_ns3_kernel']
GENERIC = ['generic_reconstruct_kernel', 'generic_gradient_h_kernel', 'generic_gradient_w_kernel']


@pytest.fixture(scope='module')
def lib():
    _lib.build()
    return _lib.load()


def _names(lib, p):
    return [lib.tnmf_kernel_name(ctypes.byref(p), op).decode() for op in OPS]


def _launches(lib, p):
    return [lib.tnmf_launch_count(ctypes.byref(p), op) for op in OPS]


@pytest.mark.parametrize('n', [16, 1])
def test_benchmark_geometry_runs_on_tensor_cores(lib, n):
    """tools/bench_3d.py: 1 x 64^3 samples, 8 atoms of 7 x 7 x 7."""
    p = _lib.make_problem(n, 1, 8, (64, 64, 64), (7, 7, 7), _lib.TNMF_F32)
    assert _names(lib, p) == TC3
    assert [lib.tnmf_kernel_family(ctypes.byref(p), op) for op in OPS] == [_lib.PATHS['tc']] * 3
    # one reconstruction per atom plane; one H update per 16 atoms; one W gradient per atom plane and 8 atoms + the
    # finishing reduction
    assert _launches(lib, p) == [7, 1, 7 + 1]
    # the per-plane W gradient partials and, for the energy without a caller's R, R-sized scratch
    assert lib.tnmf_workspace_bytes(ctypes.byref(p)) >= 4 * n * 64 ** 3


def test_launch_count_follows_the_atom_blocks(lib):
    p = _lib.make_problem(2, 2, 20, (5, 12, 9), (3, 3, 3), _lib.TNMF_F32)
    assert _names(lib, p) == TC3
    assert _launches(lib, p) == [3, 2, 3 * 3 + 1]


def test_small_and_unsupported_problems_stay_generic(lib):
    # two atoms fill an eighth of the 16-atom block (tests/test_cabi.py pins this problem to the generic kernels)
    small = _lib.make_problem(2, 1, 2, (8, 8, 8), (3, 3, 3), _lib.TNMF_F32)
    assert _names(lib, small) == GENERIC
    assert lib.tnmf_uses_tiled_path(ctypes.byref(small)) == 0
    assert _launches(lib, small) == [1, 1, 2]
    for dtype, mode in ((_lib.TNMF_F64, 'valid'), (_lib.TNMF_F32, 'full'), (_lib.TNMF_F32, 'circular')):
        p = _lib.make_problem(16, 1, 8, (64, 64, 64), (7, 7, 7), dtype, mode)
        assert _names(lib, p) == GENERIC, (dtype, mode)
        p.path = _lib.PATHS['tc']                   # forced: tensor cores where a kernel plans, generic otherwise
        assert _names(lib, p) == GENERIC, (dtype, mode)


def test_forced_and_switched_off(lib):
    p = _lib.make_problem(2, 1, 2, (8, 8, 8), (3, 3, 3), _lib.TNMF_F32)
    p.path = _lib.PATHS['tc']
    assert _names(lib, p) == TC3
    p.path = _lib.PATHS['tma']
    assert lib.tnmf_kernel_family(ctypes.byref(p), _lib.OP_GRADIENT_H) == -1
    q = _lib.make_problem(16, 1, 8, (64, 64, 64), (7, 7, 7), _lib.TNMF_F32)
    q.flags = _lib.FLAG_NO_TC_RECON
    assert _names(lib, q) == [GENERIC[0]] + TC3[1:]
    q.flags = _lib.FLAG_NO_TMEM_OPERAND
    assert _names(lib, q) == GENERIC
    # three channels: no reconstruction kernel plans (recon_os takes C <= 2), the other two do
    c3 = _lib.make_problem(2, 3, 9, (5, 12, 9), (2, 3, 3), _lib.TNMF_F32)
    assert _names(lib, c3) == [GENERIC[0]] + TC3[1:]
