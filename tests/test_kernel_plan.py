"""
CPU-side checks of the kernel plan in the C-ABI layer: which kernel serves each operation (name, family and launch
count), the status codes of the TMA kernels' fallback for misaligned operands or a missing workspace, and the window
entry points' refusal of the 2-D kernel families.  Every call here returns before any kernel launch; the pointers are
fake addresses that are (256) or are not (260) 16-byte aligned.
"""
import ctypes

import pytest

from tnmf_b200 import _lib

OPS = (_lib.OP_RECONSTRUCT, _lib.OP_GRADIENT_H, _lib.OP_GRADIENT_W)
TC, TMA, TILED, GENERIC = (_lib.PATHS[k] for k in ('tc', 'tma', 'tiled', 'generic'))
ALIGNED, MISALIGNED = ctypes.c_void_p(256), ctypes.c_void_p(260)
BIG = 1 << 40


@pytest.fixture(scope='module')
def lib():
    _lib.build()
    return _lib.load()


def problem(n, c, m, sample, atom, dtype=_lib.TNMF_F32, mode='valid', path='auto', flags=0):
    """A problem with H rows padded to 16 bytes, laid out the way B200_Backend.initialize allocates H."""
    t = [d + a - 1 if mode == 'valid' else d - a + 1 if mode == 'full' else d for d, a in zip(sample, atom)]
    pitch = (t[-1] + 3) // 4 * 4
    hsm = pitch
    for e in t[:-1]:
        hsm *= e
    return _lib.make_problem(n, c, m, sample, atom, dtype, mode, path, m * hsm, hsm, pitch if len(sample) >= 2 else 0,
                             flags)


def plan(lib, p):
    return ([lib.tnmf_kernel_name(ctypes.byref(p), op).decode() for op in OPS],
            [lib.tnmf_kernel_family(ctypes.byref(p), op) for op in OPS],
            [lib.tnmf_launch_count(ctypes.byref(p), op) for op in OPS])


CFG2 = (64, 3, 16, (256, 256), (11, 11))          # BASELINE config 2
CFG3 = (8, 1, 32, (128, 128), (15, 15))           # BASELINE config 3
CFG5 = (2, 1, 8, (512, 512), (64, 64))            # BASELINE config 5
VOL = (16, 1, 8, (64, 64, 64), (7, 7, 7))        # tools/bench_3d.py

# (problem, kernel names, families, launch counts of reconstruction, H update, W gradient); together every hot kernel
CASES = {
    'tensor_memory_operand': (problem(*CFG2), ['recon_ts_kernel', 'hupd_ts_kernel', 'gradw_ts_kernel'], [TC] * 3,
                              [1, 1, 2]),
    'narrow_atoms': (problem(*CFG3), ['recon_os_kernel', 'hupd_ts_kernel', 'gradw_ns_kernel'], [TC] * 3, [1, 2, 5]),
    # the round-1 (shared-memory operand) kernels where 'auto' still picks them
    'round1_recon_hupd': (problem(8, 3, 16, (128, 128), (13, 17)),
                          ['recon_tc_kernel', 'hupd_tc_kernel', 'gradw_ts_kernel'], [TC] * 3, [1, 1, 2]),
    'round1_gradw': (problem(8, 1, 8, (128, 128), (14, 17)),
                     ['recon_tma_kernel', 'hupd_tma_kernel', 'gradw_tc_kernel'], [TMA, TMA, TC], [2, 2, 2]),
    # tall atoms: 'auto' keeps the W gradient on TMA, forced 'tc' runs it in row chunks
    'tall_atoms_auto': (problem(*CFG5), ['recon_tma_kernel', 'tiled::hupd_kernel', 'gradw_tma_kernel'],
                        [TMA, TILED, TMA], [2, 1, 2]),
    'tall_atoms_tc': (problem(*CFG5, path='tc'), ['recon_tma_kernel', 'tiled::hupd_kernel', 'gradw_tc_kernel'],
                      [TMA, TILED, TC], [2, 1, 9]),
    'tma': (problem(*CFG2, flags=_lib.FLAG_NO_TC), ['recon_tma_kernel', 'hupd_tma_kernel', 'gradw_tma_kernel'],
            [TMA] * 3, [2, 2, 2]),
    'tiled': (problem(*CFG2, mode='circular'), ['tiled::recon_kernel', 'tiled::hupd_kernel', 'tiled::gradw_kernel'],
              [TILED] * 3, [1, 1, 2]),
    'generic': (problem(*CFG2, dtype=_lib.TNMF_F64),
                ['generic_reconstruct_kernel', 'generic_gradient_h_kernel', 'generic_gradient_w_kernel'],
                [GENERIC] * 3, [1, 1, 2]),
    'volume': (problem(*VOL), ['recon_os3_kernel', 'hupd_ts3_kernel', 'gradw_ns3_kernel'], [TC] * 3, [7, 1, 8]),
}


@pytest.mark.parametrize('case', sorted(CASES))
def test_kernel_plan(lib, case):
    p, names, families, launches = CASES[case]
    assert plan(lib, p) == (names, families, launches)


def test_every_hot_kernel_is_planned_somewhere():
    names = {n for _, ns, _, _ in CASES.values() for n in ns}
    assert len(names) == 20, sorted(names)


def test_tma_fallback_status_codes(lib):
    """A forced 'tma' that cannot run: missing workspace -> TNMF_EWORKSPACE, misaligned operand -> TNMF_EUNSUPPORTED,
    in the order each entry point checks them."""
    p = problem(*CFG2, path='tma')
    assert plan(lib, p)[0] == ['recon_tma_kernel', 'hupd_tma_kernel', 'gradw_tma_kernel']
    P, A, M = ctypes.byref(p), ALIGNED, MISALIGNED
    e = ctypes.byref(ctypes.c_double())
    # reconstruction: H must be aligned and a workspace given; the missing workspace is reported first
    assert lib.tnmf_reconstruct(P, A, A, A, None, 0, None) == _lib.TNMF_EWORKSPACE
    assert lib.tnmf_reconstruct(P, A, M, A, None, 0, None) == _lib.TNMF_EWORKSPACE
    assert lib.tnmf_reconstruct(P, A, M, A, A, BIG, None) == _lib.TNMF_EUNSUPPORTED
    # energy: the workspace is required before any kernel is chosen
    assert lib.tnmf_reconstruct_energy(P, A, A, M, A, e, None, 0, None) == _lib.TNMF_EINVAL
    assert lib.tnmf_reconstruct_energy(P, A, A, M, A, e, A, 16, None) == _lib.TNMF_EWORKSPACE
    assert lib.tnmf_reconstruct_energy(P, A, A, M, A, e, A, BIG, None) == _lib.TNMF_EUNSUPPORTED
    # H gradient / update: V and R must be aligned and a workspace given
    assert lib.tnmf_update_h(P, A, A, A, A, 0.0, None, 0.0, None, 0.0, None, 0, None) == _lib.TNMF_EWORKSPACE
    assert lib.tnmf_update_h(P, M, A, A, A, 0.0, None, 0.0, None, 0.0, None, 0, None) == _lib.TNMF_EWORKSPACE
    assert lib.tnmf_update_h(P, A, M, A, A, 0.0, None, 0.0, None, 0.0, A, BIG, None) == _lib.TNMF_EUNSUPPORTED
    assert lib.tnmf_gradient_h(P, A, A, A, A, A, None, 0, None) == _lib.TNMF_EWORKSPACE
    assert lib.tnmf_gradient_h(P, M, A, A, A, A, A, BIG, None) == _lib.TNMF_EUNSUPPORTED
    # W gradient: V, R and H must be aligned; the workspace is checked after that
    for v, r, h in ((M, A, A), (A, M, A), (A, A, M)):
        assert lib.tnmf_gradient_w(P, v, r, h, A, A, None, 0, None) == _lib.TNMF_EUNSUPPORTED
        assert lib.tnmf_gradient_w(P, v, r, h, A, A, A, BIG, None) == _lib.TNMF_EUNSUPPORTED
    assert lib.tnmf_gradient_w(P, A, A, A, A, A, None, 0, None) == _lib.TNMF_EWORKSPACE
    assert lib.tnmf_gradient_w(P, A, A, A, A, A, A, 16, None) == _lib.TNMF_EWORKSPACE


@pytest.mark.parametrize('case', ['tensor_memory_operand', 'tma'])
def test_window_entry_points_refuse_2d_kernels(lib, case):
    """The plane windows run on the generic kernels and the 3-D plane mode only."""
    p = CASES[case][0]
    P, A = ctypes.byref(p), ALIGNED
    assert lib.tnmf_update_h_planes(P, A, A, A, A, 0.0, None, 0.0, None, 0.0, 0, 1, A, BIG, None) == \
        _lib.TNMF_EUNSUPPORTED
    assert lib.tnmf_gradient_w_planes(P, A, A, A, A, A, 0, 1, A, BIG, None) == _lib.TNMF_EUNSUPPORTED
