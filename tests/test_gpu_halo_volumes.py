"""
Plane windows (tnmf_update_h_planes / tnmf_gradient_w_planes) and halo-sharded volume fits on the GPU.

The windowed H update writes the activation planes [t_lo, t_hi) only and must equal the oracle's full update there; the
windowed W gradient must equal the oracle's correlation with an H that is zero outside the window (against R of all of
H).  Float32 volumes run on the plane mode of the tensor-memory kernels (within 2e-5 of max|ref|), float64 on the generic
kernels (1e-12); the full window is bitwise equal to the unwindowed calls.  Then RowShardedNMF on two gloo ranks sharing
the GPU: a float32 volume on the tc3 kernels with sparsity and both inhibition terms within the fit bounds of DESIGN §4,
and a float64 volume on the generic kernels to 1e-9.
"""
import ctypes
import os
import socket

import numpy as np
import pytest
import torch

from oracle import tnmf_oracle as orc

pytestmark = pytest.mark.gpu

REG, LAM, LAM_X = 0.05, 0.2, 0.1


def _backend(V, W, H, mode='valid'):
    from tnmf_b200 import B200_Backend
    be = B200_Backend(reconstruction_mode=mode)
    state = np.random.get_state()
    Wd, Hd = be.initialize(V, W.shape[2:], W.shape[0], None, tuple(range(-(W.ndim - 2), 0)))
    np.random.set_state(state)
    Wd.copy_(torch.from_numpy(W))
    Hd.copy_(torch.from_numpy(H))
    return be, Wd, Hd


def _close(a, b, tol):
    a = a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)
    scale = max(float(np.abs(b).max()), 1e-30)
    err = float(np.abs(a.astype(np.float64) - b.astype(np.float64)).max()) / scale
    assert err <= tol, f'max|delta|/max|ref| = {err:.3e} > {tol:.1e}'


def _ref_update(V, W, H, mode, kernels, lo, hi):
    """The oracle's H update with sparsity and both inhibition terms, kept on the planes [lo, hi) only."""
    nmf = orc.OracleNMF(W.shape[0], W.shape[2:], reconstruction_mode=mode)
    nmf.inhibition_kernels = kernels
    nmf.V, nmf.W, nmf.H = V, W, H.copy()
    nmf.update_H(slice(None), sparsity=REG, inhibition=LAM, cross_inhibition=LAM_X)
    out = H.copy()
    out[:, :, lo:hi] = nmf.H[:, :, lo:hi]
    return out


def _ref_gradient_w(V, W, H, mode, lo, hi):
    Hw = np.zeros_like(H)
    Hw[:, :, lo:hi] = H[:, :, lo:hi]
    R = orc.reconstruct(W, H, mode)
    Hp = orc.pad_activations(Hw, W.shape[2:], mode)
    return (orc._correlate_with_activations(V, Hp, W.shape[2:]), orc._correlate_with_activations(R, Hp, W.shape[2:]))


# N, C, M, D, A: T_z = 10, p = 2.  Windows: full, interior, either edge, one plane, and two that leave a_z launches of the
# W gradient without sample planes ([0, 1): a_z = 0, 1; [9, 10): a_z = 1, 2).
SHAPE = (2, 2, 9, (8, 12, 10), (3, 3, 3))
WINDOWS = [(0, 10), (3, 7), (0, 4), (6, 10), (5, 6), (0, 1), (9, 10)]


def _data(dtype, mode, seed=5):
    N, C, M, D, A = SHAPE
    rng = np.random.default_rng(seed)
    V = rng.random((N, C) + D).astype(dtype)
    W = rng.random((M, C) + A).astype(dtype)
    H = rng.random((N, M) + orc.transform_shape(mode, D, A)).astype(dtype)
    return V, W, H


@pytest.mark.parametrize('dtype,mode', [(np.float32, 'valid'), (np.float64, 'valid'), (np.float64, 'full')])
@pytest.mark.parametrize('window', WINDOWS)
def test_windowed_operations_vs_oracle(dtype, mode, window):
    V, W, H = _data(dtype, mode)
    T0 = H.shape[2]
    lo, hi = min(window[0], T0), min(window[1], T0)
    kernels = orc.inhibition_kernels((2, 1, 1))
    V64, W64, H64 = (x.astype(np.float64) for x in (V, W, H))
    tol = 2e-5 if dtype == np.float32 else 1e-12
    be, Wd, Hd = _backend(V, W, H, mode)
    expect = ({'update_h': 'hupd_ts3_kernel', 'gradient_w': 'gradw_ns3_kernel'} if dtype == np.float32 else
              {'update_h': 'generic_gradient_h_kernel', 'gradient_w': 'generic_gradient_w_kernel'})
    neg, pos = _ref_gradient_w(V64, W64, H64, mode, lo, hi)
    out = torch.empty((2, *Wd.shape), dtype=Wd.dtype, device=Wd.device)
    be.gradient_W(V, Wd, Hd, slice(None), out, planes=(lo, hi))
    _close(out[0], neg, tol)
    _close(out[1], pos, tol)
    names = be.kernel_names()
    assert {k: names[k] for k in expect} == expect, names
    be.update_H(V, Wd, Hd, slice(None), REG, LAM, LAM_X, kernels, planes=(lo, hi))
    got = Hd.cpu().numpy()
    _close(got, _ref_update(V64, W64, H64, mode, kernels, lo, hi), tol)
    outside = np.ones(T0, bool)
    outside[lo:hi] = False
    assert np.array_equal(got[:, :, outside], H[:, :, outside])           # never written outside the window


@pytest.mark.parametrize('dtype', [np.float32, np.float64])
def test_full_window_is_bitwise_the_unwindowed_call(dtype):
    V, W, H = _data(dtype, 'valid', seed=6)
    kernels = orc.inhibition_kernels((2, 1, 1))
    outs = []
    for planes in (None, (0, H.shape[2])):
        be, Wd, Hd = _backend(V, W, H)
        g = torch.empty((2, *Wd.shape), dtype=Wd.dtype, device=Wd.device)
        be.gradient_W(V, Wd, Hd, slice(None), g, planes=planes)
        be.update_H(V, Wd, Hd, slice(None), REG, LAM, LAM_X, kernels, planes=planes)
        outs.append((g.clone(), Hd.clone()))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])


def test_windowed_w_gradient_within_the_unwindowed_workspace():
    """The unwindowed problem's tnmf_workspace_bytes bound the windowed call (include/tnmf_b200.h): a window that leaves
    a_z launches empty runs in exactly that workspace, and a smaller one is refused."""
    from tnmf_b200 import _lib
    V, W, H = _data(np.float32, 'valid', seed=7)
    be, Wd, Hd = _backend(V, W, H)
    lib = _lib.load()
    p, Hd = be._h_problem(Hd)                                   # pylint: disable=protected-access
    need = int(lib.tnmf_workspace_bytes(ctypes.byref(p)))
    Vd = be._device_V(V)                                        # pylint: disable=protected-access
    R = be.reconstruct(Wd, Hd)
    lo, hi = 0, 1                                               # a_z = 0 and 1 have no sample planes in the window
    ws = torch.full((need,), 0xff, dtype=torch.uint8, device=Vd.device)     # stale partials must not leak in
    out = torch.empty((2, *Wd.shape), dtype=Wd.dtype, device=Wd.device)
    st = torch.cuda.current_stream().cuda_stream
    args = (ctypes.byref(p), Vd.data_ptr(), R.data_ptr(), Hd.data_ptr(), out[0].data_ptr(), out[1].data_ptr(), lo, hi,
            ws.data_ptr())
    assert lib.tnmf_gradient_w_planes(*args, need - 256, st) == _lib.TNMF_EWORKSPACE
    _lib.check(lib.tnmf_gradient_w_planes(*args, need, st))
    neg, pos = _ref_gradient_w(V.astype(np.float64), W.astype(np.float64), H.astype(np.float64), 'valid', lo, hi)
    _close(out[0], neg, 2e-5)
    _close(out[1], pos, 2e-5)


def test_windowed_calls_are_unsupported_on_the_2d_families():
    from tnmf_b200 import B200_Backend
    rng = np.random.default_rng(3)
    V = rng.random((2, 3, 96, 140), dtype=np.float32)
    be = B200_Backend()
    W, H = be.initialize(V, (11, 11), 16)
    with pytest.raises(NotImplementedError):
        be.update_H(V, W, H, slice(None), planes=(0, 10))
    with pytest.raises(NotImplementedError):
        be.gradient_W(V, W, H, slice(None), torch.empty((2, *W.shape), device=W.device), planes=(0, 10))


# ---------------------------------------------------------------------------------------------------------
# halo-sharded volume fits: two gloo ranks on one GPU
# ---------------------------------------------------------------------------------------------------------
def _free_port():
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        return s.getsockname()[1]


def _rank_main(rank, world, port, V, atoms, atom_shape, mode, inhibition_range, kw_fit, out):
    import torch.distributed as dist
    from tnmf_b200 import RowShardedNMF
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    torch.cuda.set_device(0)
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        np.random.seed(43)
        nmf = RowShardedNMF(atoms, atom_shape, reconstruction_mode=mode, inhibition_range=inhibition_range)
        energies = []
        nmf.fit(V, progress_callback=lambda m, i: energies.append(m.energy()) or True, **kw_fit)
        out[rank] = (nmf.W, nmf.gather_H(), energies, nmf.ops.be.kernel_names(), nmf.ops.windowed,
                     nmf.ops.H_own is None, nmf.halo)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize('case', ['f32_tc3', 'f64_generic', 'f64_generic_full'])
def test_row_sharded_volume_fit_equals_oracle(case):
    import torch.multiprocessing as mp
    rng = np.random.default_rng(9)
    mode = 'full' if case.endswith('full') else 'valid'
    atoms, atom_shape, inhibition_range = 8, (3, 3, 3), (3, 1, 2)          # halo = r0 = 3 planes > p = 2
    if case == 'f32_tc3':
        V, iters, rtol_e, tol = rng.random((1, 1, 24, 18, 20), dtype=np.float32), 10, 1e-4, 1e-3
    else:
        V, iters, rtol_e, tol = rng.random((1, 2, 14, 9, 8)), 6, 1e-9, 1e-9
    kw_fit = dict(n_iterations=iters, sparsity_H=0.05, inhibition_strength=0.2, cross_atom_inhibition_strength=0.1)
    np.random.seed(43)
    ref = orc.OracleNMF(atoms, atom_shape, inhibition_range=inhibition_range, reconstruction_mode=mode)
    e_ref = []
    ref.fit_batch(V.astype(np.float64), progress_callback=lambda m, i: e_ref.append(float(m.energy())) or True, **kw_fit)
    world = 2
    ctx = mp.get_context('spawn')
    with ctx.Manager() as mgr:
        out = mgr.dict()
        mp.spawn(_rank_main, args=(world, _free_port(), V, atoms, atom_shape, mode, inhibition_range, kw_fit, out),
                 nprocs=world, join=True)
        results = [out[r] for r in range(world)]
    W0, H0, e0, names, windowed, no_h_own, halo = results[0]
    print(case, names, 'energy', e0[-1], e_ref[-1])
    assert halo == 3 and windowed and no_h_own
    if case == 'f32_tc3':
        assert names == {'reconstruct': 'recon_os3_kernel', 'update_h': 'hupd_ts3_kernel',
                         'gradient_w': 'gradw_ns3_kernel'}, names
    else:
        assert names['update_h'] == 'generic_gradient_h_kernel' and names['gradient_w'] == 'generic_gradient_w_kernel'
    assert np.allclose(e0, e_ref, rtol=rtol_e)
    assert np.abs(W0 - ref.W).max() <= tol * np.abs(ref.W).max()
    assert np.abs(H0 - ref.H).max() <= tol * np.abs(ref.H).max()
    for W, _, e, _, windowed_r, no_h_own_r, _ in results[1:]:
        assert np.array_equal(W, W0) and windowed_r and no_h_own_r
