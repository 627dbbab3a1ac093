"""
GPU tests of the Kullback-Leibler updates (`divergence='kl'`, DESIGN.md §3.11) against the float64 reference of
tests/kl_reference.py: the quotient kernel bit for bit against torch, single operations on every kernel family that
serves them, multi-iteration fits, the minibatch and graph-replay paths, launch bookkeeping and a two-rank sharded fit.

Bounds: single operations within 2e-5 of max|ref| in float32 and 1e-9 in float64; fits: the divergence trajectory within
1e-4 relative, W and H within 1e-3 of max|ref|.
"""
import ctypes
import os

import numpy as np
import pytest
import torch

import kl_reference as klr
from oracle import tnmf_oracle as orc

pytestmark = pytest.mark.gpu


def _backend(V, W, H, mode='valid', path='auto', **kw):
    from tnmf_b200 import B200_Backend
    be = B200_Backend(reconstruction_mode=mode, kernel_path=path, **kw)
    state = np.random.get_state()
    Wd, Hd = be.initialize(V, W.shape[2:], W.shape[0], None, tuple(range(-(W.ndim - 2), 0)))
    np.random.set_state(state)
    Wd.copy_(torch.from_numpy(W))
    Hd.copy_(torch.from_numpy(H))
    return be, Wd, Hd


def _err(a, b) -> float:
    a = a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)
    return float(np.abs(a.astype(np.float64) - b.astype(np.float64)).max()) / max(float(np.abs(b).max()), 1e-30)


def _close(a, b, tol, what=''):
    err = _err(a, b)
    assert err <= tol, f'{what}: max|delta|/max|ref| = {err:.3e} > {tol:.1e}'


def _data(N, C, M, D, A, mode, dtype, seed):
    rng = np.random.default_rng(seed)
    V = rng.random((N, C) + D).astype(dtype)
    V[V < 0.05] = 0                                     # exact zeros: Q = 0 there
    W = rng.random((M, C) + A).astype(dtype)
    H = rng.random((N, M) + orc.transform_shape(mode, D, A)).astype(dtype)
    return V, W, H


# ---------------------------------------------------------------------------------------------------------
# the quotient kernel
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('dtype', [torch.float32, torch.float64])
def test_quotient_kernel_bitwise_against_torch(dtype):
    from tnmf_b200 import _lib
    lib = _lib.load()
    code = _lib.TNMF_F32 if dtype == torch.float32 else _lib.TNMF_F64
    tau = torch.finfo(dtype).tiny
    g = torch.Generator(device='cuda').manual_seed(5)
    st = torch.cuda.current_stream().cuda_stream
    for n, lead in ((1, 0), (7, 1), (4099, 0), (4099, 3), (1 << 20, 0), ((1 << 21) + 5, 2), (12_582_917, 1)):
        V = torch.rand(n + lead, generator=g, device='cuda', dtype=dtype)
        R = torch.rand(n + lead, generator=g, device='cuda', dtype=dtype) * 2
        V[V < 0.1] = 0
        if n >= 8:                                      # R at and below tau, zero, and R exactly equal to V
            R[lead:lead + 6] = torch.tensor([tau, tau / 2, tau / 8, 0.0, tau * 2, tau], dtype=dtype)
            R[lead + 6:lead + 8] = V[lead + 6:lead + 8]
        Vs, Rs = V[lead:], R[lead:]                     # a leading slice: misaligned for the 16-byte packs when lead > 0
        want = torch.where(Vs > 0, Vs / Rs.clamp(min=tau), torch.zeros((), dtype=dtype, device='cuda'))
        V64, R64 = Vs.double(), Rs.double()
        d_ref = float(torch.sum(torch.where(V64 > 0, V64 * torch.log(torch.where(V64 > 0, V64, 1.0) /
                                                                     Rs.clamp(min=tau).double()), 0.0) - V64 + R64))
        p = _lib.make_problem(n, 1, 1, (1,), (1,), code)
        ws = torch.empty(lib.tnmf_kl_workspace_bytes(ctypes.byref(p)), dtype=torch.uint8, device='cuda')
        out = []
        for _ in range(2):
            Q = Rs.clone()
            e = torch.empty((), dtype=torch.float64, device='cuda')
            _lib.check(lib.tnmf_kl_quotient(ctypes.byref(p), Vs.data_ptr(), Q.data_ptr(), e.data_ptr(), ws.data_ptr(),
                                            ws.numel(), st))
            out.append((Q, float(e)))
        Q2 = Rs.clone()
        _lib.check(lib.tnmf_kl_quotient(ctypes.byref(p), Vs.data_ptr(), Q2.data_ptr(), None, None, 0, st))
        torch.cuda.synchronize()
        print(f'n={n} lead={lead}: D {out[0][1]:.17g} float64 sum {d_ref:.17g} rel {abs(out[0][1] - d_ref) / d_ref:.2e}')
        assert torch.equal(out[0][0], want), n
        assert torch.equal(out[1][0], want) and torch.equal(Q2, want)
        assert out[0][1] == out[1][1]
        assert abs(out[0][1] - d_ref) <= 1e-12 * abs(d_ref)


# ---------------------------------------------------------------------------------------------------------
# single KL operations on each kernel family
# ---------------------------------------------------------------------------------------------------------
TS = ('recon_ts_kernel', 'hupd_ts_kernel', 'gradw_ts_kernel')
OS = ('recon_os_kernel', 'hupd_ts_kernel', 'gradw_ns_kernel')
OS3 = ('recon_os3_kernel', 'hupd_ts3_kernel', 'gradw_ns3_kernel')
TMA = ('recon_tma_kernel', 'hupd_tma_kernel', 'gradw_tma_kernel')
TILED = ('tiled::recon_kernel', 'tiled::hupd_kernel', 'tiled::gradw_kernel')
GEN = ('generic_reconstruct_kernel', 'generic_gradient_h_kernel', 'generic_gradient_w_kernel')
OP_CASES = [
    # N, C, M, D, A, mode, dtype, backend keywords, kernels (reconstruct, update_h, gradient_w)
    (3, 3, 16, (64, 64), (11, 11), 'valid', np.float32, {}, TS),                      # cfg2-like
    (3, 3, 16, (64, 64), (11, 11), 'full', np.float32, {}, TS),
    (2, 1, 32, (64, 128), (15, 15), 'valid', np.float32, {}, OS),                     # cfg3-like
    (2, 1, 32, (64, 128), (15, 15), 'full', np.float32, {}, OS),
    (2, 1, 16, (8, 32, 32), (3, 5, 5), 'valid', np.float32, {}, OS3),                 # a volume
    (3, 3, 16, (64, 64), (11, 11), 'valid', np.float32, dict(tensor_cores=False), TMA),
    (9, 1, 17, (256,), (32,), 'valid', np.float32, dict(rows_view=True), TMA),        # 1-D rows view, TMA
    (2, 3, 4, (40, 70), (11, 11), 'valid', np.float32, dict(path='tiled'), TILED),
    (2, 3, 4, (40, 70), (11, 11), 'full', np.float32, dict(path='tiled'), TILED),
    (3, 3, 16, (64, 64), (11, 11), 'circular', np.float32, {}, TILED),
    (2, 2, 6, (1000,), (50,), 'valid', np.float32, dict(path='tiled'), TILED),        # 1-D
    (9, 1, 17, (256,), (32,), 'full', np.float32, dict(path='tiled', rows_view=True), TILED),
    (2, 2, 3, (12, 10), (3, 4), 'valid', np.float64, {}, GEN),
    (2, 2, 3, (12, 10), (3, 4), 'full', np.float64, {}, GEN),
    (2, 2, 3, (6, 7, 5), (2, 3, 2), 'circular', np.float64, {}, GEN),
]


@pytest.mark.parametrize('case', range(len(OP_CASES)))
def test_single_kl_operations_vs_reference(case):
    N, C, M, D, A, mode, dtype, kw, kernels = OP_CASES[case]
    kw = dict(kw)
    path = kw.pop('path', 'auto')
    V, W, H = _data(N, C, M, D, A, mode, dtype, 500 + case)
    V64, W64, H64 = V.astype(np.float64), W.astype(np.float64), H.astype(np.float64)
    tol = 2e-5 if dtype == np.float32 else 1e-9
    be, Wd, Hd = _backend(V, W, H, mode, path, **kw)
    # the H update on a minibatch slice and on the rest (the ones tensor is sliced like V), then on the whole batch
    H_ref = H64.copy()
    for s in (slice(0, 1), slice(1, N), slice(None)):
        neg, pos = klr.gradient_H(V64[s], W64, H_ref[s], mode)
        orc.multiplicative_update(H_ref[s], neg, pos)
        be.update_H(V, Wd, Hd, s, divergence='kl')
    assert tuple(be.kernel_names().values()) == kernels, be.kernel_names()
    e_h = _err(Hd, H_ref)
    # the W gradient and update from the device's H
    H1 = Hd.detach().cpu().numpy().astype(np.float64)
    grad = torch.empty((2, *Wd.shape), dtype=Wd.dtype, device=Wd.device)
    be.gradient_W(V, Wd, Hd, slice(None), grad, divergence='kl')
    rn, rp = klr.gradient_W(V64, W64, H1, mode)
    e_neg, e_pos = _err(grad[0], rn), _err(grad[1], rp)
    be.apply_W_update(Wd, grad)
    W_ref = W64.copy()
    orc.multiplicative_update(W_ref, rn, rp, normalization_axes=tuple(range(-len(A), 0)))
    e_w = _err(Wd, W_ref)
    e = float(be.energy(V, Wd, Hd, divergence='kl'))
    d_ref = klr.divergence(V64, orc.reconstruct(W_ref, H1, mode))
    print(f'{OP_CASES[case][:6]} {kernels}: H {e_h:.2e} gradW neg {e_neg:.2e} pos {e_pos:.2e} W {e_w:.2e} '
          f'D {abs(e - d_ref) / d_ref:.2e}')
    for err, what in ((e_h, 'H update'), (e_neg, 'W gradient neg'), (e_pos, 'W gradient pos'), (e_w, 'W update')):
        assert err <= tol, f'{what}: {err:.3e} > {tol:.1e}'
    assert abs(e - d_ref) <= tol * abs(d_ref)


# ---------------------------------------------------------------------------------------------------------
# fits
# ---------------------------------------------------------------------------------------------------------
FIT_CASES = {
    # name: N, C, M, D, A, benched batch (kernel_names() of the fit must equal those of this batch), iterations
    'cfg2': (1, 3, 16, (256, 256), (11, 11), 64, 6),
    'cfg3': (2, 1, 32, (128, 128), (15, 15), 1024, 8),
    'volume': (2, 1, 16, (8, 32, 32), (3, 5, 5), 16, 8),
}


@pytest.mark.parametrize('regularised', (False, True))
@pytest.mark.parametrize('name', sorted(FIT_CASES))
def test_kl_fit_vs_reference(name, regularised):
    from tnmf_b200 import TransformInvariantNMF
    N, C, M, D, A, n_bench, iters = FIT_CASES[name]
    rng = np.random.default_rng(11)
    V = rng.random((N, C) + D).astype(np.float32)
    V[V < 0.05] = 0
    kw = dict(n_iterations=iters)
    if regularised:
        kw.update(sparsity_H=0.05, inhibition_strength=0.1, cross_atom_inhibition_strength=0.05)
    np.random.seed(13)
    ref = klr.OracleKL(M, A)
    e_ref = []
    ref.fit_batch(V.astype(np.float64), progress_callback=lambda m, i: e_ref.append(m.energy()) or True, **kw)
    np.random.seed(13)
    nmf = TransformInvariantNMF(n_atoms=M, atom_shape=A, divergence='kl')
    e_gpu = []
    nmf.fit(V, progress_callback=lambda m, i: e_gpu.append(m._energy_function()) or True, **kw)
    assert nmf._backend.kernel_names() == nmf._backend.kernel_names(n_bench), nmf._backend.kernel_names()
    e_rel = float(np.max(np.abs(np.array(e_gpu) - e_ref) / np.array(e_ref)))
    w_err, h_err = _err(nmf.W_device, ref.W), _err(nmf.H_device, ref.H)
    print(f'{name} regularised={regularised} {nmf._backend.kernel_names()}: D {e_gpu[0]:.6g} -> {e_gpu[-1]:.6g}, '
          f'trajectory rel {e_rel:.2e}, W {w_err:.2e}, H {h_err:.2e}')
    assert e_gpu[-1] < e_gpu[0]
    assert e_rel <= 1e-4 and w_err <= 1e-3 and h_err <= 1e-3


def test_kl_minibatch_schedules_vs_reference():
    """All five schedules against the reference's (float64: summation order only); Cyclic_MU equals the full batch."""
    from tnmf_b200 import MiniBatchAlgorithm, TransformInvariantNMF
    rng = np.random.default_rng(12)
    V = rng.random((7, 2, 20, 24))
    V[V < 0.05] = 0
    kw = dict(sparsity_H=0.1, batch_size=3, n_epochs=4, sag_lambda=0.8)
    for alg in MiniBatchAlgorithm:
        np.random.seed(42)
        ref = klr.OracleKL(3, (4, 4)).fit_minibatches(V, algorithm=alg.name.lower(), **kw)
        np.random.seed(42)
        nmf = TransformInvariantNMF(n_atoms=3, atom_shape=(4, 4), divergence='kl')
        nmf.fit_minibatches(V, algorithm=alg, progress_callback=lambda *_: True, **kw)
        assert np.isclose(nmf._energy_function(), ref.energy(), rtol=1e-9), alg
        assert np.abs(nmf.W - ref.W).max() <= 1e-9 * np.abs(ref.W).max(), alg
        assert np.abs(nmf.H - ref.H).max() <= 1e-9 * np.abs(ref.H).max(), alg
    np.random.seed(42)
    full = TransformInvariantNMF(n_atoms=3, atom_shape=(4, 4), divergence='kl')
    full.fit_batch(V, n_iterations=4, sparsity_H=0.1)
    np.random.seed(42)
    cyc = TransformInvariantNMF(n_atoms=3, atom_shape=(4, 4), divergence='kl')
    cyc.fit_minibatches(V, algorithm=MiniBatchAlgorithm.Cyclic_MU, batch_size=7, n_epochs=4, sparsity_H=0.1,
                        progress_callback=lambda *_: True)
    assert np.abs(full.W - cyc.W).max() <= 1e-12 * np.abs(full.W).max()
    assert np.abs(full.H - cyc.H).max() <= 1e-12 * np.abs(full.H).max()
    assert np.isclose(full._energy_function(), cyc._energy_function(), rtol=1e-12)


def test_kl_stream_vs_reference():
    from tnmf_b200 import TransformInvariantNMF
    rng = np.random.default_rng(14)
    V = rng.random((6, 2, 20, 24)).astype(np.float32)
    np.random.seed(3)
    nmf = TransformInvariantNMF(n_atoms=3, atom_shape=(4, 4), divergence='kl')
    nmf.fit(V, subsample_size=3, n_iterations=10)
    np.random.seed(3)
    ref = klr.OracleKL(3, (4, 4)).fit_stream(V.astype(np.float64), subsample_size=3, n_iterations=10)
    assert np.isclose(nmf._energy_function(), ref.energy(), rtol=1e-4)
    assert np.abs(nmf.W - ref.W).max() <= 1e-3 * np.abs(ref.W).max()


@pytest.mark.parametrize('kw', [dict(), dict(sparsity_H=0.05, inhibition_strength=0.1, cross_atom_inhibition_strength=0.05),
                                dict(update_W=False), dict(update_H=False)])
def test_kl_graph_replay_equals_eager_launches(kw):
    from tnmf_b200 import TransformInvariantNMF
    rng = np.random.default_rng(77)
    V = rng.random((6, 3, 40, 56)).astype(np.float32)
    out = {}
    for graph in (False, True):
        nmf = TransformInvariantNMF(n_atoms=16, atom_shape=(7, 7), backend='b200', cuda_graph=graph, divergence='kl')
        for seed in (5, 6):
            np.random.seed(seed)
            nmf.fit(V, n_iterations=7, **kw)
        out[graph] = (nmf.W.copy(), nmf.H.copy(), nmf._energy_function())
    assert np.array_equal(out[False][0], out[True][0])
    assert np.array_equal(out[False][1], out[True][1])
    assert out[False][2] == out[True][2]


@pytest.mark.parametrize('graph', (False, True))
def test_kl_energy_callback_reuses_the_quotient(graph):
    """An energy read in every iteration leaves the quotient in the R buffer; the next H update opens with it (no third
    reconstruction, no second quotient), and the results are bitwise those of a fit without callback."""
    from tnmf_b200 import TransformInvariantNMF, _lib
    rng = np.random.default_rng(78)
    V = rng.random((5, 3, 40, 56)).astype(np.float32)
    energies, launches, foreign = [], {}, [0]

    def callback(nmf, iteration):
        energies.append(nmf._energy_function())
        if iteration == 4:                  # a Frobenius call writes the R buffer: the next KL H update must not trust it
            before = nmf._backend.launches
            nmf._backend.reconstruction_gradient_H(nmf._V, nmf._W, nmf._H)
            foreign[0] = nmf._backend.launches - before
        return True

    out = {}
    for cb in (None, callback):
        nmf = TransformInvariantNMF(n_atoms=16, atom_shape=(7, 7), backend='b200', cuda_graph=graph, divergence='kl')
        np.random.seed(9)
        before = nmf._backend.launches
        nmf.fit(V, n_iterations=8, progress_callback=cb)
        launches[cb is not None] = nmf._backend.launches - before
        out[cb is not None] = (nmf.W.copy(), nmf.H.copy(), nmf._energy_function())
    assert np.array_equal(out[False][0], out[True][0])
    assert np.array_equal(out[False][1], out[True][1])
    assert out[False][2] == out[True][2] == energies[-1]
    assert all(a > b for a, b in zip(energies, energies[1:]))
    per_recon = nmf._backend._n_launches(nmf._backend._last_h_problem, _lib.OP_RECONSTRUCT)
    # 8 energies (reconstruction + quotient + finishing reduction each) and the foreign call, minus the 6 opening
    # reconstructions and quotients that were skipped (iterations 1-7 except the one after the foreign write)
    assert launches[True] == launches[False] + 8 * (per_recon + 2) + foreign[0] - 6 * (per_recon + 1)


def _profiled_kl_step(rank, shape, out):
    from torch.profiler import ProfilerActivity, profile
    N, C, M, D, A = (3, 3, 16, (64, 64), (11, 11)) if shape == '2d' else (2, 1, 16, (8, 32, 32), (3, 5, 5))
    V, W, H = _data(N, C, M, D, A, 'valid', np.float32, 66)
    be, Wd, Hd = _backend(V, W, H)
    grad = torch.empty((2, *Wd.shape), dtype=Wd.dtype, device=Wd.device)

    def step():
        be.update_H(V, Wd, Hd, divergence='kl')
        be.apply_W_update(Wd, be.gradient_W(V, Wd, Hd, slice(None), grad, divergence='kl'))
        be.energy(V, Wd, Hd, divergence='kl')
    step()
    torch.cuda.synchronize()
    before = be.launches
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        step()
        torch.cuda.synchronize()
    out['names'] = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and 'tnmf' in e.name]
    out['launches'] = be.launches - before


@pytest.mark.parametrize('shape', ['2d', '3d'])
def test_kl_profiled_launches_equal_the_count(shape):
    """The profiled KL step runs in a process of its own: after earlier profiler sessions in a process, a later session
    there can miss kernel records, and tests/test_gpu_volumetric.py counts launches the same way in the test process."""
    import torch.multiprocessing as mp
    with mp.get_context('spawn').Manager() as mgr:
        out = mgr.dict()
        mp.spawn(_profiled_kl_step, args=(shape, out), nprocs=1, join=True)
        names, launches = list(out['names']), out['launches']
    assert sum('kl_quotient_kernel' in n for n in names) == 3, names
    assert sum('kl_finish_kernel' in n for n in names) == 1, names
    assert len(names) == launches, names


# ---------------------------------------------------------------------------------------------------------
# two ranks (gloo, both on cuda:0), peer exchange off (gloo) : the all-reduce of the stacked [neg; pos]
# ---------------------------------------------------------------------------------------------------------
def _free_port():
    import socket
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        return s.getsockname()[1]


def _rank_main(rank, world, port, V, kw_fit, out):
    import torch.distributed as dist
    from tnmf_b200 import TransformInvariantNMF
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    torch.cuda.set_device(0)
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        np.random.seed(21)
        nmf = TransformInvariantNMF(n_atoms=6, atom_shape=(5, 4), backend='b200', distributed=True, divergence='kl')
        energies = []
        nmf.fit(V, progress_callback=lambda m, i: energies.append(m._energy_function()) or True, **kw_fit)
        w0 = nmf.W_device.clone()
        dist.broadcast(w0, 0)
        assert torch.equal(w0, nmf.W_device)
        out[rank] = (nmf.W, nmf.H, energies)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize('dtype', [np.float64, np.float32])
def test_two_rank_kl_fit_equals_single_gpu(dtype):
    import torch.multiprocessing as mp
    from tnmf_b200 import TransformInvariantNMF
    from tnmf_b200.distributed import shard_bounds
    rng = np.random.default_rng(3)
    V = rng.random((5, 2, 24, 20)).astype(dtype)
    kw_fit = dict(n_iterations=10, sparsity_H=0.05)
    np.random.seed(21)
    one = TransformInvariantNMF(n_atoms=6, atom_shape=(5, 4), backend='b200', distributed=False, divergence='kl')
    e_one = []
    one.fit(V, progress_callback=lambda m, i: e_one.append(m._energy_function()) or True, **kw_fit)
    world = 2
    with mp.get_context('spawn').Manager() as mgr:
        out = mgr.dict()
        mp.spawn(_rank_main, args=(world, _free_port(), V, kw_fit, out), nprocs=world, join=True)
        results = [out[r] for r in range(world)]
    tol = 1e-9 if dtype == np.float64 else 1e-4
    for rank, (W, H, energies) in enumerate(results):
        lo, hi = shard_bounds(V.shape[0], world, rank)
        assert np.allclose(energies, e_one, rtol=tol)
        assert np.abs(W - one.W).max() <= tol * np.abs(one.W).max()
        assert np.abs(H - one.H[lo:hi]).max() <= tol * np.abs(one.H).max()
