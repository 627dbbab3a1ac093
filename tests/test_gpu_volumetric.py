"""
3-D (volumetric) problems on the plane mode of the tensor-memory kernels (DESIGN.md §3.10), on the GPU, against the
float64 oracle.  Tolerances as in tests/test_gpu_parity.py: single float32 operations within 2e-5 of max|ref|, fits
within 1e-4 (energy, relative) and 1e-3 of max|ref| (W, H).
"""
import numpy as np
import pytest
import torch

from oracle import tnmf_oracle as orc

pytestmark = pytest.mark.gpu

TC3 = {'reconstruct': 'recon_os3_kernel', 'update_h': 'hupd_ts3_kernel', 'gradient_w': 'gradw_ns3_kernel'}
GENERIC_RECON = dict(TC3, reconstruct='generic_reconstruct_kernel')

CASES = [
    # N, C, M, D, A, path, expected kernels
    (3, 2, 11, (3, 13, 11), (3, 3, 3), 'auto', TC3),          # A_z = D_z: the plane predicate fires at both ends
    (2, 3, 9, (5, 12, 9), (2, 3, 3), 'auto', GENERIC_RECON),  # three channels: recon_os takes C <= 2
    (2, 2, 8, (4, 10, 17), (1, 5, 5), 'auto', TC3),           # A_z = 1
    (4, 1, 5, (3, 9, 13), (2, 4, 3), 'tc', TC3),              # few atoms, forced; D_z = 3
    (2, 1, 19, (6, 11, 10), (4, 3, 7), 'auto', TC3),          # two atom blocks of the H update, three of the W gradient
]


def _backend(V, W, H, path='auto'):
    from tnmf_b200 import B200_Backend
    be = B200_Backend(reconstruction_mode='valid', kernel_path=path)
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


def _data(N, C, M, D, A, seed):
    rng = np.random.default_rng(seed)
    V = rng.random((N, C) + D).astype(np.float32)
    W = rng.random((M, C) + A).astype(np.float32)
    H = rng.random((N, M) + orc.transform_shape('valid', D, A)).astype(np.float32)
    return V, W, H


@pytest.mark.parametrize('case', range(len(CASES)))
def test_single_operations_vs_oracle(case):
    N, C, M, D, A, path, expect = CASES[case]
    V, W, H = _data(N, C, M, D, A, 900 + case)
    V64, W64, H64 = V.astype(np.float64), W.astype(np.float64), H.astype(np.float64)
    be, Wd, Hd = _backend(V, W, H, path)
    tol = 2e-5
    for s in (slice(None), slice(1, N)):                    # the whole batch and an H minibatch slice
        Hs64, Vs64 = H64[s], V64[s]
        _close(be.reconstruct(Wd, Hd[s]), orc.reconstruct(W64, Hs64), tol)
        assert be.kernel_names() == expect, be.kernel_names()
        neg, pos = be.reconstruction_gradient_H(V, Wd, Hd, s)
        rn, rp = orc.reconstruction_gradient_H(Vs64, W64, Hs64)
        _close(neg, rn, tol)
        _close(pos, rp, tol)
        neg, pos = be.reconstruction_gradient_W(V, Wd, Hd, s)
        rn, rp = orc.reconstruction_gradient_W(Vs64, W64, Hs64)
        _close(neg, rn, tol)
        _close(pos, rp, tol)
        assert be.kernel_names() == expect, be.kernel_names()
    e = be.reconstruction_energy(V, Wd, Hd)                 # energy without a caller's R: R scratch in the workspace
    assert np.isclose(e, orc.reconstruction_energy(V64, W64, H64), rtol=2e-5)
    assert be.kernel_names() == expect
    # the strided single-atom view (one atom: the generic kernels unless forced)
    _close(be.partial_reconstruct(Wd, Hd, 1), orc.reconstruct(W64[1:2], H64[:, 1:2]), tol)


def _fit_pair(ref, V, seed, path='auto', fused=True, inhibition_range=None, **kw):
    """The facade and the oracle from the same seeded start (both draw H, then W, from numpy's global generator)."""
    from tnmf_b200 import TransformInvariantNMF
    ref_traj, traj = [], []
    np.random.seed(seed)
    ref.fit_batch(V, n_iterations=20, progress_callback=lambda m, i: ref_traj.append(m.energy()) or True, **kw)
    np.random.seed(seed)
    nmf = TransformInvariantNMF(n_atoms=ref.n_atoms, atom_shape=ref.atom_shape, inhibition_range=inhibition_range,
                                kernel_path=path, fused=fused)
    nmf.fit(V.astype(np.float32), n_iterations=20,
            progress_callback=lambda m, i: traj.append(m._energy_function()) or True, **kw)
    assert np.allclose(traj, ref_traj, rtol=1e-4), (traj[-1], ref_traj[-1])
    assert np.abs(nmf.W - ref.W).max() <= 1e-3 * np.abs(ref.W).max()
    assert np.abs(nmf.H - ref.H).max() <= 1e-3 * np.abs(ref.H).max()
    return nmf


def test_benchmark_geometry_fit_vs_fft_oracle():
    """The per-sample geometry of tools/bench_3d.py (1 x 64^3, 8 atoms of 7^3), one sample, 20 iterations."""
    V = np.random.default_rng(31).random((1, 1, 64, 64, 64))
    nmf = _fit_pair(orc.OracleNMF_FFT(8, (7, 7, 7)), V, 5)
    be = nmf._backend
    assert be.kernel_names() == TC3, be.kernel_names()
    assert be.kernel_names(1) == be.kernel_names(16) == TC3


@pytest.mark.parametrize('fused', [True, False])
def test_regularised_fit_vs_oracle(fused):
    N, C, M, D, A = 3, 2, 10, (4, 12, 13), (2, 3, 4)
    V = np.random.default_rng(77).random((N, C) + D)
    nmf = _fit_pair(orc.OracleNMF(M, A, inhibition_range=(1, 2, 1)), V, 3, fused=fused, inhibition_range=(1, 2, 1),
                    sparsity_H=0.1, inhibition_strength=0.2, cross_atom_inhibition_strength=0.3)
    assert nmf._backend.kernel_names() == TC3, nmf._backend.kernel_names()


def test_cyclic_minibatches_equal_the_full_batch():
    """Cyclic_MU accumulates the minibatch gradients and updates W once per epoch: the full-batch iteration
    (tests/test_minibatch.py)."""
    from tnmf_b200 import MiniBatchAlgorithm, TransformInvariantNMF
    V = np.random.default_rng(12).random((5, 1, 4, 10, 11)).astype(np.float32)
    out = []
    for mb in (False, True):
        np.random.seed(8)
        nmf = TransformInvariantNMF(n_atoms=9, atom_shape=(2, 3, 3))
        if mb:
            nmf.fit_minibatches(V, algorithm=MiniBatchAlgorithm.Cyclic_MU, batch_size=2, n_epochs=5, sparsity_H=0.1)
        else:
            nmf.fit_batch(V, n_iterations=5, sparsity_H=0.1)
        assert nmf._backend.kernel_names(5) == TC3
        out.append((nmf.W, nmf.H, nmf._energy_function()))
    assert np.abs(out[0][0] - out[1][0]).max() <= 1e-4 * np.abs(out[0][0]).max()
    assert np.abs(out[0][1] - out[1][1]).max() <= 1e-4 * np.abs(out[0][1]).max()
    assert np.isclose(out[0][2], out[1][2], rtol=1e-5)


def _mu_step(be, V, Wd, Hd, grad):
    be.update_H(V, Wd, Hd)
    be.apply_W_update(Wd, be.gradient_W(V, Wd, Hd, slice(None), grad))


def test_graph_replay_and_reruns_are_bitwise_identical():
    N, C, M, D, A = 2, 2, 11, (3, 13, 11), (3, 3, 3)
    V, W, H = _data(N, C, M, D, A, 55)
    results = []
    for graph in (False, False, True):
        be, Wd, Hd = _backend(V, W, H)
        grad = torch.empty((2, *Wd.shape), dtype=Wd.dtype, device=Wd.device)
        _mu_step(be, V, Wd, Hd, grad)                       # warm-up: buffers, workspace, modules
        Wd.copy_(torch.from_numpy(W))
        Hd.copy_(torch.from_numpy(H))
        torch.cuda.synchronize()
        if graph:
            g = torch.cuda.CUDAGraph()
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s), torch.cuda.graph(g, stream=s):
                _mu_step(be, V, Wd, Hd, grad)
            torch.cuda.current_stream().wait_stream(s)
            Wd.copy_(torch.from_numpy(W))
            Hd.copy_(torch.from_numpy(H))
            for _ in range(3):
                g.replay()
        else:
            for _ in range(3):
                _mu_step(be, V, Wd, Hd, grad)
        torch.cuda.synchronize()
        assert be.kernel_names() == TC3
        results.append((Wd.cpu().numpy().copy(), Hd.cpu().numpy().copy()))
    for w, h in results[1:]:
        assert np.array_equal(w, results[0][0]) and np.array_equal(h, results[0][1])


def test_profiled_launches_equal_the_launch_count():
    from torch.profiler import ProfilerActivity, profile
    N, C, M, D, A = 2, 2, 20, (5, 12, 9), (3, 3, 3)
    V, W, H = _data(N, C, M, D, A, 66)
    be, Wd, Hd = _backend(V, W, H)
    grad = torch.empty((2, *Wd.shape), dtype=Wd.dtype, device=Wd.device)
    _mu_step(be, V, Wd, Hd, grad)
    be.energy(V, Wd, Hd)
    torch.cuda.synchronize()
    before = be.launches
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        _mu_step(be, V, Wd, Hd, grad)
        be.energy(V, Wd, Hd)
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and 'tnmf' in e.name]
    # three reconstructions of 3 atom planes, the H update in 2 atom blocks, the W gradient in 3 planes x 3 atom blocks
    assert sum('3_kernel' in n for n in names) == 3 * 3 + 2 + 9, names
    assert len(names) == be.launches - before, names
