"""
GPU parity tests (run on the B200 box with `-m gpu`): the CUDA path, called through the C-ABI
(tnmf_b200._lib -> libtnmf_b200.so), against
  * the golden fixtures generated from the unmodified reference (tests/golden/make_golden.py), and
  * the CPU oracle (oracle/tnmf_oracle.py) on the same seeded inputs.

Tolerances (stated per test):
  float64  : the kernels and the reference differ by summation order only -> rtol 1e-9 .. 1e-10
  float32  : energy trajectory within 1e-4 relative, W/H within 1e-3 of max|ref| after 100 iterations
             (BASELINE.json north_star; SURVEY 7 "bit-level order of operations" explains why elementwise
             relative error on H is meaningless), single operations within 2e-5 of max|ref|.
"""
import numpy as np
import pytest
import torch

from oracle import tnmf_oracle as orc

pytestmark = pytest.mark.gpu

MODES = ('valid', 'full', 'circular')
REFERENCE_TEST_1D_ENERGIES = {'valid': 2.34946, 'full': 1.87180, 'circular': 3.13228}   # tnmf/tests/test_1d.py:17-22


def _backend(V, W, H, mode='valid', path='auto', **kw):
    from tnmf_b200 import B200_Backend
    be = B200_Backend(reconstruction_mode=mode, kernel_path=path, **kw)
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


def _paths(dtype, ndim):
    if dtype == np.float32 and ndim <= 2:
        return ('generic', 'tiled')
    return ('generic',)


# ---------------------------------------------------------------------------------------------------------
# single operations against the reference's outputs (all modes, 1-D / 2-D / 3-D)
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('dtype', [np.float64, np.float32])
@pytest.mark.parametrize('mode', MODES)
@pytest.mark.parametrize('case', ['d1', 'd2', 'd3'])
def test_single_operations_vs_reference(case, mode, dtype, golden):
    g = golden('ref_ops')
    k = f'{case}_{mode}_'
    V, W, H = (g[k + n].astype(dtype) for n in 'VWH')
    tol = 1e-10 if dtype == np.float64 else 2e-5
    for path in _paths(dtype, V.ndim - 2):
        be, Wd, Hd = _backend(V, W, H, mode, path)
        assert tuple(Hd.shape[2:]) == orc.transform_shape(mode, V.shape[2:], W.shape[2:])
        _close(be.reconstruct(Wd, Hd), g[k + 'R'], tol)
        neg, pos = be.reconstruction_gradient_H(V, Wd, Hd)
        _close(neg, g[k + 'negH'], tol)
        _close(pos, g[k + 'posH'], tol)
        neg, pos = be.reconstruction_gradient_W(V, Wd, Hd)
        _close(neg, g[k + 'negW'], tol)
        _close(pos, g[k + 'posW'], tol)
        e = be.reconstruction_energy(V, Wd, Hd)
        assert np.isclose(e, g[k + 'E'], rtol=1e-10 if dtype == np.float64 else 1e-5)
        # partial reconstruction: strided single-atom view of H (tnmf/backends/_Backend.py:124-125)
        _close(be.partial_reconstruct(Wd, Hd, 1), orc.reconstruct(W[1:2].astype(np.float64),
                                                                  H[:, 1:2].astype(np.float64), mode), tol)


# ---------------------------------------------------------------------------------------------------------
# the reference's own known-answer test (tnmf/tests/test_1d.py)
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('fused', [True, False])
@pytest.mark.parametrize('mode', MODES)
def test_known_answer_test_1d(mode, fused, golden):
    from tnmf_b200 import TransformInvariantNMF
    g = golden('ref_test_1d')
    np.random.seed(42)
    nmf = TransformInvariantNMF(n_atoms=3, atom_shape=(5,), reconstruction_mode=mode, fused=fused)
    nmf.fit(g['V'], inhibition_strength=0.1, n_iterations=10)
    assert np.isclose(nmf._energy_function(), REFERENCE_TEST_1D_ENERGIES[mode])      # the reference's assertion
    assert np.isclose(nmf._energy_function(), g[f'E_{mode}'], rtol=1e-10)
    assert np.allclose(nmf.W, g[f'W_{mode}'], rtol=1e-9, atol=1e-12)
    assert np.allclose(nmf.H, g[f'H_{mode}'], rtol=1e-9, atol=1e-12)
    assert np.allclose(nmf.R, g[f'R_{mode}'], rtol=1e-9, atol=1e-12)
    assert np.allclose(nmf.W.sum(axis=-1), 1.0)                                     # tnmf/tests/test_1d.py:90-91


# ---------------------------------------------------------------------------------------------------------
# batch fits in 2-D with sparsity / inhibition / cross-atom inhibition, all modes, float64
# ---------------------------------------------------------------------------------------------------------
VARIANTS = {
    'plain': dict(),
    'sparse': dict(sparsity_H=0.1),
    'inhib': dict(inhibition_strength=0.5),
    'cross': dict(cross_atom_inhibition_strength=0.3, sparsity_H=0.05),
    'all': dict(sparsity_H=0.1, inhibition_strength=0.2, cross_atom_inhibition_strength=0.4),
}


@pytest.mark.parametrize('fused', [True, False])
@pytest.mark.parametrize('mode', MODES)
@pytest.mark.parametrize('variant', list(VARIANTS))
def test_batch_fit_2d(mode, variant, fused, golden):
    from tnmf_b200 import TransformInvariantNMF
    g = golden('ref_fit_2d')
    np.random.seed(5)
    nmf = TransformInvariantNMF(n_atoms=4, atom_shape=(5, 3), reconstruction_mode=mode, fused=fused)
    traj = []
    nmf.fit(g['V'], n_iterations=20, progress_callback=lambda m, i: traj.append(m._energy_function()) or True,
            **VARIANTS[variant])
    k = f'{mode}_{variant}_'
    assert np.allclose(traj, g[k + 'E'], rtol=1e-9)
    assert np.allclose(nmf.W, g[k + 'W'], rtol=1e-8, atol=1e-12)
    assert np.allclose(nmf.H, g[k + 'H'], rtol=1e-8, atol=1e-12)


def test_batch_fit_custom_inhibition_range(golden):
    from tnmf_b200 import TransformInvariantNMF
    g = golden('ref_fit_2d')
    np.random.seed(5)
    nmf = TransformInvariantNMF(n_atoms=4, atom_shape=(5, 3), inhibition_range=(2, 1))
    nmf.fit(g['V'], n_iterations=20, inhibition_strength=0.7)
    assert np.isclose(nmf._energy_function(), g['valid_range_E'][-1], rtol=1e-9)
    assert np.allclose(nmf.W, g['valid_range_W'], rtol=1e-8, atol=1e-12)


@pytest.mark.parametrize('path', ['generic', 'tiled', 'auto', 'tc'])
def test_batch_fit_float32_100_iterations(path, golden):
    """north_star tolerance: energy trajectory within 1e-4 relative, W/H within 1e-3 max-relative after 100
    iterations, against the reference numpy backend run in float32 - for every kernel family, the 3xTF32 tensor-core
    H update and W gradient ('tc') included."""
    from tnmf_b200 import TransformInvariantNMF
    g = golden('ref_fit_2d')
    V32 = g['V'].astype(np.float32)
    np.random.seed(5)
    nmf = TransformInvariantNMF(n_atoms=4, atom_shape=(5, 3), kernel_path=path)
    traj = []
    nmf.fit(V32, n_iterations=100, sparsity_H=0.1,
            progress_callback=lambda m, i: traj.append(m._energy_function()) or True)
    assert nmf.W.dtype == np.float32 and nmf.H.dtype == np.float32
    if path == 'tc':
        fam = nmf._backend.kernel_families()
        assert fam['update_h'] == 'tc' and fam['gradient_w'] == 'tc'
    assert np.allclose(traj, g['f32_E'], rtol=1e-4)
    assert np.abs(nmf.W - g['f32_W']).max() <= 1e-3 * np.abs(g['f32_W']).max()
    assert np.abs(nmf.H - g['f32_H']).max() <= 1e-3 * np.abs(g['f32_H']).max()


# ---------------------------------------------------------------------------------------------------------
# minibatch schedules and streams
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('fused', [True, False])
@pytest.mark.parametrize('alg', ['Cyclic_MU', 'ASG_MU', 'GSG_MU', 'ASAG_MU', 'GSAG_MU'])
def test_minibatch_schedules(alg, fused, golden):
    from tnmf_b200 import MiniBatchAlgorithm, TransformInvariantNMF
    g = golden('ref_minibatch')
    np.random.seed(42)
    nmf = TransformInvariantNMF(n_atoms=3, atom_shape=(4, 4), fused=fused)
    nmf.fit_minibatches(g['V'], sparsity_H=0.1, algorithm=MiniBatchAlgorithm[alg], batch_size=3, n_epochs=5,
                        sag_lambda=0.8, progress_callback=lambda *_: True)
    assert np.isclose(nmf._energy_function(), g[f'{alg}_E'], rtol=1e-9)
    assert np.allclose(nmf.W, g[f'{alg}_W'], rtol=1e-8, atol=1e-12)
    assert np.allclose(nmf.H, g[f'{alg}_H'], rtol=1e-8, atol=1e-12)


def test_cyclic_equals_full_batch(golden):
    """tnmf/tests/test_minibatch.py:19-20."""
    from tnmf_b200 import TransformInvariantNMF
    g = golden('ref_minibatch')
    np.random.seed(42)
    nmf = TransformInvariantNMF(n_atoms=3, atom_shape=(4, 4))
    nmf.fit_batch(g['V'], sparsity_H=0.1, n_iterations=5)
    assert np.isclose(nmf._energy_function(), g['full_batch_E'], rtol=1e-9)
    assert np.isclose(nmf._energy_function(), g['Cyclic_MU_E'], rtol=1e-9)
    assert np.allclose(nmf.W, g['full_batch_W'], rtol=1e-8)


def test_stream(golden):
    """tnmf/tests/test_stream.py:47-108: array and generator input, with and without max_subsamples."""
    from tnmf_b200 import MiniBatchAlgorithm, TransformInvariantNMF
    g = golden('ref_minibatch')
    np.random.seed(42)
    nmf = TransformInvariantNMF(n_atoms=3, atom_shape=(4, 4))
    nmf.fit(g['V'], subsample_size=3, batch_size=2, n_epochs=3, algorithm=MiniBatchAlgorithm.Cyclic_MU)
    assert np.isclose(nmf._energy_function(), g['stream_E'], rtol=1e-9)
    assert np.allclose(nmf.W, g['stream_W'], rtol=1e-8)
    assert np.allclose(nmf.H, g['stream_H'], rtol=1e-8, atol=1e-12)
    np.random.seed(42)
    nmf = TransformInvariantNMF(n_atoms=3, atom_shape=(4, 4))
    nmf.fit((v for v in g['V']), subsample_size=3, max_subsamples=2, n_iterations=4)
    assert np.isclose(nmf._energy_function(), g['stream2_E'], rtol=1e-9)
    assert np.allclose(nmf.W, g['stream2_W'], rtol=1e-8)


# ---------------------------------------------------------------------------------------------------------
# BASELINE config 1 (the reference's own CPU-runnable case), float64 and float32
# ---------------------------------------------------------------------------------------------------------
def test_cfg1_float64(golden):
    from tnmf_b200 import TransformInvariantNMF
    g = golden('ref_cfg1')
    np.random.seed(42)
    nmf = TransformInvariantNMF(n_atoms=5, atom_shape=(50,))
    traj = []
    nmf.fit(g['V'], n_iterations=100,
            progress_callback=lambda m, i: (traj.append(m._energy_function()) if i % 10 == 9 else None) or True)
    assert np.isclose(traj[-1], 3.808691, rtol=1e-6)                     # SURVEY 8c probe value
    assert np.allclose(traj, g['E'][9::10], rtol=1e-8)
    assert np.allclose(nmf.W, g['W'], rtol=1e-6, atol=1e-10)
    assert np.allclose(nmf.H[:2, :, :64], g['H_head'], rtol=1e-6, atol=1e-10)


def test_cfg1_float32_tiled(golden):
    """Same run in float32 on the tiled kernels: energy within 1e-4 relative, W within 1e-3 of max|W|."""
    from tnmf_b200 import TransformInvariantNMF
    g = golden('ref_cfg1')
    np.random.seed(42)
    nmf = TransformInvariantNMF(n_atoms=5, atom_shape=(50,), kernel_path='tiled')
    traj = []
    nmf.fit(g['V'].astype(np.float32), n_iterations=100,
            progress_callback=lambda m, i: (traj.append(m._energy_function()) if i % 10 == 9 else None) or True)
    assert np.allclose(traj, g['E'][9::10], rtol=1e-4)
    assert np.abs(nmf.W - g['W']).max() <= 1e-3 * np.abs(g['W']).max()


# ---------------------------------------------------------------------------------------------------------
# tiled kernels against the oracle on seeded inputs: shapes that exercise every tile edge
# ---------------------------------------------------------------------------------------------------------
TILED_CASES = [
    # N, C, M, D, A
    (2, 3, 4, (40, 70), (11, 11)),      # cfg2-like atoms, ragged tile edges
    (3, 1, 5, (33, 65), (15, 15)),      # cfg3-like atoms, one past the tile size
    (2, 1, 3, (20, 90), (7, 20)),       # atom wider than the ax-chunk (multi-chunk path)
    (2, 2, 6, (1000,), (50,)),          # cfg1-like 1-D
    (3, 1, 7, (300,), (128,)),          # cfg4-like 1-D atom
    (1, 5, 2, (9, 9), (3, 2)),          # more channels than a channel block, even atom width
    (4, 1, 1, (17, 13), (1, 1)),        # single atom of one pixel
    (2, 2, 3, (6, 8), (6, 8)),          # atom as large as the sample ('full': a single activation)
    (1, 1, 2, (70, 300), (5, 64)),      # wide atom, wide sample
]


@pytest.mark.parametrize('mode', MODES)
@pytest.mark.parametrize('case', range(len(TILED_CASES)))
def test_tiled_vs_oracle(case, mode):
    N, C, M, D, A = TILED_CASES[case]
    rng = np.random.default_rng(100 + case)
    V = rng.random((N, C) + D).astype(np.float32)
    W = rng.random((M, C) + A).astype(np.float32)
    H = rng.random((N, M) + orc.transform_shape(mode, D, A)).astype(np.float32)
    V64, W64, H64 = V.astype(np.float64), W.astype(np.float64), H.astype(np.float64)
    be, Wd, Hd = _backend(V, W, H, mode, 'tiled')
    assert be.uses_tiled_kernels()
    tol = 2e-5
    R = orc.reconstruct(W64, H64, mode)
    _close(be.reconstruct(Wd, Hd), R, tol)
    neg, pos = be.reconstruction_gradient_H(V, Wd, Hd)
    rn, rp = orc.reconstruction_gradient_H(V64, W64, H64, mode)
    _close(neg, rn, tol)
    _close(pos, rp, tol)
    neg, pos = be.reconstruction_gradient_W(V, Wd, Hd)
    rn, rp = orc.reconstruction_gradient_W(V64, W64, H64, mode)
    _close(neg, rn, tol)
    _close(pos, rp, tol)
    assert np.isclose(be.reconstruction_energy(V, Wd, Hd), orc.reconstruction_energy(V64, W64, H64, mode), rtol=2e-5)
    # fused update with every epilogue term against the oracle's update
    nmf = orc.OracleNMF(M, A, reconstruction_mode=mode)
    nmf.V, nmf.W, nmf.H = V64, W64.copy(), H64.copy()
    nmf.update_H(slice(None), sparsity=0.1, inhibition=0.2, cross_inhibition=0.3 if M > 1 else 0.0)
    be.update_H(V, Wd, Hd, slice(None), 0.1, 0.2, 0.3 if M > 1 else 0.0, nmf.inhibition_kernels)
    _close(Hd, nmf.H, 5e-5)
    nmf.update_W()
    grad = torch.empty((2, *Wd.shape), dtype=Wd.dtype, device=Wd.device)
    be.apply_W_update(Wd, be.gradient_W(V, Wd, Hd, slice(None), grad))
    _close(Wd, nmf.W, 5e-5)
    assert np.allclose(Wd.sum(dim=tuple(range(2, Wd.dim()))).cpu().numpy(), 1.0, atol=1e-5)


# ---------------------------------------------------------------------------------------------------------
# single-channel 1-D batches run as ONE 2-D image of signal rows (capi.cu rows_view): the 2-D kernel families against
# the oracle and against the 1-D kernels (rows_view=False), whole batches and minibatch slices
# ---------------------------------------------------------------------------------------------------------
ROWS_CASES = [
    # N, M, D, A
    (5, 7, 300, 128),       # cfg4-like atom
    (64, 5, 1000, 50),      # cfg1-like, many rows
    (3, 4, 64, 9),          # short signals
    (2, 3, 130, 5),         # signal length not a multiple of 4: V/R boxes are not TMA-able
    (9, 17, 256, 32),       # more than one atom block
]


@pytest.mark.parametrize('mode', ('valid', 'full'))
@pytest.mark.parametrize('case', range(len(ROWS_CASES)))
def test_rows_view_1d_vs_oracle(case, mode):
    N, M, D, A = ROWS_CASES[case]
    rng = np.random.default_rng(700 + case)
    V = rng.random((N, 1, D)).astype(np.float32)
    W = rng.random((M, 1, A)).astype(np.float32)
    H = rng.random((N, M) + orc.transform_shape(mode, (D,), (A,))).astype(np.float32)
    V64, W64, H64 = V.astype(np.float64), W.astype(np.float64), H.astype(np.float64)
    be, Wd, Hd = _backend(V, W, H, mode, rows_view=True)    # 'auto' takes the view from 2^20 signal elements on
    assert Hd.stride(1) % 4 == 0 and Hd.stride(0) == M * Hd.stride(1)      # padded rows, [n, m, t] order kept
    tol = 2e-5
    for s in (slice(1, N - 1), slice(N - 1, N), slice(None)):
        Hs64, Vs64 = H64[s], V64[s]
        if Hs64.shape[0] == 0:
            continue
        _close(be.reconstruct(Wd, Hd[s]), orc.reconstruct(W64, Hs64, mode), tol)
        neg, pos = be.reconstruction_gradient_H(V, Wd, Hd, s)
        rn, rp = orc.reconstruction_gradient_H(Vs64, W64, Hs64, mode)
        _close(neg, rn, tol)
        _close(pos, rp, tol)
        neg, pos = be.reconstruction_gradient_W(V, Wd, Hd, s)
        rn, rp = orc.reconstruction_gradient_W(Vs64, W64, Hs64, mode)
        _close(neg, rn, tol)
        _close(pos, rp, tol)
    fam = be.kernel_families()              # of the last problem: the whole batch
    if case in (1, 4):              # shapes the persistent TMA kernels plan for (case 0: atom too wide for so short a row)
        assert fam['update_h'] == 'tma', fam
        if mode == 'valid':
            assert fam == {'reconstruct': 'tma', 'update_h': 'tma', 'gradient_w': 'tma'}, fam
    assert np.isclose(be.reconstruction_energy(V, Wd, Hd), orc.reconstruction_energy(V64, W64, H64, mode), rtol=2e-5)
    # fused updates (all epilogue terms) against the oracle, then against the 1-D kernels on the same inputs
    nmf = orc.OracleNMF(M, (A,), reconstruction_mode=mode)
    nmf.V, nmf.W, nmf.H = V64, W64.copy(), H64.copy()
    # (the rows view serves the update without inhibition terms; with them the dense G arrays keep the 1-D kernels)
    for s in (slice(0, 1), slice(1, N)):
        nmf.update_H(s, sparsity=0.1)
        be.update_H(V, Wd, Hd, s, 0.1)
    _close(Hd, nmf.H, 5e-5)
    nmf.update_H(slice(None), sparsity=0.1, inhibition=0.2, cross_inhibition=0.3)
    be.update_H(V, Wd, Hd, slice(None), 0.1, 0.2, 0.3, nmf.inhibition_kernels)
    _close(Hd, nmf.H, 1e-4)
    nmf.update_W()
    grad = torch.empty((2, *Wd.shape), dtype=Wd.dtype, device=Wd.device)
    be.apply_W_update(Wd, be.gradient_W(V, Wd, Hd, slice(None), grad))
    _close(Wd, nmf.W, 5e-5)
    be1, W1, H1 = _backend(V, W, H, mode, rows_view=False)
    for s in (slice(0, 1), slice(1, N)):
        be1.update_H(V, W1, H1, s, 0.1)
    be1.update_H(V, W1, H1, slice(None), 0.1, 0.2, 0.3, nmf.inhibition_kernels)
    assert set(be1.kernel_families().values()) == {'tiled'}
    be1.apply_W_update(W1, be1.gradient_W(V, W1, H1, slice(None), torch.empty_like(grad)))
    _close(Hd, H1.cpu().numpy(), 5e-5)
    _close(Wd, W1.cpu().numpy(), 5e-5)


# ---------------------------------------------------------------------------------------------------------
# persistent TMA kernels against the oracle: 2-D, 'valid' / 'full', sample rows a multiple of 16 bytes
# ---------------------------------------------------------------------------------------------------------
TMA_CASES = [
    # N, C, M, D, A
    (2, 3, 4, (40, 72), (11, 11)),      # cfg2-like atoms, ragged tile edges, padded H rows (82 -> 84)
    (3, 1, 5, (33, 64), (15, 15)),      # cfg3-like atoms
    (2, 1, 3, (20, 88), (7, 20)),       # atom wider than the ax-chunk (multi-chunk path)
    (1, 5, 2, (9, 12), (3, 2)),         # more channels than a channel block, even atom width
    (4, 1, 1, (17, 16), (1, 1)),        # single atom of one pixel
    (2, 2, 3, (6, 8), (6, 8)),          # atom as large as the sample ('full': a single activation)
    (1, 1, 2, (70, 300), (5, 64)),      # wide atom, wide sample
    (3, 3, 16, (64, 64), (11, 11)),     # several atom blocks, several work units per CTA
    (5, 2, 9, (100, 36), (4, 9)),       # unbalanced atom blocks (9 = 3 x 3), tall samples
]


@pytest.mark.parametrize('mode', ('valid', 'full'))
@pytest.mark.parametrize('case', range(len(TMA_CASES)))
def test_tma_vs_oracle(case, mode):
    N, C, M, D, A = TMA_CASES[case]
    rng = np.random.default_rng(200 + case)
    V = rng.random((N, C) + D).astype(np.float32)
    W = rng.random((M, C) + A).astype(np.float32)
    H = rng.random((N, M) + orc.transform_shape(mode, D, A)).astype(np.float32)
    V64, W64, H64 = V.astype(np.float64), W.astype(np.float64), H.astype(np.float64)
    be, Wd, Hd = _backend(V, W, H, mode, 'auto', tensor_cores=False)   # 'auto' without tensor cores: pins the FP32 kernels
    tol = 2e-5
    R = orc.reconstruct(W64, H64, mode)
    _close(be.reconstruct(Wd, Hd), R, tol)
    # TMA boxes must start on a multiple of 4 elements: always possible for the H update (shifted tile origin), for
    # the other two only when off - (A_x - 1) is a multiple of 4 ('valid': always); else the cp.async kernels serve
    h_side = 'tma' if (mode == 'valid' or (A[-1] - 1) % 4 == 0) else 'tiled'
    assert be.kernel_families() == {'reconstruct': h_side, 'update_h': 'tma', 'gradient_w': h_side}
    neg, pos = be.reconstruction_gradient_H(V, Wd, Hd)
    rn, rp = orc.reconstruction_gradient_H(V64, W64, H64, mode)
    _close(neg, rn, tol)
    _close(pos, rp, tol)
    neg, pos = be.reconstruction_gradient_W(V, Wd, Hd)
    rn, rp = orc.reconstruction_gradient_W(V64, W64, H64, mode)
    _close(neg, rn, tol)
    _close(pos, rp, tol)
    assert np.isclose(be.reconstruction_energy(V, Wd, Hd), orc.reconstruction_energy(V64, W64, H64, mode), rtol=2e-5)
    # partial reconstruction: a strided single-atom view of H (tnmf/backends/_Backend.py:124-125)
    _close(be.partial_reconstruct(Wd, Hd, M - 1), orc.reconstruct(W64[M - 1:], H64[:, M - 1:], mode), tol)
    # fused update with every epilogue term against the oracle's update, on a sample slice and on the rest
    nmf = orc.OracleNMF(M, A, reconstruction_mode=mode)
    nmf.V, nmf.W, nmf.H = V64, W64.copy(), H64.copy()
    for s in (slice(0, 1), slice(1, N)):
        nmf.update_H(s, sparsity=0.1, inhibition=0.2, cross_inhibition=0.3 if M > 1 else 0.0)
        be.update_H(V, Wd, Hd, s, 0.1, 0.2, 0.3 if M > 1 else 0.0, nmf.inhibition_kernels)
    _close(Hd, nmf.H, 5e-5)
    nmf.update_W()
    grad = torch.empty((2, *Wd.shape), dtype=Wd.dtype, device=Wd.device)
    be.apply_W_update(Wd, be.gradient_W(V, Wd, Hd, slice(None), grad))
    _close(Wd, nmf.W, 5e-5)
    assert np.allclose(Wd.sum(dim=tuple(range(2, Wd.dim()))).cpu().numpy(), 1.0, atol=1e-5)


# ---------------------------------------------------------------------------------------------------------
# tensor-core (tcgen05, 3xTF32) H gradient / fused H update against the oracle
# ---------------------------------------------------------------------------------------------------------
TC_CASES = [
    # N, C, M, D, A
    (3, 3, 16, (64, 64), (11, 11)),     # cfg2-like: K = 33 -> 40, one full atom block
    (2, 1, 32, (40, 50), (15, 15)),     # cfg3-like: two atom blocks, tallest atom the TMEM ring takes
    (5, 2, 9, (100, 36), (4, 9)),       # partial atom block, tall samples (many ring wrap-arounds)
    (1, 1, 2, (30, 300), (5, 7)),       # K = 7 -> 8, columns of one sample span several tiles
    (2, 3, 5, (20, 24), (3, 3)),
    (4, 1, 1, (17, 16), (1, 1)),        # single atom of one pixel: every source row completes an output row
    (2, 2, 3, (6, 8), (6, 8)),          # atom as large as the sample ('full': a single activation)
    (40, 1, 4, (48, 500), (5, 5)),      # more tiles than SMs: several work units per CTA
    (7, 2, 17, (31, 45), (2, 13)),      # 17 atoms = a full block + 1, even atom height
]


@pytest.mark.parametrize('tmem', (True, False))        # expanded operand in tensor memory / in shared memory (round-1 kernels)
@pytest.mark.parametrize('mode', ('valid', 'full'))
@pytest.mark.parametrize('case', range(len(TC_CASES)))
def test_tc_hupdate_vs_oracle(case, mode, tmem):
    """3xTF32 products carry ~2^-21 relative error against FP32's 2^-24: single operations within 2e-5 of max|ref|
    like the FP32 kernels, the fused update within 5e-5."""
    N, C, M, D, A = TC_CASES[case]
    rng = np.random.default_rng(300 + case)
    V = rng.random((N, C) + D).astype(np.float32)
    W = rng.random((M, C) + A).astype(np.float32)
    H = rng.random((N, M) + orc.transform_shape(mode, D, A)).astype(np.float32)
    V64, W64, H64 = V.astype(np.float64), W.astype(np.float64), H.astype(np.float64)
    be, Wd, Hd = _backend(V, W, H, mode, 'tc', tmem_operand=tmem)
    be.reconstruct(Wd, Hd)
    assert be.kernel_families()['update_h'] == 'tc'
    neg, pos = be.reconstruction_gradient_H(V, Wd, Hd)
    rn, rp = orc.reconstruction_gradient_H(V64, W64, H64, mode)
    _close(neg, rn, 2e-5)
    _close(pos, rp, 2e-5)
    nmf = orc.OracleNMF(M, A, reconstruction_mode=mode)
    nmf.V, nmf.W, nmf.H = V64, W64.copy(), H64.copy()
    for s in (slice(0, 1), slice(1, N)):
        nmf.update_H(s, sparsity=0.1, inhibition=0.2, cross_inhibition=0.3 if M > 1 else 0.0)
        be.update_H(V, Wd, Hd, s, 0.1, 0.2, 0.3 if M > 1 else 0.0, nmf.inhibition_kernels)
    _close(Hd, nmf.H, 5e-5)
    # plain update (no regularisers), twice in a row: the second call reads what the first one wrote
    nmf.update_H(slice(None))
    be.update_H(V, Wd, Hd)
    nmf.update_H(slice(None))
    be.update_H(V, Wd, Hd)
    _close(Hd, nmf.H, 1e-4)


@pytest.mark.parametrize('tmem', (True, False))        # expanded operand in tensor memory / in shared memory (round-1 kernels)
@pytest.mark.parametrize('mode', ('valid', 'full'))
@pytest.mark.parametrize('case', range(len(TC_CASES)))
def test_tc_gradient_w_vs_oracle(case, mode, tmem):
    """Tensor-core W gradient (3xTF32, accumulator resident in TMEM, one partial slice per CTA) against the oracle;
    the sums run over all samples and positions, so the bound is relative to the largest entry."""
    N, C, M, D, A = TC_CASES[case]
    rng = np.random.default_rng(400 + case)
    V = rng.random((N, C) + D).astype(np.float32)
    W = rng.random((M, C) + A).astype(np.float32)
    H = rng.random((N, M) + orc.transform_shape(mode, D, A)).astype(np.float32)
    V64, W64, H64 = V.astype(np.float64), W.astype(np.float64), H.astype(np.float64)
    be, Wd, Hd = _backend(V, W, H, mode, 'tc', tmem_operand=tmem)
    be.reconstruct(Wd, Hd)
    assert be.kernel_families()['gradient_w'] == 'tc'
    neg, pos = be.reconstruction_gradient_W(V, Wd, Hd)
    rn, rp = orc.reconstruction_gradient_W(V64, W64, H64, mode)
    _close(neg, rn, 2e-5)
    _close(pos, rp, 2e-5)
    # on a slice of the samples (minibatch call), and the W update on top of it
    if N > 2:
        neg, pos = be.reconstruction_gradient_W(V, Wd, Hd, slice(1, N - 1))
        rn, rp = orc.reconstruction_gradient_W(V64[1:N - 1], W64, H64[1:N - 1], mode)
        _close(neg, rn, 2e-5)
        _close(pos, rp, 2e-5)
    nmf = orc.OracleNMF(M, A, reconstruction_mode=mode)
    nmf.V, nmf.W, nmf.H = V64, W64.copy(), H64.copy()
    nmf.update_W()
    grad = torch.empty((2, *Wd.shape), dtype=Wd.dtype, device=Wd.device)
    be.apply_W_update(Wd, be.gradient_W(V, Wd, Hd, slice(None), grad))
    _close(Wd, nmf.W, 5e-5)


NS_CASES = [
    # N, C, M, D, A: narrow atoms (C * A_x <= 16) - hi/lo, two source rows and both tensors stacked in the MMA lanes
    (2, 1, 32, (40, 50), (15, 15)),     # cfg3 atoms: four launches of 8 atoms, window of 16 positions
    (3, 1, 9, (31, 70), (4, 9)),        # even atom height (window padded 5 -> 8), odd number of source rows, 9 atoms = 8 + 1
    (2, 2, 8, (25, 40), (7, 8)),        # two channels: all 16 tap lanes of a group in use
    (40, 1, 4, (48, 500), (5, 5)),      # more work than one wave: several segments per CTA, many epochs
    (1, 1, 5, (20, 24), (3, 3)),
    (2, 2, 3, (6, 8), (6, 8)),          # atom as large as the sample
    (2, 1, 20, (64, 64), (19, 16)),     # tallest atom it takes (window of 20), C * A_x = 16
]


@pytest.mark.parametrize('mode', ('valid', 'full'))
@pytest.mark.parametrize('case', range(len(NS_CASES)))
def test_tc_gradient_w_narrow_atoms_vs_oracle(case, mode):
    """gradw_ns_kernel (BASELINE config 3's W gradient) against the oracle: both gradients, a minibatch slice, bitwise
    repeatability, and the W update on top."""
    N, C, M, D, A = NS_CASES[case]
    rng = np.random.default_rng(800 + case)
    V = rng.random((N, C) + D).astype(np.float32)
    W = rng.random((M, C) + A).astype(np.float32)
    H = rng.random((N, M) + orc.transform_shape(mode, D, A)).astype(np.float32)
    V64, W64, H64 = V.astype(np.float64), W.astype(np.float64), H.astype(np.float64)
    be, Wd, Hd = _backend(V, W, H, mode, 'tc')
    neg, pos = be.reconstruction_gradient_W(V, Wd, Hd)
    assert be.kernel_names()['gradient_w'] == 'gradw_ns_kernel', be.kernel_names()
    rn, rp = orc.reconstruction_gradient_W(V64, W64, H64, mode)
    _close(neg, rn, 2e-5)
    _close(pos, rp, 2e-5)
    neg2, pos2 = be.reconstruction_gradient_W(V, Wd, Hd)
    assert torch.equal(neg, neg2) and torch.equal(pos, pos2)
    if N > 2:
        neg, pos = be.reconstruction_gradient_W(V, Wd, Hd, slice(1, N - 1))
        rn, rp = orc.reconstruction_gradient_W(V64[1:N - 1], W64, H64[1:N - 1], mode)
        _close(neg, rn, 2e-5)
        _close(pos, rp, 2e-5)
    nmf = orc.OracleNMF(M, A, reconstruction_mode=mode)
    nmf.V, nmf.W, nmf.H = V64, W64.copy(), H64.copy()
    nmf.update_W()
    grad = torch.empty((2, *Wd.shape), dtype=Wd.dtype, device=Wd.device)
    be.apply_W_update(Wd, be.gradient_W(V, Wd, Hd, slice(None), grad))
    _close(Wd, nmf.W, 5e-5)


TALL_CASES = [
    # N, C, M, D, A  - atoms higher than the 15 rows one launch takes: the W gradient runs in atom-row chunks ('valid')
    (2, 1, 8, (40, 72), (20, 30)),      # two balanced chunks of 10 rows
    (1, 2, 5, (50, 64), (33, 16)),      # three chunks, two channels, partial atom block
    (3, 1, 4, (30, 40), (16, 5)),       # one row more than a launch takes; narrow atom (two stacked source rows)
    (1, 1, 8, (96, 128), (64, 64)),     # cfg5's atoms: all 128 MMA lanes carry taps
    (2, 1, 20, (40, 70), (31, 12)),     # two atom blocks x three chunks, last chunk shorter
]


@pytest.mark.parametrize('case', range(len(TALL_CASES)))
def test_tc_gradient_w_tall_atoms_vs_oracle(case):
    N, C, M, D, A = TALL_CASES[case]
    mode = 'valid'
    rng = np.random.default_rng(450 + case)
    V = rng.random((N, C) + D).astype(np.float32)
    W = rng.random((M, C) + A).astype(np.float32)
    H = rng.random((N, M) + orc.transform_shape(mode, D, A)).astype(np.float32)
    V64, W64, H64 = V.astype(np.float64), W.astype(np.float64), H.astype(np.float64)
    be, Wd, Hd = _backend(V, W, H, mode, 'tc')
    be.reconstruct(Wd, Hd)
    assert be.kernel_families()['gradient_w'] == 'tc'
    rn, rp = orc.reconstruction_gradient_W(V64, W64, H64, mode)
    for _ in range(2):                  # twice: the second call finds the workspace dirty
        neg, pos = be.reconstruction_gradient_W(V, Wd, Hd)
        _close(neg, rn, 2e-5)
        _close(pos, rp, 2e-5)
    if N > 2:
        neg, pos = be.reconstruction_gradient_W(V, Wd, Hd, slice(1, N - 1))
        rn, rp = orc.reconstruction_gradient_W(V64[1:N - 1], W64, H64[1:N - 1], mode)
        _close(neg, rn, 2e-5)
        _close(pos, rp, 2e-5)
    # bitwise run-to-run determinism (fixed-order finish over zero-initialised per-CTA slices)
    a = torch.stack(be.reconstruction_gradient_W(V, Wd, Hd))
    b = torch.stack(be.reconstruction_gradient_W(V, Wd, Hd))
    assert torch.equal(a, b)
    # 'full' mode has no chunked form: the FP32 kernels keep serving it (narrow atoms of up to 19 rows: gradw_ns does)
    be2, W2, H2 = _backend(V, W, rng.random((N, M) + orc.transform_shape('full', D, A)).astype(np.float32), 'full', 'tc')
    be2.reconstruct(W2, H2)
    assert be2.kernel_families()['gradient_w'] != 'tc' or be2.kernel_names()['gradient_w'] == 'gradw_ns_kernel'


@pytest.mark.parametrize('tmem', (True, False))        # expanded operand in tensor memory / in shared memory (round-1 kernels)
@pytest.mark.parametrize('mode', ('valid', 'full'))
@pytest.mark.parametrize('case', range(len(TC_CASES)))
def test_tc_reconstruct_vs_oracle(case, mode, tmem):
    """Tensor-core reconstruction (input-stationary, shifted-operand MMAs, register ring of output rows) and its fused
    energy against the oracle, plus the strided single-atom view of partial_reconstruct."""
    N, C, M, D, A = TC_CASES[case]
    rng = np.random.default_rng(500 + case)
    V = rng.random((N, C) + D).astype(np.float32)
    W = rng.random((M, C) + A).astype(np.float32)
    H = rng.random((N, M) + orc.transform_shape(mode, D, A)).astype(np.float32)
    V64, W64, H64 = V.astype(np.float64), W.astype(np.float64), H.astype(np.float64)
    be, Wd, Hd = _backend(V, W, H, mode, 'tc', tmem_operand=tmem)
    R = be.reconstruct(Wd, Hd)
    assert be.kernel_families()['reconstruct'] == 'tc'
    ref = orc.reconstruct(W64, H64, mode)
    _close(R, ref, 2e-5)
    assert np.isclose(be.reconstruction_energy(V, Wd, Hd), orc.reconstruction_energy(V64, W64, H64, mode), rtol=2e-5)
    if N > 2:                                   # a slice of the samples (minibatch call)
        _close(be.reconstruct(Wd, Hd[1:N - 1]), ref[1:N - 1], 2e-5)
    _close(be.partial_reconstruct(Wd, Hd, M - 1), orc.reconstruct(W64[M - 1:], H64[:, M - 1:], mode), 2e-5)


OS_CASES = [
    # N, C, M, D, A: narrow atoms, many atoms - the activation-row ring of recon_ts does not fit tensor memory
    (2, 1, 32, (40, 50), (15, 15)),     # cfg3 atoms: 16 accumulator slots, window of 15, four operand stages
    (3, 1, 24, (100, 37), (9, 9)),      # tall samples: the accumulator ring wraps many times; 24 atoms = 3 K steps
    (2, 2, 32, (30, 70), (8, 7)),       # two channels in one 16-column slot
    (40, 1, 17, (20, 130), (15, 3)),    # more work units than SMs; 17 atoms padded to 24
    (2, 2, 30, (64, 40), (7, 12)),      # 32-column slots: ring of 10, three stages
    (1, 1, 32, (15, 15), (15, 15)),     # atom as large as the sample ('full': one activation feeds every output row)
    (160, 1, 32, (16, 128), (15, 15)),  # 200 tiles, 22 rows per CTA: a CTA's range spans whole tiles (up to 3 segments);
                                        # 'full': a segment's last source row completes 10 rows, the next opens 15
]


@pytest.mark.parametrize('mode', ('valid', 'full'))
@pytest.mark.parametrize('case', range(len(OS_CASES)))
def test_tc_reconstruct_narrow_atoms_vs_oracle(case, mode):
    """recon_os_kernel (source-row stationary, output rows as a ring of accumulators in tensor memory; BASELINE config 3's
    reconstruction) against the oracle: R, the fused energy, a minibatch slice, bitwise repeatability (one issuing warp:
    the truncating tensor-core accumulation runs in program order)."""
    N, C, M, D, A = OS_CASES[case]
    rng = np.random.default_rng(700 + case)
    V = rng.random((N, C) + D).astype(np.float32)
    W = rng.random((M, C) + A).astype(np.float32)
    H = rng.random((N, M) + orc.transform_shape(mode, D, A)).astype(np.float32)
    V64, W64, H64 = V.astype(np.float64), W.astype(np.float64), H.astype(np.float64)
    be, Wd, Hd = _backend(V, W, H, mode, 'tc')
    R = be.reconstruct(Wd, Hd)
    assert be.kernel_names()['reconstruct'] == 'recon_os_kernel', be.kernel_names()
    ref = orc.reconstruct(W64, H64, mode)
    _close(R, ref, 2e-5)
    assert torch.equal(be.reconstruct(Wd, Hd), R)
    assert np.isclose(be.reconstruction_energy(V, Wd, Hd), orc.reconstruction_energy(V64, W64, H64, mode), rtol=2e-5)
    if N > 2:
        _close(be.reconstruct(Wd, Hd[1:N - 1]), ref[1:N - 1], 2e-5)
    # 'auto' takes the same kernel for these shapes when the batch fills the tiles
    be2, Wd2, Hd2 = _backend(V, W, H, mode, 'auto')
    nu, km = C * A[1], (M + 7) // 8 * 8
    useful = nu / ((nu + 15) // 16 * 16) * M / km * (128 - (A[1] - 1)) / 128      # share of every MMA that is real work
    if N * D[1] >= 128 and A[0] >= 3 and useful >= 0.5:
        _close(be2.reconstruct(Wd2, Hd2), ref, 2e-5)
        assert be2.kernel_names()['reconstruct'] == 'recon_os_kernel', be2.kernel_names()


@pytest.mark.parametrize('seed', range(16))
def test_tc_kernels_vs_generic_on_random_shapes(seed):
    """Randomly drawn supported shapes (ragged tiles, rows far beyond one trip round the TMEM / activation rings, atom
    counts off the blocks of 16, both modes): the tensor-core kernels against the one-thread-per-output generic kernels
    on the same device tensors."""
    rng = np.random.default_rng(9000 + seed)
    C = int(rng.integers(1, 4))
    AX = int(rng.integers(1, 64 // C // 2 + 1))
    AY = int(rng.integers(1, 16))
    M = int(rng.integers(1, 40))
    N = int(rng.integers(1, 6))
    D = (int(rng.integers(AY, AY + 90)), int(rng.integers(AX, AX + 150)))
    mode = 'valid' if seed % 2 == 0 else 'full'
    A = (AY, AX)
    V = rng.random((N, C) + D).astype(np.float32)
    W = rng.random((M, C) + A).astype(np.float32)
    H = rng.random((N, M) + orc.transform_shape(mode, D, A)).astype(np.float32)
    out = {}
    for path in ('generic', 'tc'):
        be, Wd, Hd = _backend(V, W, H, mode, path)
        R = be.reconstruct(Wd, Hd)
        if path == 'tc':
            fam = be.kernel_families()
            assert fam['update_h'] == 'tc' and fam['gradient_w'] == 'tc', (fam, C, A, M)
        nh, ph = be.reconstruction_gradient_H(V, Wd, Hd)
        nw, pw = be.reconstruction_gradient_W(V, Wd, Hd)
        be.update_H(V, Wd, Hd, slice(None), 0.05)
        out[path] = [t.cpu().numpy().astype(np.float64) for t in (nh, ph, nw, pw, Hd, R)]
    for got, ref, tol in zip(out['tc'], out['generic'], (2e-5, 2e-5, 2e-5, 2e-5, 1e-4, 2e-5)):
        _close(got, ref, tol)


@pytest.mark.parametrize('path', ['tc', 'auto'])
@pytest.mark.parametrize('mode', ('valid', 'full'))
def test_no_out_of_bounds_access_nan_guards(mode, path):
    """V and H live inside larger buffers whose surroundings are NaN (compute-sanitizer is not available on the GPU
    pool): an out-of-bounds read poisons the results, an out-of-bounds write destroys a guard.  Shapes chosen so that
    tiles are ragged in every direction and the last column tile is mostly empty."""
    N, C, M, D, A = 3, 3, 16, (37, 70), (11, 11)
    rng = np.random.default_rng(31)
    T = orc.transform_shape(mode, D, A)
    pitch = (T[1] + 3) // 4 * 4
    guard = 4096
    dev = torch.device('cuda')
    Vbig = torch.full((guard + N * C * D[0] * D[1] + guard,), float('nan'), device=dev)
    V = Vbig[guard:guard + N * C * D[0] * D[1]].view(N, C, *D)
    V.copy_(torch.from_numpy(rng.random((N, C) + D).astype(np.float32)))
    Hbig = torch.full((guard + N * M * T[0] * pitch + guard,), float('nan'), device=dev)
    Hpad = Hbig[guard:guard + N * M * T[0] * pitch].view(N, M, T[0], pitch)
    H = Hpad[..., :T[1]]
    H.copy_(torch.from_numpy(rng.random((N, M) + T).astype(np.float32)))
    W = rng.random((M, C) + A).astype(np.float32)
    from tnmf_b200 import B200_Backend
    be = B200_Backend(reconstruction_mode=mode, kernel_path=path)
    state = np.random.get_state()
    Wd, _ = be.initialize(V, A, M, None, (-2, -1))
    np.random.set_state(state)
    Wd.copy_(torch.from_numpy(W))
    V64, W64 = V.cpu().numpy().astype(np.float64), W.astype(np.float64)
    H64 = H.cpu().numpy().astype(np.float64)
    neg, pos = be.reconstruction_gradient_H(V, Wd, H)
    rn, rp = orc.reconstruction_gradient_H(V64, W64, H64, mode)
    _close(neg, rn, 2e-5)
    _close(pos, rp, 2e-5)
    neg, pos = be.reconstruction_gradient_W(V, Wd, H)
    rn, rp = orc.reconstruction_gradient_W(V64, W64, H64, mode)
    _close(neg, rn, 2e-5)
    _close(pos, rp, 2e-5)
    assert np.isclose(be.reconstruction_energy(V, Wd, H), orc.reconstruction_energy(V64, W64, H64, mode), rtol=2e-5)
    be.update_H(V, Wd, H)
    nmf = orc.OracleNMF(M, A, reconstruction_mode=mode)
    nmf.V, nmf.W, nmf.H = V64, W64.copy(), H64.copy()
    nmf.update_H(slice(None))
    _close(H, nmf.H, 1e-4)
    torch.cuda.synchronize()
    assert bool(torch.isnan(Hbig[:guard]).all()) and bool(torch.isnan(Hbig[-guard:]).all())
    assert bool(torch.isnan(Vbig[:guard]).all()) and bool(torch.isnan(Vbig[-guard:]).all())
    if pitch > T[1]:
        assert bool(torch.isnan(Hpad[..., T[1]:]).all())           # the pitch padding of every row is never written


@pytest.mark.parametrize('kw', [dict(), dict(sparsity_H=0.05, inhibition_strength=0.1, cross_atom_inhibition_strength=0.05),
                                dict(update_W=False), dict(update_H=False)])
def test_cuda_graph_replay_equals_eager_launches(kw):
    """fit_batch replays the iteration from CUDA graphs after one eager iteration; the results must be bit-identical to
    launching every kernel eagerly, for every combination of updates and regularisers, and across repeated fits (which
    reuse the H storage and re-capture)."""
    from tnmf_b200 import TransformInvariantNMF
    rng = np.random.default_rng(77)
    V = rng.random((6, 3, 40, 56)).astype(np.float32)
    out = {}
    for graph in (False, True):
        nmf = TransformInvariantNMF(n_atoms=16, atom_shape=(7, 7), backend='b200', cuda_graph=graph)
        for seed in (5, 6):                 # the second fit re-initialises into the same H storage
            np.random.seed(seed)
            nmf.fit(V, n_iterations=7, **kw)
        out[graph] = (nmf.W.copy(), nmf.H.copy(), nmf._energy_function())
    assert np.array_equal(out[False][0], out[True][0])
    assert np.array_equal(out[False][1], out[True][1])
    assert out[False][2] == out[True][2]


@pytest.mark.parametrize('graph', (False, True))
def test_energy_callback_reuses_the_reconstruction(graph):
    """A callback that reads the energy in every iteration (what the reference's INFO log line does,
    tnmf/TransformInvariantNMF.py:346) leaves the reconstruction in the backend's R buffer and the next H update opens
    with it: two reconstruction launches per iteration instead of three, results bit-identical to a fit without callback,
    energies equal to a fresh evaluation."""
    from tnmf_b200 import TransformInvariantNMF
    rng = np.random.default_rng(78)
    V = rng.random((5, 3, 40, 56)).astype(np.float32)
    energies, launches, foreign = [], {}, [0]

    def callback(nmf, iteration):
        energies.append(nmf._energy_function())
        if iteration == 4:                  # something else writes the R buffer: the next H update must not trust it
            before = nmf._backend.launches
            nmf._backend.reconstruction_gradient_H(nmf._V, nmf._W, nmf._H)
            foreign[0] = nmf._backend.launches - before
        return True

    out = {}
    for cb in (None, callback):
        nmf = TransformInvariantNMF(n_atoms=16, atom_shape=(7, 7), backend='b200', cuda_graph=graph)
        np.random.seed(9)
        before = nmf._backend.launches
        nmf.fit(V, n_iterations=8, progress_callback=cb)
        launches[cb is not None] = nmf._backend.launches - before
        out[cb is not None] = (nmf.W.copy(), nmf.H.copy(), nmf._energy_function())
    assert np.array_equal(out[False][0], out[True][0])
    assert np.array_equal(out[False][1], out[True][1])
    assert out[False][2] == out[True][2] == energies[-1]
    assert all(a > b for a, b in zip(energies, energies[1:]))
    from tnmf_b200 import _lib
    per_recon = nmf._backend._n_launches(nmf._backend._last_h_problem, _lib.OP_RECONSTRUCT)
    # 8 energy evaluations (reconstruction + finishing reduction each) and the foreign call of iteration 4, minus the 6
    # opening reconstructions that were skipped (iterations 1-7 except the one after the foreign write)
    assert launches[True] == launches[False] + 8 * (per_recon + 1) + foreign[0] - 6 * per_recon


@pytest.mark.parametrize('dtype', [torch.float32, torch.float64])
def test_allreduce_update_w_kernel_against_plain_update(dtype):
    """tnmf_allreduce_update_w (the W-gradient sum over ranks fused with the W update, NVLink peer memory) in ONE process:
    the exchange buffer of 'rank 1' is a second buffer on the same device and its contribution is planted by hand (slot
    [parity][1] of rank 0's buffer, flags = epoch) before rank 0's kernel runs.  Three consecutive calls (both slot
    parities, the epoch counter) must equal tnmf_update_w on the summed gradient - bitwise: both round the double sum of
    two floats once."""
    import ctypes
    from tnmf_b200 import B200_Backend, _lib
    rng = np.random.default_rng(3)
    M, C, A = 5, 3, (7, 6)
    V = rng.random((2, C, 20, 24)).astype(np.float32 if dtype == torch.float32 else np.float64)
    be = B200_Backend()
    W, _ = be.initialize(V, A, M, None, (-2, -1))
    lib, p = be._lib, be._problem(0, M)
    world, pairs, avol = 2, M * C, A[0] * A[1]
    count = pairs * avol
    nbytes = int(lib.tnmf_peer_buffer_bytes(ctypes.byref(p), world))
    esize = 4 if dtype == torch.float32 else 8
    data_bytes = 2 * world * 2 * count * esize
    flags_off = (data_bytes + 127) // 128 * 128
    assert nbytes == flags_off + world * pairs * 4
    bufs = [torch.zeros(nbytes, dtype=torch.uint8, device=be.device) for _ in range(world)]
    pw = _lib.PeerWorld()
    pw.world, pw.rank = world, 0
    for r in range(world):
        pw.buffers[r] = bufs[r].data_ptr()
    state = torch.zeros(2, dtype=torch.int32, device=be.device)
    data0 = bufs[0][:data_bytes].view(dtype).view(2, world, 2 * count)
    flags0 = bufs[0][flags_off:].view(torch.int32).view(world, pairs)
    W_ref = W.clone()
    for call in range(1, 4):
        g0 = torch.rand((2, M, C, *A), dtype=dtype, device=be.device) + 0.1
        g1 = torch.rand((2, M, C, *A), dtype=dtype, device=be.device) + 0.1
        data0[call & 1, 1] = g1.reshape(-1)             # what rank 1's kernel would have pushed
        flags0[1] = call
        _lib.check(lib.tnmf_allreduce_update_w(ctypes.byref(p), W.data_ptr(), g0.data_ptr(), ctypes.byref(pw),
                                               state.data_ptr(), 1e-9, None), 'allreduce_update_w')
        total = (g0.double() + g1.double()).to(dtype)
        be.apply_W_update(W_ref, total, 1e-9)
        torch.cuda.synchronize()
        assert int(state[0].item()) == call and int(state[1].item()) == 0
        assert torch.equal(W, W_ref), f'call {call}'
        # rank 0 pushed its own gradient into slot [parity][0] of BOTH buffers and raised its flags everywhere
        for b in bufs:
            assert torch.equal(b[:data_bytes].view(dtype).view(2, world, 2 * count)[call & 1, 0], g0.reshape(-1))
            assert bool((b[flags_off:].view(torch.int32).view(world, pairs)[0] == call).all())


def test_empty_and_single_sample_batches():
    """Ragged minibatches: an empty slice contributes a zero W gradient, a short last batch is served."""
    rng = np.random.default_rng(7)
    V = rng.random((3, 2, 12, 10)).astype(np.float32)
    W = rng.random((3, 2, 4, 3)).astype(np.float32)
    H = rng.random((3, 3, 15, 12)).astype(np.float32)
    be, Wd, Hd = _backend(V, W, H)
    grad = torch.full((2, *Wd.shape), 7.0, dtype=Wd.dtype, device=Wd.device)
    be.gradient_W(V, Wd, Hd, slice(0, 0), grad)
    assert float(grad.abs().max()) == 0.0
    be.update_H(V, Wd, Hd, slice(0, 0))                      # no-op
    _close(Hd, H, 0.0)
    full = torch.empty_like(grad)
    be.gradient_W(V, Wd, Hd, slice(None), full)
    parts = torch.zeros_like(grad)
    for s in (slice(0, 2), slice(2, 3)):
        parts += be.gradient_W(V, Wd, Hd, s, torch.empty_like(grad))
    _close(parts, full.cpu().numpy(), 1e-5)


# ---------------------------------------------------------------------------------------------------------
# size-independent properties at BASELINE's full 2-D sizes (the oracle cannot run these)
# ---------------------------------------------------------------------------------------------------------
FULL_SIZE = {
    'cfg2': dict(N=8, C=3, M=16, D=(256, 256), A=(11, 11)),        # full per-sample geometry, N reduced to 8
    'cfg3': dict(N=16, C=1, M=32, D=(128, 128), A=(15, 15)),
    'cfg4': dict(N=32, C=1, M=64, D=(4096,), A=(128,)),
    'cfg5': dict(N=1, C=1, M=8, D=(512, 512), A=(64, 64)),
}


@pytest.mark.parametrize('name', list(FULL_SIZE))
def test_trilinear_identities_at_full_size(name):
    """All five hot-path tensors are partial derivatives of one trilinear form F(X, W, H) (SURVEY 0):
    <X, reconstruct(W,H)> = <H, negH(X)> = <W, negW(X)>, and reconstruct is linear in H.  Checked in float32 on
    the tiled path at the full per-sample geometry of BASELINE configs 2-5."""
    c = FULL_SIZE[name]
    torch.manual_seed(1)
    from tnmf_b200 import B200_Backend
    be = B200_Backend(init='device', kernel_path='tiled')
    dev = be.device
    V = torch.rand((c['N'], c['C'], *c['D']), dtype=torch.float32, device=dev)
    W, H = be.initialize(V, c['A'], c['M'], None, tuple(range(-len(c['A']), 0)))
    assert be.uses_tiled_kernels()
    R = be.reconstruct(W, H).clone()
    f_r = float((V.double() * R.double()).sum())
    neg, pos = be.reconstruction_gradient_H(V, W, H)
    f_h = float((H.double() * neg.double()).sum())
    f_hp = float((H.double() * pos.double()).sum())
    negw, posw = be.reconstruction_gradient_W(V, W, H)
    f_w = float((W.double() * negw.double()).sum())
    f_wp = float((W.double() * posw.double()).sum())
    rr = float((R.double() ** 2).sum())
    assert np.isclose(f_h, f_r, rtol=2e-5) and np.isclose(f_w, f_r, rtol=2e-5)
    assert np.isclose(f_hp, rr, rtol=2e-5) and np.isclose(f_wp, rr, rtol=2e-5)
    # linearity in H
    H2 = torch.rand_like(H)
    R2 = be.reconstruct(W, H2).clone()
    R12 = be.reconstruct(W, H + 2 * H2)
    # float32 chains of K = M*prod(A) terms (32768 at cfg5): rounding grows like sqrt(K)*2^-24
    _close(R12, (R + 2 * R2).cpu().numpy(), 5e-5)
    # energy = 0.5*||V - R||^2
    e = be.reconstruction_energy(V, W, H)
    assert np.isclose(e, 0.5 * float(((V.double() - R.double()) ** 2).sum()), rtol=1e-6)
    # tiled and generic kernels agree on a sub-batch
    bg = B200_Backend(init='device', kernel_path='generic')
    n_sub = min(2, c['N'])
    bg.initialize(V[:n_sub], c['A'], c['M'], None, tuple(range(-len(c['A']), 0)))
    _close(bg.reconstruct(W, H[:n_sub]), R[:n_sub].cpu().numpy(), 2e-5)
    # the MU keeps everything non-negative and the energy does not increase (Lee-Seung)
    be.update_H(V, W, H)
    grad = torch.empty((2, *W.shape), dtype=W.dtype, device=dev)
    be.apply_W_update(W, be.gradient_W(V, W, H, slice(None), grad))
    assert float(H.min()) >= 0 and float(W.min()) >= 0
    assert np.allclose(W.sum(dim=tuple(range(2, W.dim()))).cpu().numpy(), 1.0, atol=1e-5)
    assert be.reconstruction_energy(V, W, H) <= e * (1 + 1e-6)


def test_missing_library_is_loud(monkeypatch):
    """No silent fallback: without the shared object the binding refuses to load."""
    from tnmf_b200 import _lib
    monkeypatch.setattr(_lib, '_lib', None)
    monkeypatch.setattr(_lib, 'LIB_PATH', '/nonexistent/libtnmf_b200.so')
    with pytest.raises(ImportError):
        _lib.load()


def test_unsupported_requests_raise():
    from tnmf_b200 import B200_Backend, TransformInvariantNMF
    with pytest.raises(NotImplementedError):
        B200_Backend(reconstruction_mode='reflect')
    with pytest.raises(ValueError):
        B200_Backend(reconstruction_mode='bogus')
    with pytest.raises(ValueError):
        TransformInvariantNMF(2, (3,), backend='numpy')
    be = B200_Backend(kernel_path='tiled')
    V = np.random.default_rng(0).random((1, 1, 4, 4, 4))
    with pytest.raises(NotImplementedError):                 # three shift axes in float64 have no tiled kernel
        W, H = be.initialize(V, (2, 2, 2), 2, None, (-3, -2, -1))
        be.reconstruct(W, H)
