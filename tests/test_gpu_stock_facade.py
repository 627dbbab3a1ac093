"""
The route a tnmf user takes without touching tnmf (INTEGRATION.md 3 i): the reference facade drives `B200_Backend`
through the abstract backend interface only, applying its duck-typed operations to the `B200Tensor`s the backend
returns - including the lateral-inhibition branch that mixes a backend tensor with an ndarray
(tnmf/TransformInvariantNMF.py:258), the cross-atom branch (`.sum(axis=1, keepdims=True)`, :263) and the write-through
`H[s]` views and `0 + tensor` accumulation of the Cyclic_MU minibatches (:457-465).

The facade's iteration code is restated in tests/stock_facade.py; the results are compared with the outputs of the
unmodified reference (facade and numpy_fft backend) stored by tests/golden/make_golden.py for the same recipes:
ref_test_1d (tnmf/tests/test_1d.py:17-22,32-53), ref_fit_2d (all regularisers) and ref_minibatch (Cyclic_MU).
"""
import numpy as np
import pytest

from oracle import tnmf_oracle as orc
from stock_facade import StockFacade

pytestmark = pytest.mark.gpu

GOLDEN_E = {'valid': 2.34946, 'full': 1.87180, 'circular': 3.13228}        # tnmf/tests/test_1d.py:17-22


def _facade(mode, n_atoms, atom_shape):
    from tnmf_b200 import B200_Backend
    return StockFacade(B200_Backend(reconstruction_mode=mode), n_atoms, atom_shape)


@pytest.mark.parametrize('mode', list(GOLDEN_E))
def test_stock_facade_drives_b200_backend_1d(mode, golden):
    g = golden('ref_test_1d')
    W, H = g[f'W_{mode}'], g[f'H_{mode}']
    np.random.seed(42)
    got = _facade(mode, 3, (5,))
    got.fit_batch(g['V'], inhibition_strength=0.1, n_iterations=10)
    assert np.isclose(got._energy_function(), GOLDEN_E[mode], rtol=1e-5)
    assert np.isclose(got._energy_function(), g[f'E_{mode}'], rtol=1e-9)
    assert np.allclose(got.W, W, rtol=1e-8, atol=1e-12) and np.allclose(got.H, H, rtol=1e-7, atol=1e-12)
    assert np.allclose(got.R, g[f'R_{mode}'], rtol=1e-8, atol=1e-12)
    assert np.allclose(got.R_partial(1), orc.reconstruct(W[1:2], H[:, 1:2], mode), rtol=1e-8, atol=1e-12)


@pytest.mark.parametrize('dtype', [np.float64, np.float32])
def test_stock_facade_2d_all_regularisers(dtype, golden):
    """The reference's float64 run; the float32 run of the same recipe follows it within float32 rounding."""
    g = golden('ref_fit_2d')
    np.random.seed(5)
    got = _facade('valid', 4, (5, 3))
    traj = []
    got.fit_batch(g['V'].astype(dtype), n_iterations=20, sparsity_H=0.1, inhibition_strength=0.2,
                  cross_atom_inhibition_strength=0.4,
                  progress_callback=lambda m, i: traj.append(m._energy_function()) or True)
    tol = 1e-8 if dtype == np.float64 else 1e-3
    assert got.W.dtype == dtype and got.H.dtype == dtype
    assert np.allclose(traj, g['valid_all_E'], rtol=1e-9 if dtype == np.float64 else 1e-4)
    assert np.abs(got.W - g['valid_all_W']).max() <= tol * np.abs(g['valid_all_W']).max()
    assert np.abs(got.H - g['valid_all_H']).max() <= tol * np.abs(g['valid_all_H']).max()


def test_stock_facade_minibatch(golden):
    """Cyclic_MU minibatches: H[s] views updated in place, the W gradient summed over the batches from `0 + tensor`."""
    g = golden('ref_minibatch')
    np.random.seed(42)
    got = _facade('valid', 3, (4, 4))
    got.fit_cyclic_minibatches(g['V'], batch_size=3, n_epochs=5, sparsity_H=0.1)
    assert np.isclose(got._energy_function(), g['Cyclic_MU_E'], rtol=1e-9)
    assert np.allclose(got.W, g['Cyclic_MU_W'], rtol=1e-8, atol=1e-12)
    assert np.allclose(got.H, g['Cyclic_MU_H'], rtol=1e-7, atol=1e-12)
