"""
CPU checks of the Kullback-Leibler updates (no device): the float64 reference of tests/kl_reference.py against
torch.autograd of D(V||R), the monotone descent of its H update, the argument validation of tnmf_kl_quotient /
tnmf_kl_workspace_bytes, and the facade's validation of `divergence`.
"""
import ctypes
import itertools

import numpy as np
import pytest
import torch

from oracle import tnmf_oracle as orc
import kl_reference as klr
from tnmf_b200 import _lib

MODES = ('valid', 'full', 'circular')
SHAPES = [
    # n, c, m, sample shape, atom shape
    (2, 2, 3, (17,), (5,)),
    (2, 2, 3, (9, 8), (3, 4)),
    (1, 2, 2, (6, 5, 7), (2, 3, 2)),
]


def _torch_reconstruct(W: torch.Tensor, H: torch.Tensor, mode: str) -> torch.Tensor:
    """Shift-and-add R[n,c,d] = sum_m sum_a W[m,c,a] * Hpad[n,m,d+p-a], written independently of the oracle."""
    k = W.dim() - 2
    A = W.shape[2:]
    Hp = H
    for i, a in enumerate(A):
        ax = 2 + i
        if a == 1 or mode == 'valid':
            continue
        if mode == 'full':
            z = torch.zeros(Hp.shape[:ax] + (a - 1,) + Hp.shape[ax + 1:], dtype=H.dtype)
            Hp = torch.cat((z, Hp, z), dim=ax)
        else:                                            # circular: wrap (p, 0)
            Hp = torch.cat((Hp.narrow(ax, Hp.shape[ax] - (a - 1), a - 1), Hp), dim=ax)
    D = tuple(t - a + 1 for t, a in zip(Hp.shape[2:], A))
    R = torch.zeros((H.shape[0], W.shape[1]) + D, dtype=H.dtype)
    for off in itertools.product(*(range(a) for a in A)):
        win = Hp
        for i, (o, a, d) in enumerate(zip(off, A, D)):
            win = win.narrow(2 + i, a - 1 - o, d)
        R = R + torch.einsum('mc,nm...->nc...', W[(slice(None), slice(None)) + off], win)
    assert R.dim() == 2 + k
    return R


def _torch_divergence(V: torch.Tensor, R: torch.Tensor) -> torch.Tensor:
    Rt = R.clamp(min=klr.tau(np.float64))
    return torch.sum(torch.where(V > 0, V * torch.log(torch.where(V > 0, V, 1.0) / Rt), 0.0) - V + R)


@pytest.mark.parametrize('mode', MODES)
@pytest.mark.parametrize('case', range(len(SHAPES)))
def test_reference_gradients_equal_autograd(case, mode):
    """pos - neg of the reference is dD/dH and dD/dW, in every mode and for 1, 2 and 3 shift axes."""
    n, c, m, D, A = SHAPES[case]
    rng = np.random.default_rng(40 + case)
    V = rng.random((n, c) + D)
    V[V < 0.15] = 0.0                           # exact zeros: their quotient is 0 and their term is R
    W = rng.random((m, c) + A) + 0.05
    H = rng.random((n, m) + orc.transform_shape(mode, D, A)) + 0.05
    Wt = torch.tensor(W, requires_grad=True)
    Ht = torch.tensor(H, requires_grad=True)
    R = _torch_reconstruct(Wt, Ht, mode)
    assert np.allclose(R.detach().numpy(), orc.reconstruct(W, H, mode), rtol=1e-13)
    d = _torch_divergence(torch.tensor(V), R)
    d.backward()
    assert np.isclose(float(d.detach()), klr.divergence(V, orc.reconstruct(W, H, mode)), rtol=1e-12)
    for grad, (neg, pos) in ((Ht.grad, klr.gradient_H(V, W, H, mode)), (Wt.grad, klr.gradient_W(V, W, H, mode))):
        want = grad.numpy()
        err = np.abs((pos - neg) - want).max() / np.abs(want).max()
        assert err <= 1e-10, err


@pytest.mark.parametrize('mode', MODES)
@pytest.mark.parametrize('case', range(len(SHAPES)))
def test_h_updates_never_increase_the_objective(case, mode):
    """H <- H * corr(Q) / (corr(1) + eps) majorises-minimises D + eps * sum H: the objective never increases."""
    n, c, m, D, A = SHAPES[case]
    rng = np.random.default_rng(60 + case)
    V = rng.random((n, c) + D)
    V[V < 0.1] = 0.0
    np.random.seed(7 + case)
    ref = klr.OracleKL(m, A, reconstruction_mode=mode)
    ref.initialize(V)
    objective = []
    for _ in range(12):
        objective.append(ref.energy() + orc.EPS * ref.H.sum())
        ref.update_H()
    objective.append(ref.energy() + orc.EPS * ref.H.sum())
    assert all(b <= a * (1 + 1e-12) for a, b in zip(objective, objective[1:])), objective
    assert objective[-1] < objective[0]


@pytest.fixture(scope='module')
def lib():
    _lib.build()
    return _lib.load()


def test_kl_entry_points_reject_bad_arguments(lib):
    p = _lib.make_problem(3, 2, 4, (20, 17), (5, 2), _lib.TNMF_F32)
    need = lib.tnmf_kl_workspace_bytes(ctypes.byref(p))
    assert need > 0 and need % 256 == 0
    for dtype, mode, shape, atoms in ((_lib.TNMF_F64, 'full', (9,), (3,)), (_lib.TNMF_F32, 'circular', (5, 6, 7), (2, 2, 2)),
                                      (_lib.TNMF_F32, 'valid', (4096, 4096), (3, 3))):
        q = _lib.make_problem(64, 3, 4, shape, atoms, dtype, mode)
        assert lib.tnmf_kl_workspace_bytes(ctypes.byref(q)) % 256 == 0 and lib.tnmf_kl_workspace_bytes(ctypes.byref(q)) > 0
    e = ctypes.c_double()
    ptr = ctypes.c_void_p(256)          # never dereferenced: every call below fails validation before a launch
    assert lib.tnmf_kl_quotient(ctypes.byref(p), None, ptr, None, None, 0, None) == _lib.TNMF_EINVAL
    assert lib.tnmf_kl_quotient(ctypes.byref(p), ptr, None, None, None, 0, None) == _lib.TNMF_EINVAL
    assert lib.tnmf_kl_quotient(None, ptr, ptr, None, None, 0, None) == _lib.TNMF_EINVAL
    assert lib.tnmf_kl_quotient(ctypes.byref(p), ptr, ptr, ctypes.byref(e), ptr, need - 1, None) == _lib.TNMF_EWORKSPACE
    assert lib.tnmf_kl_quotient(ctypes.byref(p), ptr, ptr, ctypes.byref(e), None, need, None) == _lib.TNMF_EWORKSPACE
    for field, value in (('mode', 7), ('reserved', 1), ('n_samples', -1), ('n_channels', 0)):
        bad = _lib.make_problem(3, 2, 4, (20, 17), (5, 2), _lib.TNMF_F32)
        setattr(bad, field, value)
        assert lib.tnmf_kl_quotient(ctypes.byref(bad), ptr, ptr, None, None, 0, None) == _lib.TNMF_EINVAL, field
        assert lib.tnmf_kl_workspace_bytes(ctypes.byref(bad)) == 0, field
    bad = _lib.make_problem(3, 2, 4, (4,), (5,), _lib.TNMF_F32, 'full')          # atom larger than sample
    assert lib.tnmf_kl_quotient(ctypes.byref(bad), ptr, ptr, None, None, 0, None) == _lib.TNMF_EINVAL


def test_facade_validates_the_divergence():
    from tnmf_b200 import TransformInvariantNMF
    with pytest.raises(ValueError, match='divergence'):
        TransformInvariantNMF(n_atoms=2, atom_shape=(3,), divergence='itakura-saito')
    with pytest.raises(ValueError, match='fused'):
        TransformInvariantNMF(n_atoms=2, atom_shape=(3,), divergence='kl', fused=False)
