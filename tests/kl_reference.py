"""
Float64 numpy reference of the Kullback-Leibler multiplicative updates, built from oracle/tnmf_oracle.py.

TEST HELPER ONLY.  D(V||R) = sum [V log(V / R~) - V + R] with R~ = max(R, tau), tau the smallest normal number of the
dtype, and 0 log 0 = 0.  Its gradients are the oracle's correlations with (Q, ones) in place of (V, R), Q = V / R~ (0
where V = 0):  dD/dH = corr_W(ones) - corr_W(Q),  dD/dW = corr_H(ones) - corr_H(Q).  So (neg, pos) = (corr(Q), corr(ones))
and the multiplicative update H <- H * neg / (pos + eps) is Lee and Seung's KL update.  tests/test_kl_cpu.py pins
pos - neg to torch.autograd of D.

`OracleKL` is `OracleNMF` with these gradients and this energy, so its fit loops and minibatch schedules are the
oracle's.
"""
from typing import Tuple

import numpy as np

from oracle import tnmf_oracle as orc


def tau(dtype) -> float:
    return float(np.finfo(dtype).tiny)


def quotient(V: np.ndarray, R: np.ndarray) -> np.ndarray:
    """Q = V / max(R, tau), 0 where V = 0, in the dtype of R."""
    Rt = np.maximum(R, np.asarray(tau(R.dtype), dtype=R.dtype))
    with np.errstate(divide='ignore', invalid='ignore'):
        return np.where(V > 0, V / Rt, 0).astype(R.dtype, copy=False)


def divergence(V: np.ndarray, R: np.ndarray) -> float:
    """D(V||R), every term in float64 from the given inputs."""
    V64, R64 = V.astype(np.float64), R.astype(np.float64)
    Rt = np.maximum(R, np.asarray(tau(R.dtype), dtype=R.dtype)).astype(np.float64)
    with np.errstate(divide='ignore', invalid='ignore'):
        vlog = np.where(V64 > 0, V64 * np.log(V64 / Rt), 0.0)
    return float(np.sum(vlog - V64 + R64))


def gradient_H(V: np.ndarray, W: np.ndarray, H: np.ndarray, mode: str = 'valid') -> Tuple[np.ndarray, np.ndarray]:
    """(neg, pos) of the KL H gradient, H's shape."""
    atom_shape = W.shape[2:]
    Q = quotient(V, orc.reconstruct(W, H, mode))
    neg = orc.unpad_gradient(orc._correlate_with_atoms(Q, W), atom_shape, mode, H.shape[2:])          # pylint: disable=protected-access
    pos = orc.unpad_gradient(orc._correlate_with_atoms(np.ones_like(Q), W), atom_shape, mode, H.shape[2:])  # pylint: disable=protected-access
    return neg, pos


def gradient_W(V: np.ndarray, W: np.ndarray, H: np.ndarray, mode: str = 'valid') -> Tuple[np.ndarray, np.ndarray]:
    """(neg, pos) of the KL W gradient, W's shape."""
    atom_shape = W.shape[2:]
    Q = quotient(V, orc.reconstruct(W, H, mode))
    Hp = orc.pad_activations(H, atom_shape, mode)
    return (orc._correlate_with_activations(Q, Hp, atom_shape),                  # pylint: disable=protected-access
            orc._correlate_with_activations(np.ones_like(Q), Hp, atom_shape))    # pylint: disable=protected-access


class OracleKL(orc.OracleNMF):
    """OracleNMF minimising D(V||R): the same updates, regularisers and schedules, with the KL gradients."""

    def energy(self):
        return divergence(self.V, orc.reconstruct(self.W, self.H, self.mode))

    def update_H(self, s=slice(None), sparsity=0.0, inhibition=0.0, cross_inhibition=0.0) -> None:
        Hs = self.H[s]
        neg, pos = gradient_H(self.V[s], self.W, Hs, self.mode)
        if inhibition > 0 or cross_inhibition > 0:
            G = orc.convolve_multi_1d(Hs, self.inhibition_kernels, self.shift_axes)
            if inhibition > 0:
                tmp = G - Hs
                tmp *= inhibition
                pos += tmp
            if cross_inhibition > 0:
                tmp = G.sum(axis=1, keepdims=True)
                tmp = -G + tmp
                tmp *= cross_inhibition / (self.n_atoms - 1)
                pos += tmp
        orc.multiplicative_update(Hs, neg, pos, sparsity=sparsity)

    def gradient_W(self, s=slice(None)):
        return gradient_W(self.V[s], self.W, self.H[s], self.mode)
