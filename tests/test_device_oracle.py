"""
The torch float64 reference of tests/device_oracle.py against the numpy oracle, on the CPU: the reconstruction, both
gradients, the energy, the H and W updates and one MU step, on small random 1-D, 2-D and 3-D 'valid' problems, with H
given as a pitched view and with chunks of samples that do not divide the batch.  tests/test_gpu_bench_scale.py judges
the kernels at the benchmarked batch sizes by this reference, so it has to be right first.
"""
import numpy as np
import pytest
import torch

import device_oracle as dor
from oracle import tnmf_oracle as orc

RTOL = 1e-12

# N, C, M, D, A
CASES = {
    'd1': (5, 2, 3, (37,), (6,)),
    'd2': (5, 2, 4, (13, 17), (4, 5)),
    'd3': (3, 1, 3, (7, 9, 8), (3, 2, 4)),
}


def _problem(name, pad):
    N, C, M, D, A = CASES[name]
    rng = np.random.default_rng(len(D) * 10 + pad)
    V = rng.random((N, C) + D)
    W = rng.random((M, C) + A)
    T = orc.transform_shape('valid', D, A)
    H = rng.random((N, M) + T)
    # H as the backend lays it out: the [..., :T_x] view of a buffer whose rows are `pad` elements longer (filled with
    # values that would show up in every result if the view were read past its end)
    buf = torch.full((N, M) + T[:-1] + (T[-1] + pad,), 1e6, dtype=torch.float64)
    Ht = buf[..., :T[-1]]
    Ht.copy_(torch.from_numpy(H))
    return V, W, H, torch.from_numpy(V), torch.from_numpy(W), Ht


def _check(got, want):
    np.testing.assert_allclose(got.numpy() if isinstance(got, torch.Tensor) else got, want, rtol=RTOL, atol=0)


@pytest.mark.parametrize('pad', (0, 3))
@pytest.mark.parametrize('name', list(CASES))
def test_operations_equal_the_numpy_oracle(name, pad):
    V, W, H, Vt, Wt, Ht = _problem(name, pad)
    assert pad == 0 or not Ht.is_contiguous()
    _check(dor.reconstruct(Wt, dor.f64(Ht)), orc.reconstruct(W, H))
    neg, pos = dor.gradient_H(Vt, Wt, dor.f64(Ht))
    rn, rp = orc.reconstruction_gradient_H(V, W, H)
    _check(neg, rn)
    _check(pos, rp)
    neg, pos = dor.gradient_W(Vt, Wt, dor.f64(Ht))
    rn, rp = orc.reconstruction_gradient_W(V, W, H)
    _check(neg, rn)
    _check(pos, rp)


@pytest.mark.parametrize('chunk', (1, 2, 4, 100))
@pytest.mark.parametrize('name', list(CASES))
def test_chunked_batch_equals_the_numpy_oracle(name, chunk):
    """Chunks of 2 and 4 do not divide the 5 or 3 samples; 100 is one chunk for the whole batch."""
    V, W, H, Vt, Wt, Ht = _problem(name, 3)
    R_ref = orc.reconstruct(W, H)
    R = torch.empty(R_ref.shape, dtype=torch.float64)
    seen = []

    def on_R(s, Rs):
        seen.append(s)
        R[s] = Rs

    neg, pos = dor.batch_gradient_W(Vt, Wt, Ht, chunk=chunk, on_R=on_R)
    assert seen == dor.sample_chunks(V.shape[0], chunk)
    _check(R, R_ref)
    rn, rp = orc.reconstruction_gradient_W(V, W, H)
    _check(neg, rn)
    _check(pos, rp)
    energy = sum(float(0.5 * ((Vt[s] - R[s]) ** 2).sum()) for s in seen)
    assert energy == pytest.approx(float(orc.reconstruction_energy(V, W, H)), rel=RTOL)

    # one MU step: OracleNMF.update_H, then OracleNMF.update_W with the new H
    ref = orc.OracleNMF(W.shape[0], W.shape[2:])
    ref.V, ref.W, ref.H = V, W.copy(), H.copy()
    ref.update_H()
    H1_ref = ref.H.copy()
    ref.update_W()
    H1 = torch.empty(H.shape, dtype=torch.float64)

    def on_H(s, Hs):
        H1[s] = Hs

    W1 = dor.mu_step(Vt, Wt, Ht, chunk=chunk, on_H=on_H)
    _check(H1, H1_ref)
    _check(W1, ref.W)
    # the single updates on their own
    _check(dor.update_H(Vt, Wt, dor.f64(Ht)), H1_ref)
    nmf = orc.OracleNMF(W.shape[0], W.shape[2:])
    nmf.V, nmf.W, nmf.H = V, W.copy(), H.copy()
    nmf.update_W()
    _check(dor.update_W(Wt, *dor.gradient_W(Vt, Wt, dor.f64(Ht))), nmf.W)
    # the inputs are left as they were
    assert torch.equal(Wt, torch.from_numpy(W)) and torch.equal(Ht, torch.from_numpy(H))


def test_chunk_size_keeps_the_spectra_within_the_budget():
    # cfg3: transforms of 270 x 270, 32 atoms + 1 channel: 270 * 136 * 33 * 16 bytes = 19.4 MB of spectra per sample
    assert dor.fft_shape((128, 128), (15, 15)) == (270, 270)
    n = dor.chunk_for(1, 32, (128, 128), (15, 15))
    assert n == (4 << 30) // (270 * 136 * 33 * 16)
    assert dor.chunk_for(3, 16, (256, 256), (11, 11), budget=1) == 1
    assert dor.sample_chunks(7, 3) == [slice(0, 3), slice(3, 6), slice(6, 7)]
