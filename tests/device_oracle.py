"""
Float64 reference of the 'valid'-mode MU operations in torch, for checking the kernels at the batch sizes bench.py times.

TEST HELPER ONLY.  This is a port of the Fourier-space functions of oracle/tnmf_oracle.py (`fft_reconstruct`,
`_fft_correlate`, `fft_gradient_H`, `fft_gradient_W`, with the transform lengths of `_fft_plan`) to torch.fft, so that
the reference runs on the GPU, beside the kernels it checks, at batches the numpy oracle would take hours over.  Index
conventions are the oracle's: V[n, c, *D], W[m, c, *A], H[n, m, *T], T = D + A - 1.  tests/test_device_oracle.py pins it
to the numpy oracle on the CPU.

Whole batches are processed in chunks of samples (`sample_chunks`, `chunk_for`), each cast to float64 on its device.
H may be the pitched view the backend allocates (H[..., :T_x] of a buffer with longer rows): every chunk is copied out
of it.  The reconstruction, the H gradients and the H update are per sample and come chunk by chunk; the W gradient
sums over the chunks in float64.
"""
from typing import Callable, List, Optional, Sequence, Tuple

import torch

from oracle import tnmf_oracle as orc

EPS = orc.EPS
SPECTRA_BYTES = 4 << 30         # spectra of one chunk of samples


def fft_shape(sample_shape: Sequence[int], atom_shape: Sequence[int]) -> Tuple[int, ...]:
    """Transform lengths next_fast_len(D + T - 1) per shift axis, as the numpy oracle uses them."""
    return orc._fft_plan(sample_shape, atom_shape)          # pylint: disable=protected-access


def chunk_for(n_channels: int, n_atoms: int, sample_shape: Sequence[int], atom_shape: Sequence[int],
              budget: int = SPECTRA_BYTES) -> int:
    """Samples per chunk such that the complex128 spectra of one chunk's H and V (or R) stay within `budget` bytes."""
    shape = fft_shape(sample_shape, atom_shape)
    freq = 1
    for L in shape[:-1]:
        freq *= L
    freq *= shape[-1] // 2 + 1
    return max(1, budget // ((n_atoms + n_channels) * freq * 16))


def sample_chunks(n: int, chunk: int) -> List[slice]:
    return [slice(lo, min(n, lo + chunk)) for lo in range(0, n, chunk)]


def f64(x: torch.Tensor) -> torch.Tensor:
    """Dense float64 copy on x's device (of a pitched view, too)."""
    return x.to(torch.float64).contiguous()


def _dims(k: int) -> Tuple[int, ...]:
    return tuple(range(-k, 0))


# ---------------------------------------------------------------------------------------------------
# the three contractions (float64 in, float64 out)
# ---------------------------------------------------------------------------------------------------
def reconstruct(W: torch.Tensor, H: torch.Tensor) -> torch.Tensor:
    """R = sum_m H[:, m] (*) W[m] cropped to the sample: `fft_reconstruct`."""
    k = W.dim() - 2
    atom_shape = tuple(W.shape[2:])
    sample_shape = tuple(t - a + 1 for t, a in zip(H.shape[2:], atom_shape))
    shape = fft_shape(sample_shape, atom_shape)
    Hf = torch.fft.rfftn(H, s=shape, dim=_dims(k))
    Wf = torch.fft.rfftn(W, s=shape, dim=_dims(k))
    full = torch.fft.irfftn(torch.einsum('nm...,mc...->nc...', Hf, Wf), s=shape, dim=_dims(k))
    crop = (slice(None), slice(None)) + tuple(slice(a - 1, a - 1 + d) for a, d in zip(atom_shape, sample_shape))
    return full[crop].contiguous()


def _correlate(X: torch.Tensor, Y: torch.Tensor, contraction: str, out_shape: Sequence[int], shift: Sequence[int],
               shape: Sequence[int]) -> torch.Tensor:
    """c[k] = sum_d X[d] * Y[d + k] for k = shift_i .. shift_i + out_shape_i - 1 (circular indices), contracted over the
    labelled axes: `_fft_correlate`."""
    k = len(shape)
    Xf = torch.fft.rfftn(X, s=shape, dim=_dims(k))
    Yf = torch.fft.rfftn(Y, s=shape, dim=_dims(k))
    c = torch.fft.irfftn(torch.einsum(contraction, Xf.conj(), Yf), s=shape, dim=_dims(k))
    for ax, (s0, n, L) in enumerate(zip(shift, out_shape, shape)):
        idx = torch.arange(s0, s0 + n, device=c.device) % L
        c = torch.index_select(c, ax + 2, idx)
    return c


def gradient_H(V: torch.Tensor, W: torch.Tensor, H: torch.Tensor, R: Optional[torch.Tensor] = None):
    """(neg, pos)[n,m,t] = sum_c sum_a W[m,c,a] * X[n,c,t-p+a] with X = V, R: `fft_gradient_H`."""
    atom_shape, sample_shape = tuple(W.shape[2:]), tuple(V.shape[2:])
    shape = fft_shape(sample_shape, atom_shape)
    R = reconstruct(W, H) if R is None else R
    shift = tuple(-(a - 1) for a in atom_shape)
    return tuple(_correlate(W, X, 'mc...,nc...->nm...', H.shape[2:], shift, shape) for X in (V, R))


def gradient_W(V: torch.Tensor, W: torch.Tensor, H: torch.Tensor, R: Optional[torch.Tensor] = None):
    """(neg, pos)[m,c,a] = sum_n sum_d H[n,m,d+p-a] * X[n,c,d] with X = V, R: `fft_gradient_W`."""
    atom_shape, sample_shape = tuple(W.shape[2:]), tuple(V.shape[2:])
    shape = fft_shape(sample_shape, atom_shape)
    R = reconstruct(W, H) if R is None else R
    out = []
    for X in (V, R):
        g = _correlate(X, H, 'nc...,nm...->mc...', atom_shape, (0,) * len(atom_shape), shape)     # g[k], k = p - a
        out.append(torch.flip(g, dims=tuple(range(2, g.dim()))).contiguous())
    return out[0], out[1]


# ---------------------------------------------------------------------------------------------------
# the multiplicative updates, in the order of roundings of OracleNMF.update_H / update_W (no regularisers)
# ---------------------------------------------------------------------------------------------------
def update_H(V: torch.Tensor, W: torch.Tensor, H: torch.Tensor) -> torch.Tensor:
    """H * neg / (pos + eps) of one chunk (float64 in, a new float64 tensor out)."""
    neg, pos = gradient_H(V, W, H)
    pos += EPS
    out = H * neg
    out /= pos
    return out


def update_W(W: torch.Tensor, neg: torch.Tensor, pos: torch.Tensor) -> torch.Tensor:
    """W * neg / (pos + eps), normalised over the shift axes."""
    pos = pos + EPS
    out = W * neg
    out /= pos
    out /= out.sum(dim=_dims(W.dim() - 2), keepdim=True)
    return out


# ---------------------------------------------------------------------------------------------------
# whole batches, chunk by chunk.  V and H: float32 or float64 tensors of the whole batch (H possibly pitched); W: float64
# ---------------------------------------------------------------------------------------------------
def _chunk(V, W, H) -> int:
    return chunk_for(V.shape[1], W.shape[0], V.shape[2:], W.shape[2:])


def batch_gradient_W(V: torch.Tensor, W: torch.Tensor, H: torch.Tensor, chunk: Optional[int] = None,
                     on_R: Optional[Callable[[slice, torch.Tensor], None]] = None):
    """W gradient of the whole batch, summed over the chunks in float64; `on_R(s, R)` sees each chunk's reconstruction."""
    chunk = chunk or _chunk(V, W, H)
    neg = torch.zeros(W.shape, dtype=torch.float64, device=W.device)
    pos = torch.zeros_like(neg)
    for s in sample_chunks(V.shape[0], chunk):
        Vs, Hs = f64(V[s]), f64(H[s])
        R = reconstruct(W, Hs)
        if on_R is not None:
            on_R(s, R)
        n, p = gradient_W(Vs, W, Hs, R)
        neg += n
        pos += p
    return neg, pos


def mu_step(V: torch.Tensor, W: torch.Tensor, H: torch.Tensor, chunk: Optional[int] = None,
            on_H: Optional[Callable[[slice, torch.Tensor], None]] = None) -> torch.Tensor:
    """One batch MU iteration from (W, H): the H update, then the W update with the new H (OracleNMF.update_H followed by
    OracleNMF.update_W).  Calls `on_H(s, H1)` with each chunk of the updated H and returns the updated W."""
    chunk = chunk or _chunk(V, W, H)
    neg = torch.zeros(W.shape, dtype=torch.float64, device=W.device)
    pos = torch.zeros_like(neg)
    for s in sample_chunks(V.shape[0], chunk):
        Vs = f64(V[s])
        H1 = update_H(Vs, W, f64(H[s]))
        if on_H is not None:
            on_H(s, H1)
        n, p = gradient_W(Vs, W, H1)
        neg += n
        pos += p
    return update_W(W, neg, pos)
