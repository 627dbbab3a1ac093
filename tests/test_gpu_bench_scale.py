"""
Every hot kernel at the batch sizes bench.py times, against the float64 reference of tests/device_oracle.py.

The other parity tests check the kernels against the CPU oracle at batches reduced until the oracle finishes in seconds.
The batch does not change which kernel runs, but it changes how each kernel splits its work over the CTAs and how far
its offsets reach: with 1024 cfg3 samples a CTA of the reconstruction covers several whole tiles, and with the 8192
samples bench.py also fits on one GPU, H has 5.4e9 elements, more than 2^32.  Here every workload runs at its benchmarked
batch, set up as bench.py sets it up (device initialisation, bench.seed_start_values, kernel_path='auto'), and each
operation is called on the whole batch - a slice would move the large offsets into the base pointer, where the kernel
never sees them.  The reference is the oracle's Fourier-space arithmetic in float64 on the same GPU, chunk by chunk.

Errors are max-relative, max|delta| / max|ref|, as in the rest of the suite, and are printed for every comparison
(run with -s to see them).  Tolerances:
    R, H gradients              2e-5   (cfg5 5e-5: float32 chains of K = M * prod(A) = 32768 terms, as
                                        test_trilinear_identities_at_full_size explains)
    energy                      2e-5 relative
    W gradient                  2e-5
    fused H update, W update    5e-5
    W and H after one step      1e-4
The W gradient sums N * prod(D) products per entry.  On the tensor-core kernels they are 3xTF32 products in accumulation
chains cut every 8 or 12 source rows (the tensor core truncates when it accumulates), the chains are added into per-CTA
FP32 slices with round-to-nearest, and the slices are finished in double.  A chain of k truncating adds is biased by at
most k ulp, about k * 6e-8 relative (< 1e-6 for k <= 12).  The round-to-nearest adds into a slice do not share a sign,
so their error grows like the square root of the number of adds, and the finish adds nothing at float32 precision.  The
FP32 kernels (tiled, TMA) have no truncating chains.  Neither grows with the batch like the 2e-5 budget would need.
"""
import gc
import importlib.util
import os
import time

import numpy as np
import pytest
import torch

import device_oracle as dor

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _workloads():
    """name -> (N, C, M, D, A) of every benchmarked batch: bench.WORKLOADS, the 8192 cfg3 samples bench.measure_cfg3 fits
    on one GPU, and the volume of tools/bench_3d.py."""
    import bench
    spec = importlib.util.spec_from_file_location('bench_3d', os.path.join(ROOT, 'tools', 'bench_3d.py'))
    b3 = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b3)
    out = {name: (w['N'], w['C'], w['M'], tuple(w['D']), tuple(w['A'])) for name, w in bench.WORKLOADS.items()}
    c3 = out['cfg3']
    out['cfg3_8192'] = (8192,) + c3[1:]                # measure_cfg3: `total` samples on rank 0 alone
    out['vol'] = (b3.N, b3.C, b3.M, tuple(b3.D), tuple(b3.A))
    return out


WORKLOADS = _workloads()

# the kernels kernel_path='auto' plans for these batches (tnmf_kernel_name; checked on the CPU by test_kernel_plan.py's
# problems): a planner change shows up here
KERNELS = {
    'cfg1': ('tiled::recon_kernel', 'tiled::hupd_kernel', 'tiled::gradw_kernel'),
    'cfg2': ('recon_ts_kernel', 'hupd_ts_kernel', 'gradw_ts_kernel'),
    'cfg3': ('recon_os_kernel', 'hupd_ts_kernel', 'gradw_ns_kernel'),
    'cfg3_8192': ('recon_os_kernel', 'hupd_ts_kernel', 'gradw_ns_kernel'),
    'cfg4': ('recon_tma_kernel', 'hupd_tma_kernel', 'gradw_tma_kernel'),
    'cfg5': ('recon_tma_kernel', 'tiled::hupd_kernel', 'gradw_tma_kernel'),
    'vol': ('recon_os3_kernel', 'hupd_ts3_kernel', 'gradw_ns3_kernel'),
}
GRADIENT_H = {'cfg3_8192': False}      # its two H-sized outputs would add 43 GB

TOL = {'R': 2e-5, 'energy': 2e-5, 'grad_H': 2e-5, 'grad_W': 2e-5, 'update_H': 5e-5, 'update_W': 5e-5, 'step': 1e-4}
TOL_K32768 = {'R': 5e-5, 'grad_H': 5e-5}
CASES = ('cfg1', 'cfg2', 'cfg3', 'cfg4', 'cfg5', 'vol', 'cfg3_8192')


class MaxRel:
    """max|got - ref| / max|ref| over chunks, and where the largest difference sits (sample first)."""

    def __init__(self):
        self.diff, self.ref, self.at = 0.0, 0.0, None

    def add(self, got: torch.Tensor, ref: torch.Tensor, s: slice = slice(None)):
        d = (got.to(torch.float64) - ref).abs()
        dmax = float(d.max())
        if dmax > self.diff:
            at = [int(i) for i in np.unravel_index(int(d.argmax()), tuple(d.shape))]
            at[0] += s.start or 0
            self.diff, self.at = dmax, tuple(at)
        self.ref = max(self.ref, float(ref.abs().max()))

    @property
    def err(self) -> float:
        return self.diff / max(self.ref, 1e-300)


def _bytes_needed(N, C, M, D, A, gradient_H):
    T = [d + a - 1 for d, a in zip(D, A)]
    h = N * M * int(np.prod(T[:-1])) * (T[-1] + 3) * 4            # H with its padded rows ...
    h0 = N * M * int(np.prod(T)) * 4                               # ... the saved start H ...
    v = N * C * int(np.prod(D)) * 4                                # ... V and three R-sized buffers
    return h + h0 * (3 if gradient_H else 1) + 4 * v + 4 * dor.SPECTRA_BYTES


@pytest.mark.parametrize('name', CASES)
def test_bench_scale_against_float64_reference(name):
    import bench
    from tnmf_b200 import TransformInvariantNMF
    t_start = time.perf_counter()
    N, C, M, D, A = WORKLOADS[name]
    dev = torch.device('cuda', torch.cuda.current_device())
    with_grad_H = GRADIENT_H.get(name, True)
    need = _bytes_needed(N, C, M, D, A, with_grad_H)
    gc.collect()
    torch.cuda.empty_cache()
    free, _ = torch.cuda.mem_get_info(dev)
    if free < need:
        pytest.skip(f'{name}: needs about {need / 1e9:.1f} GB of device memory, {free / 1e9:.1f} GB are free')

    # ---- set up as bench.time_steps / run_b200 do ------------------------------------------------------------------
    gen = torch.Generator(device=dev)
    gen.manual_seed(4321)
    V = torch.rand((N, C, *D), dtype=torch.float32, device=dev, generator=gen)
    nmf = TransformInvariantNMF(n_atoms=M, atom_shape=A, backend='b200', init='device', distributed=False,
                                input_is_local_shard=True, equal_shards=True, kernel_path='auto')
    nmf._initialize_matrices(V, keep_W=False)                            # pylint: disable=protected-access
    bench.seed_start_values(nmf, dev, 0)
    be, W, H = nmf._backend, nmf.W_device, nmf.H_device                  # pylint: disable=protected-access
    want = dict(zip(('reconstruct', 'update_h', 'gradient_w'), KERNELS[name]))
    assert be.kernel_names(N) == want, be.kernel_names(N)
    W0 = W.clone()
    W64 = W0.to(torch.float64)
    tol = dict(TOL, **(TOL_K32768 if name == 'cfg5' else {}))
    err, at = {}, {}
    print(f'\n{name}: {N} x {C}x{"x".join(map(str, D))}, {M} atoms {"x".join(map(str, A))}; kernels {want}; '
          f'reference chunks of {dor.chunk_for(C, M, D, A)} samples')

    # ---- reconstruction, energy, W gradient (one reference pass) ----------------------------------------------------
    R = be.reconstruct(W, H)
    assert be.kernel_names() == want, be.kernel_names()
    e_gpu = be.reconstruction_energy(V, W, H)
    gW = torch.empty((2, *W.shape), dtype=W.dtype, device=dev)
    be.gradient_W(V, W, H, slice(None), gW)
    W_upd = W.clone()
    be.apply_W_update(W_upd, gW)
    torch.cuda.synchronize(dev)
    m_R = MaxRel()
    e_ref = torch.zeros((), dtype=torch.float64, device=dev)

    def on_R(s, Rs):
        nonlocal e_ref
        m_R.add(R[s], Rs, s)
        e_ref = e_ref + 0.5 * ((V[s].to(torch.float64) - Rs) ** 2).sum()

    rn, rp = dor.batch_gradient_W(V, W64, H, on_R=on_R)
    e_ref = float(e_ref)
    err['R'], at['R'] = m_R.err, m_R.at
    err['energy'] = abs(e_gpu - e_ref) / abs(e_ref)
    for key, got, ref in (('grad_W neg', gW[0], rn), ('grad_W pos', gW[1], rp),
                          ('update_W', W_upd, dor.update_W(W64, rn, rp))):
        m = MaxRel()
        m.add(got, ref)
        err[key], at[key] = m.err, m.at
    del R, gW, W_upd, rn, rp

    # ---- H gradients (the unfused reference-interface call) ---------------------------------------------------------
    if with_grad_H:
        neg, pos = be.reconstruction_gradient_H(V, W, H)
        m_neg, m_pos = MaxRel(), MaxRel()
        for s in dor.sample_chunks(N, dor.chunk_for(C, M, D, A)):
            rn, rp = dor.gradient_H(dor.f64(V[s]), W64, dor.f64(H[s]))
            m_neg.add(neg[s], rn, s)
            m_pos.add(pos[s], rp, s)
            del rn, rp
        err['grad_H neg'], at['grad_H neg'] = m_neg.err, m_neg.at
        err['grad_H pos'], at['grad_H pos'] = m_pos.err, m_pos.at
        del neg, pos

    # ---- the fused H update, as the benchmarked step calls it --------------------------------------------------------
    H0 = H.clone(memory_format=torch.contiguous_format)
    nmf._update_H()                                                      # pylint: disable=protected-access
    torch.cuda.synchronize(dev)
    m_H = MaxRel()
    for s in dor.sample_chunks(N, dor.chunk_for(C, M, D, A)):
        m_H.add(H[s], dor.update_H(dor.f64(V[s]), W64, dor.f64(H0[s])), s)
    err['update_H'], at['update_H'] = m_H.err, m_H.at

    # ---- one benchmarked step: the graph replay of nmf._batch_step() from the start values ---------------------------
    step = nmf._batch_step()                                             # pylint: disable=protected-access
    H.copy_(H0)
    step()                                      # call 1 runs eagerly ...
    H.copy_(H0)
    W.copy_(W0)
    step()                                      # ... call 2 captures the iteration and replays the graph
    assert step._entry is not None              # pylint: disable=protected-access
    torch.cuda.synchronize(dev)
    m_sH = MaxRel()
    W1 = dor.mu_step(V, W64, H0, on_H=lambda s, H1: m_sH.add(H[s], H1, s))
    m_sW = MaxRel()
    m_sW.add(W, W1)
    err['step W'], at['step W'] = m_sW.err, m_sW.at
    err['step H'], at['step H'] = m_sH.err, m_sH.at

    del step, nmf, be, W, H, H0, V, W0, W64, W1
    gc.collect()
    torch.cuda.empty_cache()

    failed = []
    for key, e in err.items():
        limit = tol[key.split()[0]]
        ok = e <= limit
        failed += [] if ok else [key]
        print(f'{name}: {key:<11} max-rel {e:.2e}  tol {limit:.0e}  {"ok" if ok else "FAIL"}'
              + (f'  worst at {at[key]}' if key in at else ''))
    print(f'{name}: {time.perf_counter() - t_start:.1f} s')
    assert not failed, f'{name}: ' + ', '.join(f'{k} {err[k]:.2e} at {at.get(k)}' for k in failed)
