"""
Halo (row) sharding with three shift axes and with the inhibition terms, on the CPU: `gloo` ranks on 127.0.0.1 drive
`tnmf_b200.halo.RowShardedNMF` with the float64 oracle as the per-band arithmetic (the role B200Ops plays on the GPU).

The halo is h = max(p, inhibition_range[0]) rows of the first shift axis (z-planes of a volume); with true values in the
halos every band's H update, inhibition terms and W-gradient share on its owned rows equal the global ones, so the
sharded fit must equal the single-process oracle fit up to summation order.
"""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import tnmf_oracle as orc


class InhibitionOracleOps:
    """The CPU oracle as RowShardedNMF's arithmetic provider, with the optional inhibition keywords of `update_H`."""

    def __init__(self, mode='valid'):
        self.mode = mode

    def setup(self, V_local, atom_shape, n_atoms, W0, H0):
        self.V = np.array(V_local, dtype=np.float64)
        return torch.from_numpy(np.array(W0, dtype=np.float64)), torch.from_numpy(np.array(H0, dtype=np.float64))

    def update_H(self, W, H, sparsity, eps, inhibition=0., cross_inhibition=0., inhibition_kernels=None):
        Hn = H.numpy()
        neg, pos = orc.reconstruction_gradient_H(self.V, W.numpy(), Hn, self.mode)
        if inhibition > 0 or cross_inhibition > 0:          # tnmf/TransformInvariantNMF.py:253-269 on the whole band
            G = orc.convolve_multi_1d(Hn, inhibition_kernels, tuple(range(-(Hn.ndim - 2), 0)))
            if inhibition > 0:
                tmp = G - Hn
                tmp *= inhibition
                pos += tmp
            if cross_inhibition > 0:
                tmp = G.sum(axis=1, keepdims=True)
                tmp = -G + tmp
                tmp *= cross_inhibition / (Hn.shape[1] - 1)
                pos += tmp
        orc.multiplicative_update(Hn, neg, pos, sparsity)

    def gradient_W(self, W, H, own):
        Hn, Wn = H.numpy(), W.numpy()
        R = orc.reconstruct(Wn, Hn, self.mode)
        H_own = np.zeros_like(Hn)
        H_own[:, :, own[0]:own[1]] = Hn[:, :, own[0]:own[1]]
        Hp = orc.pad_activations(H_own, Wn.shape[2:], self.mode)
        return torch.from_numpy(np.stack([orc._correlate_with_activations(self.V, Hp, Wn.shape[2:]),
                                          orc._correlate_with_activations(R, Hp, Wn.shape[2:])]))

    def apply_W(self, W, grad, eps):
        g = grad.numpy()
        orc.multiplicative_update(W.numpy(), g[0].copy(), g[1].copy(), normalization_axes=tuple(range(2, W.dim())))

    def energy_rows(self, W, H, rows):
        R = orc.reconstruct(W.numpy(), H.numpy(), self.mode)
        d = self.V[:, :, rows[0]:rows[1]] - R[:, :, rows[0]:rows[1]]
        return torch.tensor(0.5 * np.sum(d * d))


def _free_port():
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        return s.getsockname()[1]


def _rank_main(rank, world, port, V, atoms, atom_shape, mode, inhibition_range, iters, kw, out):
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        from tnmf_b200.halo import RowShardedNMF
        np.random.seed(31)
        nmf = RowShardedNMF(atoms, atom_shape, ops=InhibitionOracleOps(mode), reconstruction_mode=mode,
                            inhibition_range=inhibition_range)
        energies = []
        nmf.fit(V, n_iterations=iters, progress_callback=lambda m, i: energies.append(m.energy()) or True, **kw)
        out[rank] = (nmf.W, nmf.gather_H(), energies, nmf.plan, nmf.halo)
    finally:
        dist.destroy_process_group()


def _plans(t, d, p, world, mode, halo):
    from tnmf_b200.halo import row_plan
    return [row_plan(t, d, p, world, r, mode, halo) for r in range(world)]


@pytest.mark.parametrize('mode', ['valid', 'full'])
def test_row_plan_with_a_wider_halo(mode):
    for d, a, world, h in ((30, 3, 2, 4), (30, 3, 3, 5), (41, 5, 4, 6), (24, 1, 3, 2), (40, 4, 2, 3)):
        p = a - 1
        t = d + p if mode == 'valid' else d - p
        plans = _plans(t, d, p, world, mode, h)
        assert plans[0]['t0'] == 0 and plans[-1]['t1'] == t                       # the bands tile the activation rows
        assert all(x['t1'] == y['t0'] for x, y in zip(plans, plans[1:]))
        for pl in plans:
            assert pl['lower'][1] - pl['lower'][0] == min(h, pl['t0'])             # h rows, fewer at the global edges
            assert pl['upper'][1] - pl['upper'][0] == min(h, t - pl['t1'])
            assert pl['h0'] == pl['t0'] - (pl['lower'][1] - pl['lower'][0])
            assert pl['own'] == (pl['t0'] - pl['h0'], pl['t1'] - pl['h0'])
            # the band is an ordinary problem of the same mode: T_local = D_local +- p
            assert pl['upper'][1] == (pl['v1'] - pl['v0']) + (p if mode == 'valid' else -p)
            assert 0 <= pl['v0'] < pl['v1'] <= d
        # the energy rows partition the sample rows
        e = [(pl['e_rows'][0] + pl['v0'], pl['e_rows'][1] + pl['v0']) for pl in plans]
        assert e[0][0] == 0 and e[-1][1] == d and all(x[1] == y[0] for x, y in zip(e, e[1:]))
        assert all(pl['v0'] <= lo <= hi <= pl['v1'] for pl, (lo, hi) in zip(plans, e))
    # the default halo is p: the plans of the narrower call are unchanged
    t = 27 if mode == 'valid' else 21
    assert _plans(t, 24, 3, 3, mode, None) == _plans(t, 24, 3, 3, mode, 3)


def test_row_plan_rejects_bands_thinner_than_the_halo():
    from tnmf_b200.halo import row_plan
    with pytest.raises(ValueError):
        row_plan(20, 18, 2, 4, 0, 'valid', 6)                  # bands of 5 rows, halo of 6
    with pytest.raises(ValueError):
        row_plan(14, 16, 2, 3, 1, 'full', 5)                   # bands of 4 rows, halo of 5
    with pytest.raises(ValueError):
        row_plan(20, 18, 2, 2, 0, 'valid', 1)                  # a halo narrower than the atom
    row_plan(20, 18, 2, 4, 0, 'valid', 5)                      # bands of 5 rows, halo of 5: fine


def _run(world, V, atoms, atom_shape, mode, inhibition_range, iters, kw):
    ctx = mp.get_context('spawn')
    with ctx.Manager() as mgr:
        out = mgr.dict()
        mp.spawn(_rank_main, args=(world, _free_port(), V, atoms, atom_shape, mode, inhibition_range, iters, kw, out),
                 nprocs=world, join=True)
        return [out[r] for r in range(world)]


_KW = dict(sparsity_H=0.05, inhibition_strength=0.2, cross_atom_inhibition_strength=0.1)


@pytest.mark.parametrize('mode', ['valid', 'full'])
@pytest.mark.parametrize('world,shape,atom_shape,inhibition_range', [
    (2, (2, 2, 14, 6, 5), (3, 2, 2), None),                    # volumes: halo = p = 2 planes
    (3, (1, 1, 17, 5, 6), (3, 3, 2), (3, 1, 2)),               # halo = r0 = 3 planes > p
    (2, (2, 1, 26, 9), (3, 3), (4, 1)),                        # 2-D, halo = r0 = 4 rows > p
])
def test_row_sharded_fit_with_inhibition_equals_single_process(world, shape, atom_shape, inhibition_range, mode):
    rng = np.random.default_rng(7)
    V = rng.random(shape)
    iters, atoms = 6, 3
    np.random.seed(31)
    ref = orc.OracleNMF(n_atoms=atoms, atom_shape=atom_shape, inhibition_range=inhibition_range,
                        reconstruction_mode=mode)
    e_ref = []
    ref.fit_batch(V, n_iterations=iters, progress_callback=lambda m, i: e_ref.append(float(m.energy())) or True, **_KW)
    results = _run(world, V, atoms, atom_shape, mode, inhibition_range, iters, _KW)
    W0, H0, e0, _, halo = results[0]
    r0 = (atom_shape[0] - 1) if inhibition_range is None else inhibition_range[0]
    assert halo == max(atom_shape[0] - 1, r0)
    assert H0.shape == ref.H.shape
    assert np.allclose(e0, e_ref, rtol=1e-9)
    assert np.allclose(W0, ref.W, rtol=1e-9, atol=1e-14)
    assert np.allclose(H0, ref.H, rtol=1e-9, atol=1e-14)
    for W, _, e, _, _ in results[1:]:
        assert np.array_equal(W, W0) and np.allclose(e, e0, rtol=1e-12)


def _narrow_rank_main(rank, world, port, V, out):
    """_rank_main with the halo held at p rows whatever the inhibition range."""
    from tnmf_b200 import halo as halo_mod
    wide = halo_mod.RowShardedNMF.__init__

    def narrow(self, *a, **k):
        wide(self, *a, **k)
        self.halo = self.atom_shape[0] - 1
    halo_mod.RowShardedNMF.__init__ = narrow
    _rank_main(rank, world, port, V, 3, (3, 3), 'valid', (4, 1), 3, dict(inhibition_strength=0.5), out)


def test_a_halo_of_p_misses_the_inhibition_of_a_wider_range():
    """The widening is needed: with inhibition_range[0] > p and the halo held at p rows, the bands' G differs from the
    global G next to the band edges and the sharded fit departs from the single-process one."""
    V = np.random.default_rng(7).random((2, 1, 26, 9))
    np.random.seed(31)
    ref = orc.OracleNMF(n_atoms=3, atom_shape=(3, 3), inhibition_range=(4, 1))
    ref.fit_batch(V, n_iterations=3, inhibition_strength=0.5)
    W, _, _, _, halo = _run(2, V, 3, (3, 3), 'valid', (4, 1), 3, dict(inhibition_strength=0.5))[0]
    assert halo == 4 and np.allclose(W, ref.W, rtol=1e-9, atol=1e-14)
    ctx = mp.get_context('spawn')
    with ctx.Manager() as mgr:
        out = mgr.dict()
        mp.spawn(_narrow_rank_main, args=(2, _free_port(), V, out), nprocs=2, join=True)
        W_narrow = out[0][0]
    assert not np.allclose(W_narrow, ref.W, rtol=1e-9, atol=1e-14)
