"""
Spatial (halo) sharding: ONE problem whose samples are too large - or too few - to shard over samples is cut along
the first shift axis ("rows": rows of an image, z-planes of a volume) and every rank owns a band of activation rows
(SURVEY 8 f4).  The derivation below indexes the first shift axis only; the trailing axes (one or two) ride along
unchanged, so the same code serves 1-D, 2-D and 3-D problems.

Derivation for the default mode ('valid', tnmf/backends/_Backend.py:60-73: T = D + A - 1, p = A_y - 1; 'full' is the mirror
image with the halos on the sample side, see `row_plan`).  Globally
    R[y]    = sum_ay W[ay] * H[y + p - ay]            R row y needs the activation rows [y, y + p]
    negH[t] = sum_ay W[ay] * V[t - p + ay]            activation row t needs the sample rows [t - p, t]
    negW[ay] = sum_t H[t] * V[t - p + ay]             a plain sum over activation rows
(tnmf/backends/NumPy.py:69-132).  Rank k owns the activation rows [t_k, t_{k+1}).  Its LOCAL problem is the ordinary
'valid' problem on the sample rows [Y0, Y1) = [max(0, t_k - p), min(D_y, t_{k+1})): the activation rows of that problem
are [Y0, Y1 + p) - the owned band plus up to p HALO rows on either side, which belong to the neighbours.  With true
values in the halos the local reconstruction IS the global one on [Y0, Y1), and the local H update is the global one on
every owned row (its window [t - p, t] lies inside [Y0, Y1)); the halo rows it also produces are wrong and are simply
overwritten by the next exchange.  The W gradient is linear in H, so correlating with a copy of H whose halo rows are
zero gives exactly this band's share of the sum; the shares are summed over the ranks like the sample shards' are.

Inhibition.  The lateral and cross-atom terms (tnmf/TransformInvariantNMF.py:253-269) add G = H convolved with the
inhibition kernels (zero boundary) and its sum over the atoms to the H update.  Along the sharded axis the kernel has
the radius r0 = inhibition_range[0]: G on activation row t needs the H rows [t - r0, t + r0].  The halo is therefore
h = max(p, r0) rows on either side (`row_plan(..., halo=h)`; the sample rows widen with it).  With true values in the
halos the band's G - and so the atom sum of G - on every OWNED row equals the global one: the zero boundary of the
band's convolution falls inside its halos, except at the global edges, where it is the global boundary too.

One iteration = exchange halos (h rows with each neighbour: the path's one real exchange step besides the W-gradient
sum) -> R -> H update -> exchange halos -> R' -> masked W gradient -> sum over ranks -> W update.  With three shift axes
`B200Ops` restricts the H update and the W gradient to the owned planes (tnmf_update_h_planes / tnmf_gradient_w_planes)
instead of updating halo planes the exchange overwrites and correlating with a zero-haloed copy of H.
The arithmetic comes from an `ops` provider: `B200Ops` (the CUDA kernels through B200_Backend) on the GPU box; the CPU
test drives the same class with the oracle as provider over gloo (tests/test_distributed_cpu.py).
"""
from typing import List, Optional, Tuple, Union

import numpy as np
import torch
import torch.distributed as dist

from .distributed import shard_bounds


def row_plan(t_rows: int, d_rows: int, p: int, world: int, rank: int, mode: str = 'valid',
             halo: Optional[int] = None) -> dict:
    """Bands of the activation rows: owned rows [t0, t1) of the global tensor, the sample rows [v0, v1) of the band's local
    problem, the global row h0 of the first LOCAL activation row, and - in local activation rows - where the owned band
    (`own`) and the halos (`lower`, `upper`) sit; `e_rows` = the local sample rows whose energy this rank adds up.
    `halo` = h >= p rows on either side (default p; wider for the inhibition terms, see the module docstring).

    'valid' (T = D + p): local problem = sample rows [max(0, t0 - h), min(D, t1 + h - p)), activation rows from the same
    row on, i.e. [max(0, t0 - h), min(T, t1 + h)).
    'full'  (T = D - p, R[y] needs the activation rows [y - p, y], activation row t the sample rows [t, t + p]): the owned
    band needs R on [t0, t1 + p), which needs the activation rows [t0 - p, t1 + p): local activation rows
    [h0, h1) = [max(0, t0 - h), min(T, t1 + h)), local sample rows [h0, h1 + p)."""
    if mode not in ('valid', 'full'):
        raise NotImplementedError(f"halo sharding is not defined for reconstruction mode '{mode}'")
    if t_rows != (d_rows + p if mode == 'valid' else d_rows - p):
        raise ValueError('activation and sample extents do not belong to this mode')
    h = p if halo is None else int(halo)
    if h < p:
        raise ValueError(f'a halo of {h} rows does not cover the atom ({p} rows)')
    if world > 1 and t_rows // world < max(h, 1):
        raise ValueError(f'{world} ranks leave bands of {t_rows // world} rows, thinner than the halo of {h} rows')
    t0, t1 = shard_bounds(t_rows, world, rank)
    if mode == 'valid':
        v0, v1 = max(0, t0 - h), min(d_rows, t1 + h - p)
        h0, h1 = v0, v1 + p
        e0, e1 = (min(d_rows, t0) if rank else 0), min(d_rows, t1)         # (the last rank: t1 = T > D)
    else:
        h0, h1 = max(0, t0 - h), min(t_rows, t1 + h)
        v0, v1 = h0, h1 + p
        e0, e1 = t0, (t1 if rank < world - 1 else d_rows)
    return dict(t0=t0, t1=t1, v0=v0, v1=v1, h0=h0, own=(t0 - h0, t1 - h0), lower=(0, t0 - h0), upper=(t1 - h0, h1 - h0),
                e_rows=(e0 - v0, e1 - v0))


class RowSharding:
    """The halo exchange and the two sums of the row-sharded iteration (torch.distributed; NCCL or gloo)."""

    def __init__(self, group=None):
        if not (dist.is_available() and dist.is_initialized()):
            raise RuntimeError('row sharding needs an initialised torch.distributed process group')
        self.group = group
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        self.via_host = 'nccl' not in str(dist.get_backend(group)).lower()     # gloo moves host tensors
        self.exchanges = 0

    def _peer(self, r: int) -> int:
        return r if self.group is None else dist.get_global_rank(self.group, r)

    def exchange_halos(self, H: torch.Tensor, plan: dict, h: int) -> None:
        """Fill the halo rows of the local activation tensor H[n, m, rows, ...] from the neighbours' owned rows and
        send them ours: the lower halo of rank k+1 is our last h owned rows, the upper halo of rank k-1 our first
        (bands are at least h rows thick, `row_plan`)."""
        (o0, o1), (l0, l1), (u0, u1) = plan['own'], plan['lower'], plan['upper']
        ops, recvs = [], []

        def stage(t):
            t = t.contiguous()
            return t.cpu() if self.via_host else t

        if self.rank > 0 and l1 > l0:           # neighbour below: it needs our first rows, we need its last h
            n_up = min(h, o1 - o0)
            send = stage(H[:, :, o0:o0 + n_up])
            recv = torch.empty_like(stage(H[:, :, l0:l1]))
            ops += [dist.P2POp(dist.isend, send, self._peer(self.rank - 1), self.group),
                    dist.P2POp(dist.irecv, recv, self._peer(self.rank - 1), self.group)]
            recvs.append((recv, (l0, l1)))
        if self.rank < self.world - 1 and u1 > u0:
            send = stage(H[:, :, o1 - h:o1])
            recv = torch.empty_like(stage(H[:, :, u0:u1]))
            ops += [dist.P2POp(dist.isend, send, self._peer(self.rank + 1), self.group),
                    dist.P2POp(dist.irecv, recv, self._peer(self.rank + 1), self.group)]
            recvs.append((recv, (u0, u1)))
        if ops:
            for req in dist.batch_isend_irecv(ops):
                req.wait()
            for recv, (a, b) in recvs:
                H[:, :, a:b].copy_(recv.to(H.device))
        self.exchanges += 1

    def sum_(self, t: torch.Tensor) -> torch.Tensor:
        if self.world > 1:
            if self.via_host and t.is_cuda:
                h = t.cpu()
                dist.all_reduce(h, group=self.group)
                t.copy_(h)
            else:
                dist.all_reduce(t, group=self.group)
        return t


class B200Ops:
    """The arithmetic of one band on the CUDA kernels (B200_Backend on the band's local problem).

    With three shift axes the H update and the W gradient run on the owned planes only (`plane_window`, default True:
    tnmf_update_h_planes / tnmf_gradient_w_planes); otherwise the H update also produces the halo rows, which the next
    exchange overwrites, and the W gradient correlates with `H_own`, a copy of H whose halo rows are zero.
    `plane_window=False` keeps the second form for volumes too (diagnostics: it measures what the window saves)."""

    def __init__(self, reconstruction_mode: str = 'valid', plane_window: bool = True, **backend_kwargs):
        from .backend import B200_Backend
        self.be = B200_Backend(reconstruction_mode=reconstruction_mode, **backend_kwargs)
        self.plane_window = bool(plane_window)
        self.windowed = False
        self.V = None
        self.H_own = None

    def setup(self, V_local, atom_shape, n_atoms, W0, H0):
        state = np.random.get_state()
        W, H = self.be.initialize(V_local, atom_shape, n_atoms, None, tuple(range(-len(atom_shape), 0)))
        np.random.set_state(state)              # the band's own draw is discarded: W0 / H0 come from the caller
        self.V = V_local
        W.copy_(torch.as_tensor(W0).to(W.device, W.dtype))
        H.copy_(torch.as_tensor(H0).to(H.device, H.dtype))
        self.grad = torch.empty((2, *W.shape), dtype=W.dtype, device=W.device)
        self.windowed = self.plane_window and len(atom_shape) == 3
        if not self.windowed:
            pad = self.be._h_padding(H.shape)   # pylint: disable=protected-access  (same padded row pitch as H)
            self.H_own = torch.zeros((*H.shape[:-1], H.shape[-1] + pad), dtype=H.dtype, device=H.device)[..., :H.shape[-1]]
        return W, H

    def update_H(self, W, H, sparsity, eps, own: Optional[Tuple[int, int]] = None, inhibition: float = 0.,
                 cross_inhibition: float = 0., inhibition_kernels=None):
        """The fused H update of the band; `own` (passed while `windowed`): write the owned activation rows only."""
        self.be.update_H(self.V, W, H, slice(None), sparsity, inhibition, cross_inhibition, inhibition_kernels, eps,
                         planes=own if self.windowed else None)

    def gradient_W(self, W, H, own: Tuple[int, int]) -> torch.Tensor:
        """Stacked (neg, pos) of the W gradient over the OWNED activation rows: R from the full local H (true halos),
        the correlation with the owned rows only (a plane window, or a copy of H whose halo rows are zero)."""
        if self.windowed:
            return self.be.gradient_W(self.V, W, H, slice(None), self.grad, planes=own)
        self.H_own.zero_()
        self.H_own[:, :, own[0]:own[1]] = H[:, :, own[0]:own[1]]
        return self.be.gradient_W(self.V, W, self.H_own, slice(None), self.grad, H_for_R=H)

    def apply_W(self, W, grad, eps):
        self.be.apply_W_update(W, grad, eps)

    def energy_rows(self, W, H, rows: Tuple[int, int]) -> torch.Tensor:
        R = self.be.reconstruct(W, H)
        V = self.be._device_V(self.V)           # pylint: disable=protected-access
        d = (V[:, :, rows[0]:rows[1]].double() - R[:, :, rows[0]:rows[1]].double())
        return 0.5 * (d * d).sum()


class RowShardedNMF:
    r"""
    Batch multiplicative updates (tnmf/TransformInvariantNMF.py:282-348) with the activation rows sharded over the ranks.

    Every rank passes the same global V (only its band of sample rows is kept on the device).  `W` is identical on all
    ranks, `H` is the rank's band of activation rows [t0, t1).  Supported: one to three shift axes (the bands cut the
    first: rows of an image, z-planes of a volume), 'valid' and 'full' modes, sparsity, lateral and cross-atom
    inhibition.  `inhibition_range` has the meaning and default of `TransformInvariantNMF`'s (a - 1 per axis); the halo
    is max(A_0 - 1, inhibition_range[0]) rows, whether or not a fit uses the inhibition terms.
    """

    def __init__(self, n_atoms: int, atom_shape: Tuple[int, ...], process_group=None, ops=None,
                 reconstruction_mode: str = 'valid', inhibition_range: Union[int, Tuple[int, ...], None] = None,
                 **backend_kwargs):
        self.n_atoms, self.atom_shape = int(n_atoms), tuple(int(a) for a in atom_shape)
        self.mode = reconstruction_mode
        if self.mode not in ('valid', 'full'):
            raise NotImplementedError(f"halo sharding is not defined for reconstruction mode '{self.mode}'")
        if inhibition_range is None:
            inhibition_range = tuple(a - 1 for a in self.atom_shape)         # just covers the atom
        elif isinstance(inhibition_range, int):
            inhibition_range = (inhibition_range,) * len(self.atom_shape)
        self.inhibition_range = tuple(int(r) for r in inhibition_range)
        if len(self.inhibition_range) != len(self.atom_shape):
            raise ValueError('inhibition_range needs one radius per shift axis')
        self.inhibition_kernels = tuple(1 - (np.arange(-r, r + 1) / (r + 1)) ** 2 for r in self.inhibition_range)
        self.halo = max(self.atom_shape[0] - 1, self.inhibition_range[0])
        self.eps = 1.e-9
        self.sharding = RowSharding(process_group)
        self.ops = ops if ops is not None else B200Ops(reconstruction_mode=self.mode, **backend_kwargs)
        self.plan = None
        self._W = self._H = None

    def initialize(self, V) -> None:
        """Same seeded start as a single-process fit (tnmf/backends/_Backend.py:83-98: H drawn first, then W, float64
        draws cast to V.dtype): every rank draws the full tensors and keeps its band."""
        V = np.asarray(V)
        sh, p = self.sharding, self.atom_shape[0] - 1
        sign = 1 if self.mode == 'valid' else -1
        t_shape = tuple(d + sign * (a - 1) for d, a in zip(V.shape[2:], self.atom_shape))
        self.plan = row_plan(t_shape[0], V.shape[2], p, sh.world, sh.rank, self.mode, self.halo)
        H0 = np.asarray(1 - np.random.rand(V.shape[0], self.n_atoms, *t_shape), dtype=V.dtype)
        W0 = np.asarray(1 - np.random.rand(self.n_atoms, V.shape[1], *self.atom_shape), dtype=V.dtype)
        W0 /= W0.sum(axis=tuple(range(2, W0.ndim)), keepdims=True)
        if sh.world > 1:                        # one dictionary for all ranks, whatever the state of their generators
            box = [W0]
            dist.broadcast_object_list(box, src=sh._peer(0), group=sh.group)      # pylint: disable=protected-access
            W0 = box[0]
        pl = self.plan
        V_local = np.ascontiguousarray(V[:, :, pl['v0']:pl['v1']])
        H_local = np.ascontiguousarray(H0[:, :, pl['h0']:pl['h0'] + pl['upper'][1]])
        self._W, self._H = self.ops.setup(V_local, self.atom_shape, self.n_atoms, W0, H_local)

    def step(self, sparsity: float = 0., inhibition_strength: float = 0., cross_atom_inhibition_strength: float = 0.) -> None:
        sh, pl = self.sharding, self.plan
        # the ops' update_H(W, H, sparsity, eps) takes the optional terms as keywords, and only those in use
        kw = {}
        if getattr(self.ops, 'windowed', False):
            kw['own'] = pl['own']
        if inhibition_strength > 0:
            kw['inhibition'] = float(inhibition_strength)
        if cross_atom_inhibition_strength > 0:
            kw['cross_inhibition'] = float(cross_atom_inhibition_strength)
        if inhibition_strength > 0 or cross_atom_inhibition_strength > 0:
            kw['inhibition_kernels'] = self.inhibition_kernels
        sh.exchange_halos(self._H, pl, self.halo)
        self.ops.update_H(self._W, self._H, sparsity, self.eps, **kw)
        sh.exchange_halos(self._H, pl, self.halo)
        grad = sh.sum_(self.ops.gradient_W(self._W, self._H, pl['own']))
        self.ops.apply_W(self._W, grad, self.eps)

    def fit(self, V, n_iterations: int = 1000, sparsity_H: float = 0., inhibition_strength: float = 0.,
            cross_atom_inhibition_strength: float = 0., progress_callback=None) -> None:
        assert np.all(np.asarray(V) >= 0) and sparsity_H >= 0
        assert inhibition_strength >= 0 and cross_atom_inhibition_strength >= 0
        self.initialize(V)
        for iteration in range(n_iterations):
            self.step(sparsity_H, inhibition_strength, cross_atom_inhibition_strength)
            if progress_callback is not None and not progress_callback(self, iteration):
                break

    def energy(self) -> float:
        """0.5 * ||V - R||^2 of the whole problem: every rank sums a disjoint band of sample rows."""
        sh, pl = self.sharding, self.plan
        sh.exchange_halos(self._H, pl, self.halo)
        e = self.ops.energy_rows(self._W, self._H, pl['e_rows'])
        e = torch.as_tensor(e, dtype=torch.float64).reshape(1).clone()
        return float(sh.sum_(e).item())

    @property
    def W(self) -> np.ndarray:
        return np.ascontiguousarray(torch.as_tensor(self._W).detach().cpu().numpy())

    @property
    def H(self) -> np.ndarray:
        """The owned band: rows [plan['t0'], plan['t1']) of the global activation tensor."""
        a, b = self.plan['own']
        return np.ascontiguousarray(torch.as_tensor(self._H)[:, :, a:b].detach().cpu().numpy())

    def gather_H(self) -> Optional[np.ndarray]:
        """The global activation tensor on rank 0 (None elsewhere); for tests and small problems."""
        sh = self.sharding
        mine = torch.from_numpy(self.H)
        bands: List[Optional[torch.Tensor]] = [None] * sh.world
        dist.all_gather_object(bands, mine, group=sh.group)
        return np.concatenate([b.numpy() for b in bands], axis=2) if sh.rank == 0 else None
