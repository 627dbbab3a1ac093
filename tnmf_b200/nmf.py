"""
Host-side driver of the B200 backend: the same public surface as the reference facade
`tnmf.TransformInvariantNMF` (tnmf/TransformInvariantNMF.py:58-531) - constructor arguments, `fit`,
`fit_batch`, `fit_minibatches`, `fit_stream`, the `W`/`H`/`V`/`R` properties, `R_partial`, the
`MiniBatchAlgorithm` enum and the `progress_callback` protocol - so that user code switches by changing the
import (or, with the reference installed, by registering `B200_Backend` in its backend map; INTEGRATION.md).

What differs is where the arithmetic runs: every update is a short sequence of stream-ordered kernel launches
on device-resident W/H/V (tnmf_b200.backend), the facade's multiplicative-update arithmetic is fused into the
kernels, nothing synchronises with the host inside the iteration loop unless the caller asks for the energy,
and samples can be sharded over the GPUs of a box (tnmf_b200.distributed).
"""
import logging
from enum import Enum
from itertools import count, islice
from typing import Callable, Iterable, Iterator, List, Optional, Tuple, Union

import numpy as np
import torch

from .backend import B200_Backend
from .distributed import SampleSharding, equal_batch_slices

sliceNone = slice(None)


class MiniBatchAlgorithm(Enum):
    """Minibatch schedules of Serizel et al. 2016, numbered as in tnmf/TransformInvariantNMF.py:47-55."""
    Cyclic_MU = 4
    ASG_MU = 5
    GSG_MU = 6
    ASAG_MU = 7
    GSAG_MU = 8


class TransformInvariantNMF:
    r"""
    Shift-invariant non-negative matrix factorisation  V[n,c,:] ~ sum_m W[m,c,:] * H[n,m,:]  by multiplicative
    updates on the Frobenius energy or the Kullback-Leibler divergence, on one or several B200 GPUs.

    Parameters (first six as in tnmf/TransformInvariantNMF.py:142-151)
    ----------
    n_atoms, atom_shape, inhibition_range, backend, logger, verbose
        `backend` must be 'b200' (this package ships exactly one arithmetic provider).
    distributed : None (default: on iff torch.distributed is initialised) or bool
        Shard the samples over the ranks of `process_group`; see tnmf_b200.distributed.
    input_is_local_shard : bool, default False
        False: every rank passes the same global V and keeps its contiguous block of samples.
        True: every rank passes only its own samples.
    equal_shards : bool, default False
        With `input_is_local_shard`: the caller guarantees that all ranks pass equally many samples on every fit
        (checked once per shape), which removes the per-fit exchange of the sample counts.
    fused : bool, default True
        False drives the backend through the reference interface only (reconstruction_gradient_H/W + the
        update arithmetic as tensor operations), i.e. exactly the call sequence of the stock facade.
    peer_exchange : bool, default True
        Sharded runs over NCCL only: sum the W gradient over the ranks inside the W-update kernel, through NVLink peer
        memory (`tnmf_allreduce_update_w`), instead of an NCCL all-reduce between the W gradient and the W update.  Falls
        back to the all-reduce where peer memory cannot be mapped.
    cuda_graph : bool, default True
        Batch algorithm only: after one eager iteration the kernel launches of an iteration are captured into CUDA
        graphs (everything up to the all-reduce of the W gradient, and the W update after it) and replayed, which
        removes the host-side launch cost (about 1 ms of a 4.6 ms iteration on cfg2).  Results are bit-identical.
    divergence : 'frobenius' (default) | 'kl'
        The loss the updates minimise: 0.5*||V - R||^2, or the generalised Kullback-Leibler divergence
        D(V||R) = sum V log(V/R) - V + R (Lee & Seung's KL updates; DESIGN.md §3.11), the usual loss for counts and
        magnitudes.  `energy_device()` and the energy of the progress log report the chosen loss.  'kl' needs
        `fused=True`.
    **kwargs : forwarded to `B200_Backend` (reconstruction_mode, device, init, kernel_path)
    """

    def __init__(self, n_atoms: int, atom_shape: Tuple[int, ...], inhibition_range: Union[int, Tuple[int, ...]] = None,
                 backend: str = 'b200', logger: logging.Logger = None, verbose: int = 0,
                 distributed: Optional[bool] = None, process_group=None, input_is_local_shard: bool = False,
                 fused: bool = True, cuda_graph: bool = True, equal_shards: bool = False, peer_exchange: bool = True,
                 divergence: str = 'frobenius', **kwargs):
        if divergence not in ('frobenius', 'kl'):
            raise ValueError(f'divergence must be "frobenius" or "kl" (got {divergence!r})')
        if divergence == 'kl' and not fused:
            raise ValueError('divergence="kl" needs fused=True (the unfused mode is the Frobenius call sequence of the '
                             'reference facade)')
        self._divergence = divergence
        # the backend hears of the divergence only when it is not the default
        self._div_kw = {} if divergence == 'frobenius' else {'divergence': divergence}
        self.atom_shape = tuple(atom_shape)
        if inhibition_range is None:
            self._inhibition_range = tuple(a - 1 for a in self.atom_shape)   # just covers the atom
        elif isinstance(inhibition_range, int):
            self._inhibition_range = (inhibition_range,) * len(self.atom_shape)
        else:
            self._inhibition_range = tuple(inhibition_range)
        assert len(self._inhibition_range) == len(self.atom_shape)
        # 1 - (j/(r+1))^2, j = -r..r   (tnmf/TransformInvariantNMF.py:163)
        self._inhibition_kernels_1D = tuple(1 - (np.arange(-r, r + 1) / (r + 1)) ** 2 for r in self._inhibition_range)
        self.n_atoms = n_atoms
        self._axes_W_normalization = tuple(range(-len(self.atom_shape), 0))
        self.eps = 1.e-9

        if isinstance(backend, str):
            if backend.lower() != 'b200':
                raise ValueError(f'tnmf_b200 provides the "b200" backend only (got "{backend}"); the CPU backends live '
                                 f'in the reference package')
            self._backend = B200_Backend(**kwargs)
        else:
            self._backend = backend
        self._fused = bool(fused)
        self._cuda_graph = bool(cuda_graph)
        self._sharding = SampleSharding(process_group, distributed)
        self._input_is_local = bool(input_is_local_shard)
        self._equal_shards = bool(equal_shards)
        self._counts_for = None
        self._use_peer = bool(peer_exchange) and self._fused
        self._peer = None           # PeerExchange of the current dictionary shape (None: NCCL all-reduce)
        self._peer_for = None
        self._step_cache = None     # (key, _GraphedStep): CUDA graphs survive across fits while every buffer stays put

        self._logger = logger if logger is not None else logging.getLogger(self.__class__.__name__)
        self._logger.setLevel([logging.ERROR, logging.WARNING, logging.INFO, logging.DEBUG][verbose])
        self._logger.debug('Using b200 backend.')

        self._W = None
        self._H = None
        self._V = None
        self._n_global = None
        self._n_local_max = None
        self._grad = None           # stacked (neg, pos) W-gradient buffer, the all-reduce payload
        self._R_current = False     # the backend's R buffer holds reconstruct(W, H) of the current W and H (left there by
                                    # an energy evaluation): the next H update starts from it instead of reconstructing
        self._shuffle_idx = None    # kept for interface parity; the reference never shuffles (SURVEY App. B.2)

    # ---------------------------------------------------------------------------------------------
    # results
    # ---------------------------------------------------------------------------------------------
    @property
    def W(self) -> np.ndarray:
        return self._backend.to_ndarray(self._W)

    @property
    def H(self) -> np.ndarray:
        """Activations (of this rank's samples when sharded)."""
        return self._backend.to_ndarray(self._H)

    @property
    def V(self):
        return self._V

    @property
    def R(self) -> np.ndarray:
        return self._backend.to_ndarray(self._reconstruct())

    def R_partial(self, i_atom: int) -> np.ndarray:
        return self._backend.to_ndarray(self._backend.partial_reconstruct(self._W, self._H, i_atom))

    @property
    def W_device(self) -> torch.Tensor:
        return self._W

    @property
    def H_device(self) -> torch.Tensor:
        return self._H

    def _reconstruct(self):
        return self._backend.reconstruct(self._W, self._H)

    def energy_device(self) -> torch.Tensor:
        """0.5*||V-R||^2 (with divergence='kl': D(V||R)) over all samples of all ranks as a device-resident double (no host
        sync).  The reconstruction it
        is computed from stays in the backend's R buffer: it is the one the next H update opens with, so an energy read
        in every iteration (a progress callback, the INFO log line of tnmf/TransformInvariantNMF.py:346) costs no third
        reconstruction per iteration."""
        e = self._backend.energy(self._V, self._W, self._H, keep_R=self._fused, **self._div_kw)
        self._R_current = self._fused
        return self._sharding.sum_scalar(e)

    def _energy_function(self) -> float:
        return float(self.energy_device().item())

    # ---------------------------------------------------------------------------------------------
    # updates
    # ---------------------------------------------------------------------------------------------
    def _multiplicative_update(self, arr, neg, pos, sparsity: float = 0., normalization_axes=None):
        """Unfused form, operation for operation as tnmf/TransformInvariantNMF.py:217-238."""
        assert sparsity >= 0
        regularization = self.eps
        if sparsity > 0:
            regularization += sparsity
        pos += regularization
        arr *= neg
        arr /= pos
        if normalization_axes is not None:
            self._backend.normalize(arr, axis=normalization_axes)

    def _update_H(self, s: slice = sliceNone, sparsity: float = 0., inhibition: float = 0., cross_inhibition: float = 0.,
                  reuse_R: bool = False):
        self._R_current = False
        if self._fused:
            self._backend.update_H(self._V, self._W, self._H, s, sparsity, inhibition, cross_inhibition,
                                   self._inhibition_kernels_1D, self.eps, reuse_R=reuse_R and s is sliceNone,
                                   **self._div_kw)
            return
        # reference call sequence, tnmf/TransformInvariantNMF.py:246-271
        neg, pos = self._backend.reconstruction_gradient_H(self._V, self._W, self._H, s)
        assert neg.shape == self._H[s].shape and pos.shape == self._H[s].shape
        if inhibition > 0 or cross_inhibition > 0:
            axes = range(-len(self.atom_shape), 0)
            g = self._backend.convolve_multi_1d(self._H[s], self._inhibition_kernels_1D, axes)
            if inhibition > 0:
                tmp = g - self._H[s]
                tmp *= inhibition
                pos += tmp
            if cross_inhibition > 0:
                tmp = g.sum(dim=1, keepdim=True)
                tmp = -g + tmp
                tmp *= cross_inhibition / (self.n_atoms - 1)
                pos += tmp
        self._multiplicative_update(self._H[s], neg, pos, sparsity=sparsity)

    def _gradient_W(self, s: slice = sliceNone, reduce: bool = True) -> torch.Tensor:
        """Stacked (neg, pos) of the W gradient on local samples s, summed over ranks when `reduce`."""
        if self._fused:
            grad = self._backend.gradient_W(self._V, self._W, self._H, s, self._grad, **self._div_kw)
        else:
            neg, pos = self._backend.reconstruction_gradient_W(self._V, self._W, self._H, s)
            assert neg.shape == self._W.shape and pos.shape == self._W.shape
            self._grad[0].copy_(neg)
            self._grad[1].copy_(pos)
            grad = self._grad
        return self._sharding.sum_gradient(grad) if reduce else grad

    def _apply_W(self, grad: torch.Tensor):
        self._R_current = False
        if self._fused:
            self._backend.apply_W_update(self._W, grad, self.eps)
        else:
            self._multiplicative_update(self._W, grad[0].clone(), grad[1].clone(),
                                        normalization_axes=self._axes_W_normalization)

    def _reduce_apply_W(self, grad: torch.Tensor):
        """Sum `grad` over the ranks and apply the W update: one kernel over NVLink peer memory, or all-reduce + update."""
        if self._peer is not None:
            self._R_current = False
            self._backend.allreduce_update_W(self._W, grad, self._peer, self.eps)
        else:
            self._apply_W(self._sharding.sum_gradient(grad))

    def _update_W(self, s: slice = sliceNone):
        self._reduce_apply_W(self._gradient_W(s, reduce=False))

    # ---------------------------------------------------------------------------------------------
    # initialisation
    # ---------------------------------------------------------------------------------------------
    def _assert_non_negative(self):
        """The facade's `assert V.min() >= 0` (tnmf/TransformInvariantNMF.py:326,404), evaluated on the device copy of this
        rank's samples right after the upload was queued: a pass over a 50 MB host batch costs the host 5-30 ms (and a
        single-threaded one under torchrun), the device 10 us."""
        assert bool((self._backend.min_of_V() >= 0).item()), 'V must be non-negative'

    def _initialize_matrices(self, V, keep_W: bool):
        sh = self._sharding
        if not isinstance(V, (np.ndarray, torch.Tensor)):
            V = np.asarray(V)
        self._V = V
        sample_range = None
        if sh.is_sharded and not self._input_is_local:
            sample_range = sh.bounds(V.shape[0])
            self._n_global = int(V.shape[0])
            self._n_local_max = sh.max_local(V.shape[0])
        elif sh.is_sharded:
            # every rank passes its own samples: the global count and the largest shard need one exchange.  It is
            # cached while the caller promises equal shards (`equal_shards=True`: streams of equally sized subsamples)
            # - the two collectives and their host read-back are the only host synchronisation of a fit.
            if not (self._equal_shards and self._counts_for == int(V.shape[0])):
                counts = torch.tensor([V.shape[0], -V.shape[0]], dtype=torch.int64, device=self._backend.device)
                torch.distributed.all_reduce(counts, op=torch.distributed.ReduceOp.MAX, group=sh.group)
                n_max, n_min = int(counts[0].item()), -int(counts[1].item())
                if self._equal_shards and n_max != n_min:
                    raise ValueError(f'equal_shards=True, but the ranks hold between {n_min} and {n_max} samples')
                n = torch.tensor([V.shape[0]], dtype=torch.int64, device=self._backend.device)
                sh.sum_scalar(n)
                self._n_global, self._n_local_max = int(n.item()), n_max
                self._counts_for = int(V.shape[0])
        else:
            self._n_global = int(V.shape[0])
            self._n_local_max = int(V.shape[0])
        fresh_W = not (keep_W and self._W is not None)
        self._R_current = False
        self._W, self._H = self._backend.initialize(V, self.atom_shape, self.n_atoms, None if fresh_W else self._W,
                                                    self._axes_W_normalization, sample_range=sample_range)
        if sample_range is not None:
            self._V = V[sample_range[0]:sample_range[1]]
            self._backend._V_src = self._V          # pylint: disable=protected-access
        if fresh_W and sh.is_sharded:
            # every rank must start from the same dictionary, whatever the state of its random generator
            sh.broadcast(self._W, 0)
        if self._grad is None or self._grad.shape[1:] != self._W.shape or self._grad.dtype != self._W.dtype:
            self._grad = torch.empty((2, *self._W.shape), dtype=self._W.dtype, device=self._W.device)
        if self._use_peer and sh.is_sharded and self._peer_for != (tuple(self._W.shape), self._W.dtype):
            # collective (every rank gets here with the same dictionary shape): map the peers' exchange buffers once
            self._peer_for = (tuple(self._W.shape), self._W.dtype)
            self._peer = self._backend.peer_exchange(sh)

    # ---------------------------------------------------------------------------------------------
    # batch algorithm (tnmf/TransformInvariantNMF.py:282-348)
    # ---------------------------------------------------------------------------------------------
    def fit_batch(self, V, n_iterations: int = 1000, update_H: bool = True, update_W: bool = True,
                  keep_W: bool = False, sparsity_H: float = 0., inhibition_strength: float = 0.,
                  cross_atom_inhibition_strength: float = 0.,
                  progress_callback: Callable[['TransformInvariantNMF', int], bool] = None):
        assert update_H or update_W
        assert sparsity_H >= 0 and inhibition_strength >= 0 and cross_atom_inhibition_strength >= 0
        self._initialize_matrices(V, keep_W)
        self._assert_non_negative()
        step = self._batch_step(update_H, update_W, sparsity_H, inhibition_strength, cross_atom_inhibition_strength)
        for iteration in range(n_iterations):
            step()
            if progress_callback is not None:
                if not progress_callback(self, iteration):
                    break
            elif self._logger.isEnabledFor(logging.INFO):
                # the reference evaluates the energy for this line on every iteration even when the line is
                # filtered out (tnmf/TransformInvariantNMF.py:346); here it costs nothing unless it is shown
                self._logger.info(f"Iteration: {iteration}\tEnergy function: {self._energy_function()}")
        self._logger.info("TNMF finished.")

    def _batch_step(self, update_H: bool = True, update_W: bool = True, sparsity: float = 0., inhibition: float = 0.,
                    cross_inhibition: float = 0.):
        """Callable performing one batch iteration (tnmf/TransformInvariantNMF.py:334-345) on the current W/H/V:
        eagerly the first time, from CUDA graphs afterwards (see `cuda_graph`)."""
        def front(reuse_R=False):       # everything before the collective
            if update_H:
                self._update_H(sliceNone, sparsity, inhibition, cross_inhibition, reuse_R=reuse_R)
            if update_W:
                self._gradient_W(sliceNone, reduce=False)

        def take_R():           # True once after an energy evaluation left the current reconstruction behind
            have, self._R_current = self._R_current and update_H, False
            return have and self._backend.holds_R_of(self._W, self._H, **self._div_kw)

        def back():             # the W update proper (with the sum over ranks inside when the peers are mapped)
            if update_W and self._peer is not None:
                self._reduce_apply_W(self._grad)
            elif update_W:
                self._apply_W(self._grad)

        def reduce():
            if update_W and self._peer is None:
                self._sharding.sum_gradient(self._grad)

        if not (self._cuda_graph and self._fused and self._H.is_cuda and self._H.shape[0] > 0):
            def eager():
                front(take_R())
                reduce()
                back()
            return eager
        if self._step_cache is None:
            self._step_cache = {}
        key = (bool(update_H), bool(update_W), float(sparsity), float(inhibition), float(cross_inhibition),
               tuple(self._H.shape), tuple(self._H.stride()), self._divergence)
        return _GraphedStep(self._backend, front, reduce, back, self._sharding, self._step_cache, key,
                            (self._H, self._backend._device_V(self._V), self._W, self._grad), take_R)   # pylint: disable=protected-access

    # ---------------------------------------------------------------------------------------------
    # minibatch algorithms (tnmf/TransformInvariantNMF.py:350-504)
    # ---------------------------------------------------------------------------------------------
    def _blend(self, stat: Optional[torch.Tensor], grad: torch.Tensor, lam: float) -> torch.Tensor:
        """Accumulate (lam == 1) or exponentially average a W gradient (tnmf/TransformInvariantNMF.py:444-455)."""
        if stat is None:
            return grad.clone() if lam == 1 else grad * lam
        if lam == 1:
            stat += grad
        else:
            stat *= (1 - lam)
            stat += lam * grad
        return stat

    @staticmethod
    def _shuffled(batches: List[slice]) -> List[slice]:
        return [batches[i] for i in np.random.permutation(len(batches))]      # tnmf/TransformInvariantNMF.py:40-44

    def _epoch(self, algorithm: MiniBatchAlgorithm, stat, batches, kw_h, lam):
        if algorithm == MiniBatchAlgorithm.Cyclic_MU:              # :457-465
            acc = None
            for b in batches:
                self._update_H(b, **kw_h)
                acc = self._blend(acc, self._gradient_W(b, reduce=False), 1.)
            self._reduce_apply_W(acc)
        elif algorithm == MiniBatchAlgorithm.ASG_MU:               # :467-472
            for b in self._shuffled(batches):
                self._update_H(b, **kw_h)
                self._update_W(b)
        elif algorithm == MiniBatchAlgorithm.GSG_MU:               # :474-479
            b = slice(0, 0)
            for b in self._shuffled(batches):
                self._update_H(b, **kw_h)
            self._update_W(b)
        elif algorithm == MiniBatchAlgorithm.ASAG_MU:              # :481-491
            for b in self._shuffled(batches):
                self._update_H(b, **kw_h)
                stat = self._blend(stat, self._gradient_W(b), lam)
                self._apply_W(stat)
                stat[1] += self.eps      # the reference's `pos += eps` acts on the running average itself (:490)
        elif algorithm == MiniBatchAlgorithm.GSAG_MU:              # :493-504
            b = slice(0, 0)
            for b in self._shuffled(batches):
                self._update_H(b, **kw_h)
            stat = self._blend(stat, self._gradient_W(b), lam)
            self._apply_W(stat)
            stat[1] += self.eps
        return stat

    def fit_minibatches(self, V, algorithm: MiniBatchAlgorithm = MiniBatchAlgorithm.ASG_MU, batch_size: int = 3,
                        n_epochs: int = 1000, sag_lambda: float = 0.2, keep_W: bool = False, sparsity_H: float = 0.,
                        inhibition_strength: float = 0., cross_atom_inhibition_strength: float = 0.,
                        progress_callback: Callable[['TransformInvariantNMF', int], bool] = None):
        assert sparsity_H >= 0 and inhibition_strength >= 0 and cross_atom_inhibition_strength >= 0
        assert isinstance(algorithm, MiniBatchAlgorithm)
        # the reference's `algorithm in (5, 6, 7, 8)` is never true for an Enum, so the samples are never shuffled
        # (tnmf/TransformInvariantNMF.py:410-411); only the batch order is (algorithms 5-8)
        self._initialize_matrices(V, keep_W)
        self._assert_non_negative()
        batches = equal_batch_slices(self._H.shape[0], self._n_local_max, batch_size)
        kw_h = dict(sparsity=sparsity_H, inhibition=inhibition_strength, cross_inhibition=cross_atom_inhibition_strength)
        stat = None
        for epoch in range(n_epochs):
            stat = self._epoch(algorithm, stat, batches, kw_h, sag_lambda)
            if progress_callback is not None:
                if not progress_callback(self, epoch):
                    break
            elif self._logger.isEnabledFor(logging.INFO):
                self._logger.info(f"Epoch: {epoch}\tEnergy function: {self._energy_function()}")
        self._logger.info("MiniBatch TNMF finished.")

    # ---------------------------------------------------------------------------------------------
    # streams (tnmf/TransformInvariantNMF.py:506-523)
    # ---------------------------------------------------------------------------------------------
    def fit_stream(self, V: Union[Iterator, Iterable], subsample_size: int = 3, max_subsamples: int = None, **kwargs):
        """Fit subsample after subsample, keeping W and redrawing H (tnmf/TransformInvariantNMF.py:506-523).
        The next subsample is staged in pinned host memory and copied to the device on a side stream while the
        current one is being fitted."""
        feeder = _SubsampleFeeder(V, subsample_size, self._backend.device)
        sh = self._sharding
        for isub in count(0):
            subsample = feeder.next()
            if sh.is_sharded and self._input_is_local and not self._equal_shards:
                # every fit issues collectives: ranks whose streams differ in length must stop together, or the
                # longer ones would wait in the all-reduce for ever.  (`equal_shards=True` promises equal streams.)
                have = torch.tensor([0 if subsample is None else 1], dtype=torch.int32, device=self._backend.device)
                torch.distributed.all_reduce(have, op=torch.distributed.ReduceOp.MIN, group=sh.group)
                if int(have.item()) == 0:
                    if subsample is not None:
                        self._logger.warning("Another rank's sample iterator is exhausted: stopping with samples left.")
                    subsample = None
            if subsample is None:
                self._logger.info("Sample iterator exhausted. TNMF on full iterator finished.")
                return
            self._logger.info(f"Processing subsample {isub}.")
            last = max_subsamples is not None and isub == max_subsamples - 1
            if not last:
                feeder.prefetch()
            self.fit(subsample, keep_W=True, **kwargs)
            if last:
                self._logger.info(f"Processed {max_subsamples} subsamples. TNMF on iterator will stop.")
                return

    def fit(self, V, **kwargs):
        """Route on the keyword names exactly like tnmf/TransformInvariantNMF.py:525-531."""
        if 'subsample_size' in kwargs or 'max_subsamples' in kwargs:
            self.fit_stream(V, **kwargs)
        elif 'batch_size' in kwargs or 'algorithm' in kwargs:
            self.fit_minibatches(V, **kwargs)
        else:
            self.fit_batch(V, **kwargs)


class _GraphedStep:
    """One batch iteration = front (H update, local W gradient) -> all-reduce -> back (W update).  Call 1 runs eagerly
    (it sizes the workspace and the reconstruction buffer); call 2 captures the iteration into a CUDA graph - ONE graph,
    the NCCL all-reduce included, so a multi-GPU step is a single launch with no host work between the W gradient and
    the W update (with a process group that cannot be captured, gloo, the all-reduce stays an eager call between two
    graphs) - and every call from then on replays it.  Captured graphs hold raw pointers: the step keeps every buffer the
    kernels touch alive, re-captures when the backend had to replace one (`B200_Backend.buffers_epoch`), and the
    facade caches the graphs across fits for as long as all pointers repeat (`cache`)."""

    def __init__(self, backend, front, reduce, back, sharding, cache: dict, key: tuple, tensors: tuple, take_R=None):
        self._backend, self._front, self._reduce, self._back = backend, front, reduce, back
        self._take_R = take_R if take_R is not None else (lambda: False)
        self._sharded = sharding.is_sharded
        self._one_graph = not self._sharded or sharding.capturable
        self._calls = 0
        self._cache, self._key, self._tensors = cache, key, tensors
        self._entry = None          # (graphs, launches per replay, buffers epoch, tensors kept alive)
        self._entry_reuse = None    # the same iteration without its opening reconstruction (see `energy_device`)

    def _capture(self, fn):
        # capture_begin / capture_end on a side stream instead of the `torch.cuda.graph` context manager: the latter
        # runs gc.collect() and torch.cuda.empty_cache() on entry, which costs about a second with GBs of H cached
        dev = self._backend.device
        g = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        before = self._backend.launches
        with torch.cuda.stream(side):
            g.capture_begin()
            try:
                fn()
            finally:
                g.capture_end()
        torch.cuda.current_stream(dev).wait_stream(side)
        launches = self._backend.launches - before
        self._backend.launches = before
        return g, launches

    def _full_key(self):
        be = self._backend
        return self._key + tuple(t.data_ptr() for t in self._tensors) + be.buffer_pointers()

    def _eager(self, reuse_R=False):
        self._front(reuse_R)
        self._reduce()
        self._back()

    def _entry_for(self, reuse_R: bool):
        """The captured graphs of the iteration (with or without its opening reconstruction), capturing them on first use."""
        be = self._backend
        name = '_entry_reuse' if reuse_R else '_entry'
        entry = getattr(self, name)
        if entry is None:
            key = self._full_key() + (reuse_R,)
            entry = self._cache.get(key)
            if entry is None or entry[2] != be.buffers_epoch:
                torch.cuda.current_stream(be.device).synchronize()
                if self._one_graph:
                    g, n = self._capture(lambda: self._eager(reuse_R))
                    graphs = (g,)
                else:
                    (g0, n0), (g1, n1) = self._capture(lambda: self._front(reuse_R)), self._capture(self._back)
                    graphs, n = (g0, g1), n0 + n1
                while len(self._cache) >= 4:
                    self._cache.pop(next(iter(self._cache)))
                entry = (graphs, n, be.buffers_epoch, self._tensors + be.buffer_tensors(), key)
                self._cache[key] = entry
            setattr(self, name, entry)
        return entry

    def __call__(self):
        self._calls += 1
        be = self._backend
        reuse_R = self._take_R()
        if self._calls == 1 or be.kernel_events is not None:        # per-kernel timing needs eager launches
            self._eager(reuse_R)
            return
        for name in ('_entry', '_entry_reuse'):
            entry = getattr(self, name)
            if entry is not None and entry[2] != be.buffers_epoch:
                self._cache.pop(entry[4], None)                     # a buffer moved under the captured pointers
                self._entry = self._entry_reuse = None
                self._eager(reuse_R)
                return
        entry = self._entry_for(reuse_R)
        graphs = entry[0]
        graphs[0].replay()
        if len(graphs) > 1:
            self._reduce()
            graphs[1].replay()
        be.launches += entry[1]


class _SubsampleFeeder:
    """Cuts a sample source into subsamples and moves them to the device one step ahead of the fit.

    Arrays / tensors are cut into contiguous blocks (same samples, same order as iterating them one by one as
    tnmf/TransformInvariantNMF.py:514 does); any other iterable is consumed with `islice`."""

    def __init__(self, source, subsample_size: int, device):
        self._size = int(subsample_size)
        self._device = device
        self._array = source if isinstance(source, (np.ndarray, torch.Tensor)) else None
        self._iter = None if self._array is not None else iter(source)
        self._pos = 0
        self._copy_stream = torch.cuda.Stream(device=device)
        self._pinned = [None, None]
        self._pinned_busy = [None, None]    # event of the last copy out of each pinned buffer
        self._slot = 0
        self._staged = None         # (device tensor, ready event)

    def _next_host(self):
        if self._array is not None:
            if self._pos >= self._array.shape[0]:
                return None
            block = self._array[self._pos:self._pos + self._size]
            self._pos += self._size
            return block
        chunk = list(islice(self._iter, self._size))
        return np.asarray(chunk) if chunk else None

    def _stage(self):
        block = self._next_host()
        if block is None:
            return None
        if isinstance(block, torch.Tensor) and block.is_cuda:
            return block, None
        host = block if isinstance(block, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(block))
        if not host.is_pinned():
            slot = self._slot
            self._slot ^= 1
            if self._pinned_busy[slot] is not None:
                self._pinned_busy[slot].synchronize()       # the copy that last read this buffer has finished
            buf = self._pinned[slot]
            if buf is None or buf.shape != host.shape or buf.dtype != host.dtype:
                buf = torch.empty(host.shape, dtype=host.dtype, pin_memory=True)
                self._pinned[slot] = buf
            buf.copy_(host)
            host = buf
        else:
            slot = None
        with torch.cuda.stream(self._copy_stream):
            dev = host.to(self._device, non_blocking=True)
            ready = torch.cuda.Event()
            ready.record(self._copy_stream)
        if slot is not None:
            self._pinned_busy[slot] = ready
        dev.record_stream(torch.cuda.current_stream(self._device))
        return dev, ready

    def prefetch(self):
        if self._staged is None:
            self._staged = self._stage() or ()

    def next(self):
        staged = self._staged if self._staged is not None else (self._stage() or ())
        self._staged = None
        if not staged:
            return None
        dev, ready = staged
        if ready is not None:
            torch.cuda.current_stream(self._device).wait_event(ready)
        return dev
