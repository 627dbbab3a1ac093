"""
The iteration code of the reference facade (emdgroup/tnmf, tnmf/TransformInvariantNMF.py) as it reaches a backend,
restated for tests/test_gpu_stock_facade.py.  It touches the backend through the abstract interface of
tnmf/backends/_Backend.py only, and it applies to what the backend returns exactly the duck-typed operations the
reference applies (SURVEY 8 a9): in-place arithmetic on `H[s]` views, `pos += float`, `pos += tensor`, a backend tensor
minus the ndarray `self.H[s]` (:258), unary minus and `.sum(axis=1, keepdims=True)` (:263), and `0 + tensor` in the
Cyclic_MU accumulation (:457-465).  It holds no arithmetic of its own besides those operations.
"""
from oracle.tnmf_oracle import inhibition_kernels, minibatch_slices


class StockFacade:
    eps = 1.e-9

    def __init__(self, backend, n_atoms, atom_shape, inhibition_range=None):
        self._backend = backend
        self.n_atoms = n_atoms
        self.atom_shape = tuple(atom_shape)
        if inhibition_range is None:                        # :154-163
            inhibition_range = tuple(a - 1 for a in self.atom_shape)
        self._inhibition_kernels_1D = inhibition_kernels(inhibition_range)
        self._axes_W_normalization = tuple(range(-len(self.atom_shape), 0))
        self._V = self._W = self._H = None

    # results, as ndarrays (:188-209)
    @property
    def W(self):
        return self._backend.to_ndarray(self._W)

    @property
    def H(self):
        return self._backend.to_ndarray(self._H)

    @property
    def R(self):
        return self._backend.to_ndarray(self._backend.reconstruct(self._W, self._H))

    def R_partial(self, i_atom):
        return self._backend.to_ndarray(self._backend.partial_reconstruct(self._W, self._H, i_atom))

    def _energy_function(self):
        return self._backend.reconstruction_energy(self._V, self._W, self._H)

    # updates (:217-271)
    def _multiplicative_update(self, arr, neg, pos, sparsity=0., normalization_axes=None):
        regularization = self.eps
        if sparsity > 0:
            regularization += sparsity
        pos += regularization
        arr *= neg
        arr /= pos
        if normalization_axes is not None:
            self._backend.normalize(arr, axis=normalization_axes)

    def _update_H(self, s=slice(None), sparsity=0., inhibition=0., cross_inhibition=0.):
        neg, pos = self._backend.reconstruction_gradient_H(self._V, self._W, self._H, s)
        if inhibition > 0 or cross_inhibition > 0:
            axes = range(-len(self.atom_shape), 0)
            inhibition_gradient = self._backend.convolve_multi_1d(self._H[s], self._inhibition_kernels_1D, axes)
            if inhibition > 0:
                tmp = inhibition_gradient - self.H[s]       # backend tensor minus ndarray
                tmp *= inhibition
                pos += tmp
            if cross_inhibition > 0:
                tmp = inhibition_gradient.sum(axis=1, keepdims=True)
                tmp = -inhibition_gradient + tmp
                tmp *= cross_inhibition / (self.n_atoms - 1)
                pos += tmp
        self._multiplicative_update(self._H[s], neg, pos, sparsity=sparsity)

    def _update_W(self, s=slice(None)):
        neg, pos = self._backend.reconstruction_gradient_W(self._V, self._W, self._H, s)
        self._multiplicative_update(self._W, neg, pos, normalization_axes=self._axes_W_normalization)

    def _initialize_matrices(self, V):                      # :273-280
        self._V = V
        self._W, self._H = self._backend.initialize(V, self.atom_shape, self.n_atoms, None, self._axes_W_normalization)

    # algorithms
    def fit_batch(self, V, n_iterations=1000, sparsity_H=0., inhibition_strength=0., cross_atom_inhibition_strength=0.,
                  progress_callback=None):                  # :282-348
        self._initialize_matrices(V)
        for iteration in range(n_iterations):
            self._update_H(slice(None), sparsity_H, inhibition_strength, cross_atom_inhibition_strength)
            self._update_W()
            if progress_callback is not None and not progress_callback(self, iteration):
                break

    def fit_cyclic_minibatches(self, V, batch_size=3, n_epochs=1000, sparsity_H=0.):   # :350-465, Cyclic_MU
        self._initialize_matrices(V)
        batches = minibatch_slices(len(V), batch_size)
        for _ in range(n_epochs):
            neg, pos = 0, 0
            for s in batches:
                self._update_H(s, sparsity_H)
                neg_s, pos_s = self._backend.reconstruction_gradient_W(self._V, self._W, self._H, s)
                neg = neg + neg_s
                pos = pos + pos_s
            self._multiplicative_update(self._W, neg, pos, normalization_axes=self._axes_W_normalization)
