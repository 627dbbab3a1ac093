"""
`B200_Backend`: the B200-native implementation of tnmf's backend interface.

It sits next to the reference's numpy / numpy_fft / numpy_caching_fft / pytorch backends
(tnmf/backends/*.py) behind the same abstract class (tnmf/backends/_Backend.py:13-130).  All arithmetic is done
by the hand-written sm_100a kernels of libtnmf_b200.so, reached through the C-ABI in include/tnmf_b200.h;
PyTorch only owns the device buffers and the stream.  There is no CPU fallback: without a CUDA device or
without the shared object every operation raises.

Two groups of methods:
  * the reference interface proper (`initialize`, `reconstruct`, `reconstruction_gradient_H/W`,
    `reconstruction_energy`, `normalize`, `convolve_multi_1d`, `to_ndarray`, `partial_reconstruct`), which the
    stock facade can drive unchanged, and
  * fused entry points (`update_H`, `gradient_W`, `apply_W_update`, `energy`) used by
    `tnmf_b200.TransformInvariantNMF`, which fold the facade's multiplicative-update arithmetic
    (tnmf/TransformInvariantNMF.py:217-271) into the kernels' epilogues.

Three shift axes (volumes, videos as (t, y, x)): float32 'valid' problems run the reconstruction, the H update and the W
gradient on the tcgen05 kernels over (sample, z-plane) pairs wherever they plan (DESIGN.md §3.10); float64, 'full' and
'circular' volumes, and shapes no tensor-core kernel plans for, run on the generic kernels.  'auto' picks the path.
"""
import ctypes
from contextlib import contextmanager
from typing import Optional, Sequence, Tuple, Union

import numpy as np
import torch

from . import _lib
from .interface import Backend, sliceNone

_DTYPE_CODE = {torch.float32: _lib.TNMF_F32, torch.float64: _lib.TNMF_F64}
_NP_TO_TORCH = {np.dtype('float32'): torch.float32, np.dtype('float64'): torch.float64}


def _stream_ptr(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


class B200Tensor(torch.Tensor):
    """The tensor type `B200_Backend` hands to the facade: a torch CUDA tensor that also accepts numpy operands.

    The stock facade applies a small set of duck-typed operations to what a backend returns (SURVEY 8 a9) and, in the
    lateral-inhibition branch, mixes a backend tensor with an ndarray (`inhibition_gradient - self.H[s]`,
    tnmf/TransformInvariantNMF.py:258).  The reference's own model for a backend-owned array type is
    tnmf/backends/NumPy_CachingFFT.py:52-77; here every ndarray operand of a torch operation is moved to the tensor's
    device and dtype first, and numpy defers to the reflected operators (`ndarray - tensor`)."""
    __array_priority__ = 1000
    __array_ufunc__ = None          # numpy binary operators return NotImplemented: Python then calls the reflected one here

    def _operand(self, other):
        return torch.as_tensor(other, dtype=self.dtype).to(self.device) if isinstance(other, np.ndarray) else other


def _install_operators():
    for name in ('add', 'sub', 'mul', 'truediv'):
        for fmt in ('__{}__', '__r{}__', '__i{}__'):
            dunder = fmt.format(name)
            base = getattr(torch.Tensor, dunder)

            def op(self, other, _base=base):
                return _base(self, self._operand(other))
            op.__name__ = dunder
            setattr(B200Tensor, dunder, op)


_install_operators()


def _facade_tensor(t: torch.Tensor) -> torch.Tensor:
    return t if isinstance(t, B200Tensor) else t.as_subclass(B200Tensor)


class B200_Backend(Backend):  # pylint: disable=invalid-name
    r"""
    Parameters
    ----------
    reconstruction_mode : 'valid' (default), 'full' or 'circular'
        As in the reference (tnmf/backends/_Backend.py:22-26, 60-73).  'reflect' is not pinned by the reference's
        own tests and raises NotImplementedError, the convention of tnmf/backends/NumPy.py:26-27.
    device : torch device, default: current CUDA device
    init : 'numpy' (default) draws H then W from the global legacy numpy RNG exactly like
        tnmf/backends/_Backend.py:83-98 (bit-identical seeded initialisation); 'device' draws them with the
        device RNG (for problem sizes whose float64 host draw would not fit host memory).
    kernel_path : 'auto' | 'generic' | 'tiled' | 'tma' | 'tc'   (diagnostics; see include/tnmf_b200.h)
    tensor_cores : True (default) | False | subset of ('reconstruct', 'update_h', 'gradient_w')
        which operations 'auto' may put on the tcgen05 kernels (diagnostics: pins the FP32 kernels in tests)
    rows_view : None (default: batches of >= 2^20 signal elements) | True | False
        run single-channel 1-D batches as one 2-D image of signal rows (DESIGN.md 3.7)
    tma : bool, default True; False keeps 'auto' off the TMA family
    tmem_operand : bool, default True; False keeps the tensor-core kernels on their shared-memory-operand form
    All of them travel to the library in `tnmf_problem.flags`; nothing is read from the environment.
    """

    _TC_FLAGS = {'update_h': _lib.FLAG_NO_TC_HUPD, 'reconstruct': _lib.FLAG_NO_TC_RECON, 'gradient_w': _lib.FLAG_NO_TC_GRADW}

    def __init__(self, reconstruction_mode: str = 'valid', device=None, init: str = 'numpy',
                 kernel_path: str = 'auto', tensor_cores=True, rows_view: Optional[bool] = None, tma: bool = True,
                 tmem_operand: bool = True):
        super().__init__(reconstruction_mode=reconstruction_mode)
        if reconstruction_mode in ('reflect', 'same'):
            raise NotImplementedError(f'reconstruction mode "{reconstruction_mode}" is not provided by the b200 backend')
        if reconstruction_mode not in _lib.MODES:
            raise ValueError(f'Unsupported reconstruction mode "{reconstruction_mode}". '
                             f'Please choose "valid", "full" or "circular".')
        if init not in ('numpy', 'device'):
            raise ValueError('init must be "numpy" or "device"')
        if kernel_path not in _lib.PATHS:
            raise ValueError('kernel_path must be one of ' + ', '.join(_lib.PATHS))
        if not torch.cuda.is_available():
            raise RuntimeError('the b200 backend needs a CUDA device (it has no CPU fallback)')
        self._lib = _lib.load()
        self.device = torch.device(device) if device is not None else torch.device('cuda', torch.cuda.current_device())
        self._init = init
        self._path = kernel_path
        allowed = set(self._TC_FLAGS) if tensor_cores is True else set() if not tensor_cores else set(tensor_cores)
        if not allowed <= set(self._TC_FLAGS):
            raise ValueError('tensor_cores must be a bool or a subset of ' + ', '.join(self._TC_FLAGS))
        self._flags = sum(f for op, f in self._TC_FLAGS.items() if op not in allowed)
        if rows_view is not None:
            self._flags |= _lib.FLAG_ROWS_VIEW_ALWAYS if rows_view else _lib.FLAG_NO_ROWS_VIEW
        if not tma:
            self._flags |= _lib.FLAG_NO_TMA
        if not tmem_operand:
            self._flags |= _lib.FLAG_NO_TMEM_OPERAND
        self.n_atoms = None
        self._dtype = None
        self._V_src = None      # the object the caller passes as V ...
        self._V_dev = None      # ... and its device copy
        self._R_buf = None
        self._H_store = None
        self._V_store = None
        self._W_store = None
        self._ws = None
        self.buffers_epoch = 0  # bumped whenever one of the buffers above is replaced (captured CUDA graphs watch it)
        self._energy_buf = None
        self._R_token = None    # (W pointer, H pointer, samples, divergence) whose reconstruction `energy(keep_R=True)` left
                                # in _R_buf ('kl': the quotient V / R in its place)
        self._ones = None       # V-shaped tensor of ones: the second operand of the KL correlations (`divergence='kl'`)
        self._problems = {}
        self._taps = {}
        self._last_h_problem = None
        self.launches = 0       # number of kernels of this library launched so far (bench.py reports it)
        self.kernel_events = None   # set to {} to record a (start, end) CUDA-event pair around every hot-path call

    # -----------------------------------------------------------------------------------------------
    # plumbing
    # -----------------------------------------------------------------------------------------------
    @contextmanager
    def _timed(self, name: str):
        """CUDA events on the launching stream around one C-ABI call (only while `kernel_events` is a dict)."""
        if self.kernel_events is None:
            yield
            return
        st = torch.cuda.current_stream(self.device)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(st)
        yield
        b.record(st)
        self.kernel_events.setdefault(name, []).append((a, b))

    def _to_device(self, arr, dtype=None) -> torch.Tensor:
        if isinstance(arr, torch.Tensor):
            t = arr
        else:
            t = torch.from_numpy(np.ascontiguousarray(arr))
        if dtype is not None and t.dtype != dtype:
            t = t.to(dtype)
        if t.device != self.device:
            t = t.to(self.device, non_blocking=True)
        return t.contiguous()

    def _upload_V(self, V_local) -> torch.Tensor:
        """Device copy of the samples.  Host data lands in a buffer that is reused while the shape repeats (repeated
        fits, streams): a stable address keeps captured CUDA graphs valid across fits and saves the allocation."""
        if isinstance(V_local, torch.Tensor) and V_local.device == self.device:
            return V_local.to(self._dtype).contiguous()
        host = V_local if isinstance(V_local, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(V_local))
        buf = self._V_store
        if buf is None or buf.shape != host.shape or buf.dtype != self._dtype:
            buf = self._V_store = torch.empty(host.shape, dtype=self._dtype, device=self.device)
        buf.copy_(host, non_blocking=True)
        return buf

    def _stored_W(self, w_shape) -> torch.Tensor:
        buf = self._W_store
        if buf is None or tuple(buf.shape) != tuple(w_shape) or buf.dtype != self._dtype:
            buf = self._W_store = torch.empty(w_shape, dtype=self._dtype, device=self.device)
        return buf

    def _device_V(self, V) -> torch.Tensor:
        """Device copy of V.  Like the reference's caching backends (tnmf/backends/NumPy.py:53,101,
        NumPy_CachingFFT.py:259,273) the copy made at `initialize` is reused while the same object is passed."""
        if isinstance(V, torch.Tensor) and V.device == self.device and V.is_contiguous():
            return V
        if V is self._V_src and self._V_dev is not None:
            return self._V_dev
        dev = self._to_device(V, self._dtype)
        self._V_src, self._V_dev = V, dev
        return dev

    def _problem(self, n: int, n_atoms: int, hsn: int = 0, hsm: int = 0, pitch: int = 0) -> _lib.Problem:
        key = (n, n_atoms, hsn, hsm, pitch)
        p = self._problems.get(key)
        if p is None:
            p = _lib.make_problem(n, self.n_channels, n_atoms, self._sample_shape, self.atom_shape,
                                  _DTYPE_CODE[self._dtype], self._reconstruction_mode, self._path, hsn, hsm, pitch,
                                  self._flags)
            self._problems[key] = p
        return p

    def _h_problem(self, H: torch.Tensor) -> Tuple[_lib.Problem, torch.Tensor]:
        """Problem descriptor for an activation tensor that may be a view (leading-axis slice, single atom)."""
        k = len(self.atom_shape)
        tail = H.shape[2:]
        assert len(tail) == k
        # the last axis must be dense; the second-to-last may carry a padded pitch (see `initialize`); any
        # axis before that must follow densely from the pitch
        strides = H.stride()[2:]
        pitch = int(tail[-1])
        ok = tail[-1] == 1 or strides[-1] == 1
        if k >= 2:
            if tail[-2] != 1:
                pitch = int(strides[-2])
                ok = ok and pitch >= tail[-1]
            expect = pitch * tail[-2]
            for size, stride in zip(reversed(tail[:-2]), reversed(strides[:-2])):
                if size != 1 and stride != expect:
                    ok = False
                expect *= size
        if not ok:
            H = H.contiguous()
            pitch = int(tail[-1])
        hsn, hsm = max(int(H.stride(0)), 1), max(int(H.stride(1)), 1)   # strides of size-1 axes are never used
        p = self._problem(H.shape[0], H.shape[1], hsn, hsm, 0 if pitch == tail[-1] else pitch)
        self._last_h_problem = p
        return p, H

    def _h_padding(self, shape) -> int:
        """Elements appended to every row of an activation tensor of this shape.  For float32 problems with two shift
        axes (and single-channel 1-D problems, which the library may run as one 2-D image of signal rows) the rows are
        padded to a multiple of 4 elements (16 bytes): the TMA kernels cut their boxes out of H and need that stride."""
        pad = (-shape[-1]) % 4
        rows = len(self.atom_shape) == 1 and self.n_channels == 1 and self._reconstruction_mode != 'circular'
        if self._dtype != torch.float32 or not (len(self.atom_shape) == 2 or rows) or self._path == 'generic':
            pad = 0
        return pad

    def _alloc_H(self, shape, random: bool) -> torch.Tensor:
        """Activation tensor of the reference's shape [n, M, *T]: the [..., :T_x] view of a buffer whose rows carry the
        padding of `_h_padding`."""
        pad = self._h_padding(shape)
        padded = (*shape[:-1], shape[-1] + pad)
        # the storage of the previous fit is reused when the shape repeats (fit_stream, repeated fits): a fresh
        # cudaMalloc of a multi-GB H costs tens of milliseconds
        buf = self._H_store
        if buf is None or tuple(buf.shape) != tuple(padded) or buf.dtype != self._dtype:
            self._H_store = None
            buf = self._H_store = torch.empty(padded, dtype=self._dtype, device=self.device)
            self.buffers_epoch += 1
        if random:
            buf.uniform_().neg_().add_(1)       # 1 - U[0, 1), like tnmf/backends/_Backend.py:92
        return buf[..., :shape[-1]] if pad else buf

    def _workspace(self, p: _lib.Problem, need: Optional[int] = None) -> Tuple[torch.Tensor, int]:
        if need is None:
            need = getattr(p, 'ws_need', None)
        if need is None:
            need = p.ws_need = int(self._lib.tnmf_workspace_bytes(ctypes.byref(p)))
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(max(need, 256), dtype=torch.uint8, device=self.device)
            self.buffers_epoch += 1
        return self._ws, self._ws.numel()

    def _R_for(self, n: int) -> torch.Tensor:
        shape = (n, self.n_channels, *self._sample_shape)
        numel = int(np.prod(shape))
        if self._R_buf is None or self._R_buf.numel() < numel or self._R_buf.dtype != self._dtype:
            self._R_buf = torch.empty(max(numel, 1), dtype=self._dtype, device=self.device)
            self.buffers_epoch += 1
        self._R_token = None            # whoever asks for the buffer is about to write it
        return self._R_buf[:numel].view(shape)

    def holds_R_of(self, W: torch.Tensor, H: torch.Tensor, divergence: str = 'frobenius') -> bool:
        """True while the R buffer holds the reconstruction (under 'kl': the quotient V / R) an `energy(..., keep_R=True)`
        call of this divergence computed from exactly these tensors and no other operation has written the buffer since
        (the caller vouches that W and H did not change)."""
        return self._R_token is not None and self._R_token == (W.data_ptr(), H.data_ptr(), int(H.shape[0]), divergence)

    def min_of_V(self) -> torch.Tensor:
        """Smallest element of the device copy of the samples (a device scalar; the facade's non-negativity assert)."""
        return torch.amin(self._V_dev) if self._V_dev.numel() else torch.zeros((), device=self.device)

    def buffer_tensors(self) -> tuple:
        """The scratch buffers kernels of this backend write to (kept alive by whoever captured their addresses)."""
        return tuple(t for t in (self._ws, self._R_buf, self._H_store, self._ones) if t is not None)

    def buffer_pointers(self) -> tuple:
        return tuple(t.data_ptr() for t in self.buffer_tensors())

    def _planned_problem(self, n: Optional[int]) -> _lib.Problem:
        """The last problem run (n None), or a batch of `n` samples laid out the way `initialize` would lay it out."""
        if n is None:
            return self._last_h_problem
        shape = (int(n), self.n_atoms, *self._transform_shape)
        pad = self._h_padding(shape)
        hsm = int(np.prod(shape[2:-1], dtype=np.int64)) * (shape[-1] + pad)
        return self._problem(int(n), self.n_atoms, self.n_atoms * hsm, hsm,
                             (shape[-1] + pad) if pad and len(self.atom_shape) >= 2 else 0)

    def kernel_families(self, n: Optional[int] = None) -> dict:
        """Which kernel family (generic / tiled / tma / tc) serves each hot-path operation: of the last problem run, or
        of a batch of `n` samples laid out the way `initialize` would (nothing is allocated)."""
        names = {v: k for k, v in _lib.PATHS.items()}
        p = self._planned_problem(n)
        return {op: names.get(int(self._lib.tnmf_kernel_family(ctypes.byref(p), code)), 'none')
                for op, code in (('reconstruct', _lib.OP_RECONSTRUCT), ('update_h', _lib.OP_GRADIENT_H),
                                 ('gradient_w', _lib.OP_GRADIENT_W))}

    def kernel_names(self, n: Optional[int] = None) -> dict:
        """The hot kernel (__global__ function name, as an ncu launch list shows it) behind each operation; arguments as
        for `kernel_families`."""
        p = self._planned_problem(n)
        return {op: self._lib.tnmf_kernel_name(ctypes.byref(p), code).decode()
                for op, code in (('reconstruct', _lib.OP_RECONSTRUCT), ('update_h', _lib.OP_GRADIENT_H),
                                 ('gradient_w', _lib.OP_GRADIENT_W))}

    def uses_tiled_kernels(self, n: Optional[int] = None) -> bool:
        p = self._problem(self.n_samples if n is None else n, self.n_atoms)
        return bool(self._lib.tnmf_uses_tiled_path(ctypes.byref(p)))

    # -----------------------------------------------------------------------------------------------
    # reference interface: initialisation (tnmf/backends/_Backend.py:35-98)
    # -----------------------------------------------------------------------------------------------
    def _set_dimensions(self, V, atom_shape):
        self.atom_shape = tuple(int(a) for a in atom_shape)
        self.n_samples = int(V.shape[0])
        self.n_channels = int(V.shape[1])
        self._sample_shape = tuple(int(d) for d in V.shape[2:])
        if len(self._sample_shape) != len(self.atom_shape):
            raise ValueError('atom_shape and the sample shape must have the same number of shift axes')
        p = _lib.make_problem(1, 1, 1, self._sample_shape, self.atom_shape, 0, self._reconstruction_mode)
        t = (ctypes.c_int32 * 3)()
        _lib.check(self._lib.tnmf_transform_shape(ctypes.byref(p), t), 'transform shape')
        self._transform_shape = tuple(int(t[i]) for i in range(len(self.atom_shape)))
        self._n_shift_dimensions = len(self.atom_shape)
        self._shift_dimensions = tuple(range(-1, -len(self.atom_shape) - 1, -1))
        self._problems = {}

    def initialize(self, V, atom_shape: Tuple[int, ...], n_atoms: int, W=None,
                   axes_W_normalization: Optional[Union[int, Tuple[int, ...]]] = None,
                   sample_range: Optional[Tuple[int, int]] = None):
        """Allocate H (and W unless one is handed back in, `keep_W`), upload V.

        `sample_range=(lo, hi)` keeps only that block of samples on this device (multi-GPU sample sharding);
        with init='numpy' the random draw still covers all samples so that every shard sees exactly the
        numbers a single-device run would."""
        n_total = int(V.shape[0])
        lo, hi = (0, n_total) if sample_range is None else sample_range
        if isinstance(V, torch.Tensor):
            if V.dtype not in _DTYPE_CODE:
                raise NotImplementedError(f'dtype {V.dtype} is not supported (float32 / float64)')
            self._dtype = V.dtype
        else:
            if np.dtype(V.dtype) not in _NP_TO_TORCH:
                raise NotImplementedError(f'dtype {V.dtype} is not supported (float32 / float64)')
            self._dtype = _NP_TO_TORCH[np.dtype(V.dtype)]
        V_local = V if sample_range is None else V[lo:hi]
        self._set_dimensions(V_local, atom_shape)
        self.n_atoms = int(n_atoms)
        self._V_src, self._V_dev = None, None
        self._V_src, self._V_dev = V, self._upload_V(V_local)

        h_shape = (hi - lo, self.n_atoms, *self._transform_shape)
        w_shape = (self.n_atoms, self.n_channels, *self.atom_shape)
        if self._init == 'numpy':
            # identical stream of random numbers as the reference: H first, then W, float64 draws cast to V.dtype
            np_dtype = np.float32 if self._dtype == torch.float32 else np.float64
            h_host = np.asarray(1 - np.random.rand(n_total, self.n_atoms, *self._transform_shape), dtype=np_dtype)
            H = self._alloc_H(h_shape, random=False)
            H.copy_(torch.from_numpy(h_host[lo:hi]))
            del h_host
            if W is None:
                w_host = np.asarray(1 - np.random.rand(*w_shape), dtype=np_dtype)
                W = self._stored_W(w_shape)
                W.copy_(torch.from_numpy(w_host))
                self.normalize(W, axes_W_normalization)
        else:
            H = self._alloc_H(h_shape, random=True)
            if W is None:
                W = self._stored_W(w_shape)
                W.uniform_().neg_().add_(1)
                self.normalize(W, axes_W_normalization)
        if not isinstance(W, torch.Tensor) or W.device != self.device:
            W = self._to_device(W, self._dtype)          # a W kept from a run of another backend
        if tuple(W.shape) != w_shape:
            raise ValueError(f'W has shape {tuple(W.shape)}, expected {w_shape}')
        return _facade_tensor(W), _facade_tensor(H)

    @staticmethod
    def to_ndarray(arr) -> np.ndarray:
        if isinstance(arr, torch.Tensor):
            return np.ascontiguousarray(arr.detach().cpu().numpy())
        return np.asarray(arr)

    # -----------------------------------------------------------------------------------------------
    # reference interface: small helpers
    # -----------------------------------------------------------------------------------------------
    @staticmethod
    def normalize(arr: torch.Tensor, axis: Optional[Union[int, Tuple[int, ...]]] = None):
        """In place arr /= arr.sum(axis, keepdims=True)   (tnmf/backends/_Backend.py:75-77)."""
        nd = arr.dim()
        if axis is None:
            axes = tuple(range(nd))
        elif isinstance(axis, int):
            axes = (axis % nd,)
        else:
            axes = tuple(sorted(a % nd for a in axis))
        if not arr.is_cuda or not arr.is_contiguous() or arr.dtype not in _DTYPE_CODE \
                or axes != tuple(range(axes[0], axes[-1] + 1)):
            raise NotImplementedError('normalize needs a contiguous CUDA tensor and adjacent axes')
        outer = int(np.prod(arr.shape[:axes[0]], dtype=np.int64))
        length = int(np.prod(arr.shape[axes[0]:axes[-1] + 1], dtype=np.int64))
        inner = int(np.prod(arr.shape[axes[-1] + 1:], dtype=np.int64))
        lib = _lib.load()
        _lib.check(lib.tnmf_normalize(_DTYPE_CODE[arr.dtype], arr.data_ptr(), outer, length, inner,
                                      _stream_ptr(arr.device)), 'normalize')

    @staticmethod
    def convolve_multi_1d(arr: torch.Tensor, kernels: Sequence[np.ndarray], axes: Sequence[int]) -> torch.Tensor:
        """Separable zero-boundary convolution (tnmf/backends/_NumPyBackend.py:56-64)."""
        assert len(kernels) == len(axes)
        lib = _lib.load()
        src = arr if arr.is_contiguous() else arr.contiguous()
        code = _DTYPE_CODE[src.dtype]
        out = src
        for a, kern in zip(axes, kernels):
            a = a % src.dim()
            taps = torch.as_tensor(np.ascontiguousarray(kern, dtype=np.float64)).to(src.device)
            dst = torch.empty_like(src)
            outer = int(np.prod(src.shape[:a], dtype=np.int64))
            inner = int(np.prod(src.shape[a + 1:], dtype=np.int64))
            _lib.check(lib.tnmf_convolve_1d(code, out.data_ptr(), dst.data_ptr(), outer, int(src.shape[a]), inner,
                                            taps.data_ptr(), int(taps.numel()), _stream_ptr(src.device)),
                       'convolve_multi_1d')
            out = dst
        if out is arr:
            out = arr.clone()
        return _facade_tensor(out)

    # -----------------------------------------------------------------------------------------------
    # reference interface: the four hot-path operations
    # -----------------------------------------------------------------------------------------------
    def reconstruct(self, W: torch.Tensor, H: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """R = sum_m W[m] * H[:, m]   (tnmf/backends/_Backend.py:120-122).  Accepts H views (partial_reconstruct)."""
        p, H = self._h_problem(H)
        if W.shape[0] != H.shape[1]:
            raise ValueError('W and H disagree on the number of atoms')
        W = W if W.is_contiguous() else W.contiguous()
        R = out if out is not None else torch.empty((H.shape[0], self.n_channels, *self._sample_shape),
                                                    dtype=self._dtype, device=self.device)
        ws, ws_bytes = self._workspace(p)
        with self._timed('reconstruct'):
            _lib.check(self._lib.tnmf_reconstruct(ctypes.byref(p), W.data_ptr(), H.data_ptr(), R.data_ptr(),
                                                  ws.data_ptr(), ws_bytes, _stream_ptr(self.device)), 'reconstruct')
        self.launches += self._n_launches(p, _lib.OP_RECONSTRUCT)
        return _facade_tensor(R)

    def _n_launches(self, p: _lib.Problem, op: int) -> int:
        """Kernels one call of operation `op` launches (the TMA family pre-arranges the atoms in a tiny extra kernel, the
        tensor-core kernels take 16 atoms per launch, the W gradient always has its finishing reduction)."""
        return max(int(self._lib.tnmf_launch_count(ctypes.byref(p), op)), 0)

    def reconstruction_gradient_H(self, V, W, H, s: slice = sliceNone):
        """(neg, pos) with the shape of H[s]   (tnmf/backends/_Backend.py:110-118)."""
        Hs = H[s]
        Vs = self._device_V(V)[s]
        R = self.reconstruct(W, Hs, out=self._R_for(Hs.shape[0]))
        p = self._problem(Hs.shape[0], self.n_atoms)
        neg = torch.empty(Hs.shape, dtype=self._dtype, device=self.device)
        pos = torch.empty_like(neg)
        ws, ws_bytes = self._workspace(p)
        _lib.check(self._lib.tnmf_gradient_h(ctypes.byref(p), Vs.data_ptr(), R.data_ptr(), W.data_ptr(),
                                             neg.data_ptr(), pos.data_ptr(), ws.data_ptr(), ws_bytes,
                                             _stream_ptr(self.device)), 'gradient_h')
        self.launches += self._n_launches(p, _lib.OP_GRADIENT_H)
        return _facade_tensor(neg), _facade_tensor(pos)

    def reconstruction_gradient_W(self, V, W, H, s: slice = sliceNone):
        """(neg, pos) with the shape of W   (tnmf/backends/_Backend.py:100-108)."""
        out = torch.empty((2, *W.shape), dtype=self._dtype, device=self.device)
        self.gradient_W(V, W, H, s, out)
        return _facade_tensor(out[0]), _facade_tensor(out[1])

    def reconstruction_energy(self, V, W, H) -> float:
        """0.5 * ||V - R||^2 as a Python float   (tnmf/backends/_Backend.py:127-130)."""
        return float(self.energy(V, W, H).item())

    # -----------------------------------------------------------------------------------------------
    # fused entry points used by tnmf_b200.TransformInvariantNMF
    #
    # `divergence='kl'` (DESIGN.md §3.11): the generalised Kullback-Leibler divergence D(V||R) instead of 0.5*||V - R||^2.
    # Its gradients are the Frobenius ones with (Q, ones) in place of (V, R), Q = V / R: so the same fused kernels run,
    # after one elementwise pass (tnmf_kl_quotient) turns the reconstruction in the R buffer into Q.
    # -----------------------------------------------------------------------------------------------
    @staticmethod
    def _is_kl(divergence: str) -> bool:
        if divergence not in ('frobenius', 'kl'):
            raise ValueError(f'divergence must be "frobenius" or "kl" (got {divergence!r})')
        return divergence == 'kl'

    def _ones_for(self, V_full: torch.Tensor) -> torch.Tensor:
        """Ones shaped like the device copy of the samples; minibatches slice it like V."""
        if self._ones is None or self._ones.shape != V_full.shape or self._ones.dtype != self._dtype:
            self._ones = None
            self._ones = torch.ones(V_full.shape, dtype=self._dtype, device=self.device)
            self.buffers_epoch += 1
        return self._ones

    def _kl_quotient(self, Vs: torch.Tensor, R: torch.Tensor, divergence: Optional[torch.Tensor] = None) -> None:
        """R <- V / max(R, tau) in place (0 where V == 0); the divergence of the R passed in goes to `divergence`."""
        p = self._problem(int(R.shape[0]), self.n_atoms)
        need = getattr(p, 'kl_ws_need', None)
        if need is None:
            need = p.kl_ws_need = int(self._lib.tnmf_kl_workspace_bytes(ctypes.byref(p)))
        ws, ws_bytes = self._workspace(p, need)
        with self._timed('kl_quotient'):
            _lib.check(self._lib.tnmf_kl_quotient(ctypes.byref(p), Vs.data_ptr(), R.data_ptr(),
                                                  None if divergence is None else divergence.data_ptr(), ws.data_ptr(),
                                                  ws_bytes, _stream_ptr(self.device)), 'kl_quotient')
        self.launches += 1 if divergence is None else 2

    def energy(self, V, W, H, s: slice = sliceNone, keep_R: bool = False, divergence: str = 'frobenius') -> torch.Tensor:
        """Device-resident double scalar 0.5*||V[s] - reconstruct(W, H[s])||^2 (no host synchronisation).  With `keep_R`
        the reconstruction is also written to the R buffer, where `update_H(..., reuse_R=True)` picks it up.
        `divergence='kl'`: D(V[s] || reconstruct(W, H[s])); the R buffer then holds the quotient V / R."""
        Hs = H[s]
        Vs = self._device_V(V)[s]
        keep_R = keep_R and Hs.shape[0] > 0 and Hs.data_ptr() == H.data_ptr() and Hs.shape[0] == H.shape[0]
        if self._is_kl(divergence):
            e = torch.empty((), dtype=torch.float64, device=self.device)
            R = self.reconstruct(W, Hs, out=self._R_for(Hs.shape[0]))
            self._kl_quotient(Vs, R, e)
            if keep_R:
                self._R_token = (W.data_ptr(), Hs.data_ptr(), int(Hs.shape[0]), divergence)
            return e
        R = self._R_for(Hs.shape[0]) if keep_R else None
        p, Hs = self._h_problem(Hs)
        ws, ws_bytes = self._workspace(p)
        e = torch.empty((), dtype=torch.float64, device=self.device)
        _lib.check(self._lib.tnmf_reconstruct_energy(ctypes.byref(p), Vs.data_ptr(), W.data_ptr(), Hs.data_ptr(),
                                                     R.data_ptr() if keep_R else None, e.data_ptr(), ws.data_ptr(),
                                                     ws_bytes, _stream_ptr(self.device)), 'reconstruct_energy')
        self.launches += 1 + self._n_launches(p, _lib.OP_RECONSTRUCT)
        if keep_R:
            self._R_token = (W.data_ptr(), Hs.data_ptr(), int(Hs.shape[0]), divergence)
        return e

    def _inhibition_taps(self, kernels: Sequence[np.ndarray]):
        key = tuple(k.tobytes() for k in kernels)
        taps = self._taps.get(key)
        if taps is None:
            taps = [torch.as_tensor(np.ascontiguousarray(k, dtype=np.float64)).to(self.device) for k in kernels]
            self._taps = {key: taps}
        return taps

    def update_H(self, V, W, H, s: slice = sliceNone, sparsity: float = 0., inhibition: float = 0.,
                 cross_inhibition: float = 0., inhibition_kernels: Optional[Sequence[np.ndarray]] = None,
                 eps: float = 1.e-9, reuse_R: bool = False, planes: Optional[Tuple[int, int]] = None,
                 divergence: str = 'frobenius') -> None:
        """One in-place multiplicative update of H[s]: reconstruct, both correlations, sparsity / inhibition terms and
        H <- (H*neg)/pos in one fused kernel   (tnmf/TransformInvariantNMF.py:246-271 + :217-235).
        `planes=(t_lo, t_hi)` updates only those activation indices along the first shift axis (tnmf_update_h_planes:
        three shift axes, or any problem on the generic kernels); the reconstruction and the inhibition terms still see
        all of H.  `divergence='kl'`: the KL update, the same kernel on (V / R, ones) instead of (V, R)."""
        kl = self._is_kl(divergence)
        Hs = H[s]
        if Hs.shape[0] == 0:
            return
        V_full = self._device_V(V)
        Vs = V_full[s]
        n = Hs.shape[0]
        have_R = reuse_R and self.holds_R_of(W, Hs, divergence)    # left by `energy(keep_R=True)` for these very W, H
        R = self._R_for(n)                              # (clears the token: H changes below)
        if not have_R:
            R = self.reconstruct(W, Hs, out=R)
            if kl:
                self._kl_quotient(Vs, R)
        if kl:
            Vs, R = R, self._ones_for(V_full)[s]
        p, Hs = self._h_problem(Hs)
        G_ptr, Gsum_ptr = None, None
        lam, lam_cross = 0.0, 0.0
        st = _stream_ptr(self.device)
        if inhibition > 0 or cross_inhibition > 0:
            taps = self._inhibition_taps(inhibition_kernels)
            code = _DTYPE_CODE[self._dtype]
            G = Hs.contiguous()      # the separable convolution reads dense [outer, len, inner] views
            k = len(self.atom_shape)
            for i, tp in enumerate(taps):
                axis = Hs.dim() - k + i
                dst = torch.empty_like(Hs)
                outer = int(np.prod(Hs.shape[:axis], dtype=np.int64))
                inner = int(np.prod(Hs.shape[axis + 1:], dtype=np.int64))
                _lib.check(self._lib.tnmf_convolve_1d(code, G.data_ptr(), dst.data_ptr(), outer, int(Hs.shape[axis]),
                                                      inner, tp.data_ptr(), int(tp.numel()), st), 'convolve_1d')
                self.launches += 1
                G = dst
            G_ptr = G.data_ptr()
            lam = float(inhibition) if inhibition > 0 else 0.0
            if cross_inhibition > 0:
                inner = int(np.prod(Hs.shape[2:], dtype=np.int64))
                Gsum = torch.empty((n, 1, *Hs.shape[2:]), dtype=self._dtype, device=self.device)
                _lib.check(self._lib.tnmf_sum_atoms(code, G.data_ptr(), Gsum.data_ptr(), n, self.n_atoms, inner, st),
                           'sum_atoms')
                self.launches += 1
                Gsum_ptr = Gsum.data_ptr()
                lam_cross = float(cross_inhibition) / (self.n_atoms - 1)
        reg = eps + sparsity if sparsity > 0 else eps
        ws, ws_bytes = self._workspace(p)
        with self._timed('update_h'):
            if planes is None:
                _lib.check(self._lib.tnmf_update_h(ctypes.byref(p), Vs.data_ptr(), R.data_ptr(), W.data_ptr(),
                                                   Hs.data_ptr(), float(reg), G_ptr, lam, Gsum_ptr, lam_cross,
                                                   ws.data_ptr(), ws_bytes, st), 'update_h')
            else:
                _lib.check(self._lib.tnmf_update_h_planes(ctypes.byref(p), Vs.data_ptr(), R.data_ptr(), W.data_ptr(),
                                                          Hs.data_ptr(), float(reg), G_ptr, lam, Gsum_ptr, lam_cross,
                                                          int(planes[0]), int(planes[1]), ws.data_ptr(), ws_bytes, st),
                           'update_h_planes')
        self.launches += self._n_launches(p, _lib.OP_GRADIENT_H)

    def gradient_W(self, V, W, H, s: slice, out: torch.Tensor, H_for_R: Optional[torch.Tensor] = None,
                   planes: Optional[Tuple[int, int]] = None, divergence: str = 'frobenius') -> torch.Tensor:
        """out[0] = neg, out[1] = pos of the W gradient on samples s (split-K + deterministic final reduction).
        `H_for_R`: reconstruct from these activations instead of H (halo sharding correlates with a band of H - the other
        rows zeroed - against the reconstruction of all of it; tnmf_b200/halo.py).
        `planes=(t_lo, t_hi)`: correlate with those activation indices along the first shift axis only, as if H were zero
        elsewhere, against the reconstruction of all of H (tnmf_gradient_w_planes; the same kernels as `update_H`'s).
        `divergence='kl'`: the KL gradient, the same kernel on (V / R, ones) instead of (V, R)."""
        kl = self._is_kl(divergence)
        Hs = H[s]
        V_full = self._device_V(V)
        Vs = V_full[s]
        n = Hs.shape[0]
        p, Hs = self._h_problem(Hs)
        if n == 0:
            out.zero_()
            return out
        R = self.reconstruct(W, Hs if H_for_R is None else H_for_R[s], out=self._R_for(n))
        if kl:
            self._kl_quotient(Vs, R)
            Vs, R = R, self._ones_for(V_full)[s]
        if H_for_R is not None:
            p, Hs = self._h_problem(Hs)         # (reconstruct recorded the other tensor's problem)
        ws, ws_bytes = self._workspace(p)
        with self._timed('gradient_w'):
            if planes is None:
                _lib.check(self._lib.tnmf_gradient_w(ctypes.byref(p), Vs.data_ptr(), R.data_ptr(), Hs.data_ptr(),
                                                     out[0].data_ptr(), out[1].data_ptr(), ws.data_ptr(), ws_bytes,
                                                     _stream_ptr(self.device)), 'gradient_w')
            else:
                _lib.check(self._lib.tnmf_gradient_w_planes(ctypes.byref(p), Vs.data_ptr(), R.data_ptr(), Hs.data_ptr(),
                                                            out[0].data_ptr(), out[1].data_ptr(), int(planes[0]),
                                                            int(planes[1]), ws.data_ptr(), ws_bytes,
                                                            _stream_ptr(self.device)), 'gradient_w_planes')
        self.launches += self._n_launches(p, _lib.OP_GRADIENT_W)
        return out

    def peer_exchange(self, sharding):
        """Map the ranks' NVLink exchange buffers for `allreduce_update_W` (collective; None where unavailable)."""
        from .distributed import PeerExchange
        return PeerExchange.create(self._lib, self._problem(0, self.n_atoms), sharding, self.device)

    def allreduce_update_W(self, W: torch.Tensor, grad: torch.Tensor, px, eps: float = 1.e-9) -> None:
        """`apply_W_update` on the sum of `grad` over all ranks, in one kernel over NVLink peer memory (collective)."""
        assert grad.is_contiguous() and W.is_contiguous()
        p = self._problem(0, self.n_atoms)
        with self._timed('update_w'):
            _lib.check(self._lib.tnmf_allreduce_update_w(ctypes.byref(p), W.data_ptr(), grad.data_ptr(),
                                                         ctypes.byref(px.world), px.state.data_ptr(), float(eps),
                                                         _stream_ptr(self.device)), 'allreduce_update_w')
        px.calls += 1
        self.launches += 1

    def apply_W_update(self, W: torch.Tensor, grad: torch.Tensor, eps: float = 1.e-9) -> None:
        """W <- (W*neg)/(pos+eps), then per-(atom, channel) normalisation, in place
        (tnmf/TransformInvariantNMF.py:217-244, tnmf/backends/_Backend.py:75-77).  grad = stacked (neg, pos)."""
        p = self._problem(0, self.n_atoms)
        with self._timed('update_w'):
            _lib.check(self._lib.tnmf_update_w(ctypes.byref(p), W.data_ptr(), grad[0].data_ptr(), grad[1].data_ptr(),
                                               float(eps), _stream_ptr(self.device)), 'update_w')
        self.launches += 1
