"""
ctypes binding of libtnmf_b200.so (the C-ABI declared in include/tnmf_b200.h) and its in-tree build recipe.

The library is the only arithmetic provider of this package: there is no CPU fallback and no alternative
code path.  If the shared object is missing or does not export the declared symbols, importing the binding
fails loudly.
"""
import ctypes
import os
import shutil
import subprocess
from typing import Optional, Sequence

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
LIB_PATH = os.environ.get('TNMF_LIB_PATH') or os.path.join(HERE, 'libtnmf_b200.so')      # override: experiments only
SOURCES = ('capi.cu', 'generic_kernels.cu', 'elementwise.cu', 'tiled_kernels.cu', 'tma_kernels.cu', 'tc_hupd.cu', 'tc_gradw.cu', 'tc_recon.cu',
           'tc_gradw_ts.cu', 'tc_recon_ts.cu', 'tc_hupd_ts.cu', 'tc_recon_os.cu', 'tc_gradw_ns.cu', 'peer_update_w.cu')
# compiled once per atom-width chunk (-DTNMF_AXC=...): the register-tiled kernels
CHUNKED_SOURCES = ('tiled_recon.cu', 'tiled_hupd.cu', 'tiled_gradw.cu', 'tma_recon.cu', 'tma_hupd.cu', 'tma_gradw.cu')
CHUNKS = (4, 8, 12, 16)
HEADERS = ('common.cuh', 'tiled_common.cuh', 'tma_common.cuh', 'tc_common.cuh', os.path.join('..', '..', 'include', 'tnmf_b200.h'))

# NB: no --use_fast_math: divisions must round like the reference's IEEE arithmetic.
NVCC_FLAGS = ('-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo', '-O3', '-std=c++17',
              '-Xcompiler', '-fPIC')

TNMF_F32, TNMF_F64 = 0, 1
MODES = {'valid': 0, 'full': 1, 'circular': 2}
PATHS = {'auto': 0, 'generic': 1, 'tiled': 2, 'tma': 3, 'tc': 4}
OP_RECONSTRUCT, OP_GRADIENT_H, OP_GRADIENT_W = 0, 1, 2
TNMF_OK, TNMF_EINVAL, TNMF_EUNSUPPORTED, TNMF_EWORKSPACE, TNMF_ECUDA = 0, 1, 2, 3, 1000
ABI_VERSION = 6
# tnmf_problem.flags (include/tnmf_b200.h)
FLAG_NO_ROWS_VIEW, FLAG_ROWS_VIEW_ALWAYS = 1, 2
FLAG_NO_TC_HUPD, FLAG_NO_TC_RECON, FLAG_NO_TC_GRADW, FLAG_NO_TC, FLAG_NO_TMA, FLAG_NO_TMEM_OPERAND = 4, 8, 16, 28, 32, 64


class Problem(ctypes.Structure):
    """Mirror of `struct tnmf_problem` (include/tnmf_b200.h)."""
    _fields_ = [
        ('ndim', ctypes.c_int32), ('dtype', ctypes.c_int32), ('mode', ctypes.c_int32), ('path', ctypes.c_int32),
        ('n_samples', ctypes.c_int32), ('n_channels', ctypes.c_int32), ('n_atoms', ctypes.c_int32),
        ('h_pitch', ctypes.c_int32),
        ('sample_shape', ctypes.c_int32 * 3), ('atom_shape', ctypes.c_int32 * 3),
        ('h_stride_n', ctypes.c_int64), ('h_stride_m', ctypes.c_int64),
        ('flags', ctypes.c_int32), ('reserved', ctypes.c_int32),
    ]


MAX_PEERS = 16


class PeerWorld(ctypes.Structure):
    """Mirror of `struct tnmf_peer_world` (include/tnmf_b200.h)."""
    _fields_ = [('world', ctypes.c_int32), ('rank', ctypes.c_int32), ('buffers', ctypes.c_void_p * MAX_PEERS)]


_P = ctypes.POINTER(Problem)
_vp, _i32, _i64, _dbl, _sz = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_double, ctypes.c_size_t

# name -> (restype, argtypes); every symbol include/tnmf_b200.h declares
SIGNATURES = {
    'tnmf_abi_version': (ctypes.c_int, []),
    'tnmf_status_string': (ctypes.c_char_p, [ctypes.c_int]),
    'tnmf_transform_shape': (ctypes.c_int, [_P, ctypes.POINTER(ctypes.c_int32)]),
    'tnmf_workspace_bytes': (_sz, [_P]),
    'tnmf_uses_tiled_path': (ctypes.c_int, [_P]),
    'tnmf_kernel_family': (ctypes.c_int, [_P, ctypes.c_int]),
    'tnmf_kernel_name': (ctypes.c_char_p, [_P, ctypes.c_int]),
    'tnmf_launch_count': (ctypes.c_int, [_P, ctypes.c_int]),
    'tnmf_reconstruct': (ctypes.c_int, [_P, _vp, _vp, _vp, _vp, _sz, _vp]),
    'tnmf_reconstruct_energy': (ctypes.c_int, [_P, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    'tnmf_gradient_h': (ctypes.c_int, [_P, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    'tnmf_update_h': (ctypes.c_int, [_P, _vp, _vp, _vp, _vp, _dbl, _vp, _dbl, _vp, _dbl, _vp, _sz, _vp]),
    'tnmf_gradient_w': (ctypes.c_int, [_P, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    'tnmf_update_h_planes': (ctypes.c_int, [_P, _vp, _vp, _vp, _vp, _dbl, _vp, _dbl, _vp, _dbl, _i32, _i32, _vp, _sz, _vp]),
    'tnmf_gradient_w_planes': (ctypes.c_int, [_P, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _vp, _sz, _vp]),
    'tnmf_update_w': (ctypes.c_int, [_P, _vp, _vp, _vp, _dbl, _vp]),
    'tnmf_peer_buffer_bytes': (_sz, [_P, _i32]),
    'tnmf_allreduce_update_w': (ctypes.c_int, [_P, _vp, _vp, ctypes.POINTER(PeerWorld), _vp, _dbl, _vp]),
    'tnmf_normalize': (ctypes.c_int, [_i32, _vp, _i64, _i64, _i64, _vp]),
    'tnmf_convolve_1d': (ctypes.c_int, [_i32, _vp, _vp, _i64, _i64, _i64, _vp, _i32, _vp]),
    'tnmf_sum_atoms': (ctypes.c_int, [_i32, _vp, _vp, _i64, _i64, _i64, _vp]),
    'tnmf_fp32_peak_probe': (ctypes.c_int, [_vp, _i32, ctypes.POINTER(ctypes.c_double), _vp]),
}


def needs_build() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, s) for s in SOURCES + CHUNKED_SOURCES]
    deps += [os.path.normpath(os.path.join(CSRC, h)) for h in HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False, jobs: Optional[int] = None) -> str:
    """Compile the CUDA sources for sm_100a into tnmf_b200/libtnmf_b200.so (in-tree, travels with the repo)."""
    if not force and not needs_build():
        return LIB_PATH
    nvcc = shutil.which('nvcc') or '/usr/local/cuda/bin/nvcc'
    if not os.path.exists(nvcc):
        raise RuntimeError('nvcc not found: cannot build libtnmf_b200.so')
    objdir = os.path.join(HERE, '_obj')
    os.makedirs(objdir, exist_ok=True)
    units = [(s, s.replace('.cu', '.o'), []) for s in SOURCES]
    units += [(s, s.replace('.cu', f'_axc{c}.o'), [f'-DTNMF_AXC={c}']) for s in CHUNKED_SOURCES for c in CHUNKS]
    jobs = jobs or max(1, min(len(units), os.cpu_count() or 1))
    # incremental: a unit is recompiled when its object is older than its source, any header or this recipe
    common = [os.path.normpath(os.path.join(CSRC, h)) for h in HEADERS] + [os.path.abspath(__file__)]
    newest_common = max(os.path.getmtime(d) for d in common)
    extra = os.environ.get('TNMF_NVCC_EXTRA', '')
    stamp = os.path.join(objdir, 'flags.txt')
    if force or not os.path.exists(stamp) or open(stamp).read() != extra:
        newest_common = float('inf')
    objs = [os.path.join(objdir, obj) for _, obj, _ in units]
    pending = [u for u in units
               if not os.path.exists(os.path.join(objdir, u[1]))
               or os.path.getmtime(os.path.join(objdir, u[1])) < max(newest_common, os.path.getmtime(os.path.join(CSRC, u[0])))]
    running, log = [], []
    while pending or running:
        while pending and len(running) < jobs:
            src, obj, defs = pending.pop(0)
            obj = os.path.join(objdir, obj)
            cmd = [nvcc, *NVCC_FLAGS, *os.environ.get('TNMF_NVCC_EXTRA', '').split(), *defs, '-Xptxas', '-v', '-c', os.path.join(CSRC, src), '-o', obj]
            running.append((f'{src} {" ".join(defs)}',
                            subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        name, pr = running.pop(0)
        out, _ = pr.communicate()
        log.append(f'== {name}\n{out}')
        if pr.returncode != 0:
            for _, other in running:
                other.kill()
            raise RuntimeError(f'nvcc failed on {name}:\n{out}')
    with open(stamp, 'w') as f:
        f.write(extra)
    with open(os.path.join(objdir, 'ptxas.log'), 'a' if not force else 'w') as f:
        f.write('\n'.join(log))
    if verbose:
        print('\n'.join(log))
    tmp = LIB_PATH + '.tmp'
    subprocess.run([nvcc, '-shared', '-o', tmp, *objs, '-lcudart'], check=True)
    os.replace(tmp, LIB_PATH)
    return LIB_PATH


_lib: Optional[ctypes.CDLL] = None


def load() -> ctypes.CDLL:
    """Load the shared object and bind every declared symbol.  Raises if anything is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f'{LIB_PATH} is missing: run `python -c "import __graft_entry__ as g; g.build()"` '
                          f'(tnmf_b200 has no CPU fallback)')
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if lib.tnmf_abi_version() != ABI_VERSION:
        raise ImportError(f'libtnmf_b200.so has ABI {lib.tnmf_abi_version()}, binding expects {ABI_VERSION}')
    _lib = lib
    return lib


def check(status: int, what: str = '') -> None:
    """Translate a status code into the reference's error conventions (SURVEY 8b)."""
    if status == TNMF_OK:
        return
    msg = load().tnmf_status_string(status).decode()
    if what:
        msg = f'{what}: {msg}'
    if status == TNMF_EUNSUPPORTED:
        raise NotImplementedError(msg)
    if status == TNMF_EINVAL:
        raise ValueError(msg)
    raise RuntimeError(msg)


def make_problem(n_samples: int, n_channels: int, n_atoms: int, sample_shape: Sequence[int],
                 atom_shape: Sequence[int], dtype_code: int, mode: str = 'valid', path: str = 'auto',
                 h_stride_n: int = 0, h_stride_m: int = 0, h_pitch: int = 0, flags: int = 0) -> Problem:
    if mode not in MODES:
        raise ValueError(f'Unsupported reconstruction mode "{mode}". Please choose "valid", "full" or "circular".')
    if len(sample_shape) != len(atom_shape):
        raise ValueError('sample and atom rank differ')
    if not 1 <= len(sample_shape) <= 3:
        raise NotImplementedError('tnmf_b200 supports 1 to 3 shift axes')
    p = Problem()
    p.ndim, p.dtype, p.mode, p.path = len(sample_shape), dtype_code, MODES[mode], PATHS[path]
    p.n_samples, p.n_channels, p.n_atoms = int(n_samples), int(n_channels), int(n_atoms)
    for i, (d, a) in enumerate(zip(sample_shape, atom_shape)):
        p.sample_shape[i] = int(d)
        p.atom_shape[i] = int(a)
    p.h_stride_n, p.h_stride_m, p.h_pitch = int(h_stride_n), int(h_stride_m), int(h_pitch)
    p.flags, p.reserved = int(flags), 0
    return p
