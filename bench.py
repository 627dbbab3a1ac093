#!/usr/bin/env python
"""
bench.py - throughput of the shift-invariant NMF multiplicative-update (MU) iteration.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload cfg2|cfg3|...]
                    [--dump-outputs DIR]

A "step" is one batch MU iteration (H update, W update; tnmf/TransformInvariantNMF.py:334-346 of the
reference) over a synthetic batch.  The metric is BASELINE.json's: sample-iterations per second.

`--dump-outputs DIR` (own arm) writes W and H as they stand after the last timed step to DIR/W.npy and DIR/H.npy
(rank 0's samples), H as a fixed sample DIR/H_sample.npy where all of it would exceed 64 MB (see `dump_outputs`).  The
batch and the start values of W and H come from seeded generators of this script, so with the same arguments two
builds of the library start from the same numbers and can be compared output for output.

  * own arm (`--impl b200`): the hand-written sm_100a kernels of libtnmf_b200.so driven through
    `tnmf_b200.TransformInvariantNMF`.  `value` is measured with the batch resident in HBM (CUDA events, max over
    ranks); `e2e` is the same metric through the public `fit()` call with a pinned HOST batch: upload of V, device
    initialisation, K iterations, download of W and of the energy, all inside the timed region.
    N > 1 (torchrun, one rank per GPU): weak scaling - every rank owns a batch of the workload's size, the only
    collective is the all-reduce of the stacked W-gradient numerator/denominator each iteration.
  * reference arm (`--impl reference`): the CPU restatement of the reference's algorithm (oracle/) on a bounded
    sample of the same workload, on all host cores: the Fourier-domain form of the reference's default
    numpy_fft / numpy_caching_fft backends (scipy.fft with workers=-1, exactly the reference's threading), with the
    coordinate-space form of its `numpy` backend timed beside it.  /root/reference is a pure-Python package that
    does not travel to the GPU box, so the oracle port - pinned to the reference's golden vectors - is the timed
    CPU implementation.

One JSON line on stdout (rank 0).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

if '--impl' in sys.argv and 'reference' in sys.argv:
    # The CPU arm uses every host core.  torchrun exports OMP_NUM_THREADS=1 to its workers, which would throttle the BLAS
    # behind numpy.einsum (round 1: 7.8 -> 2.8 sample-it/s under torchrun); the variables are read when numpy loads.
    for _v in ('OMP_NUM_THREADS', 'OPENBLAS_NUM_THREADS', 'MKL_NUM_THREADS'):
        os.environ[_v] = str(os.cpu_count() or 1)

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = 'sample-iterations/sec for 2-D shift-NMF MU at 1/2/4/8 B200; % of roofline'
UNIT = 'sample-iterations/s'

# the configurations of BASELINE.json (SURVEY 8): samples per GPU, channels, sample shape, atoms, atom shape
WORKLOADS = {
    'cfg1': dict(N=100, C=1, D=(1000,), M=5, A=(50,), text='1-D: 100 x 1 x 1000, 5 atoms x 50'),
    'cfg2': dict(N=64, C=3, D=(256, 256), M=16, A=(11, 11), text='2-D images: 64 x 3x256x256, 16 atoms 3x11x11'),
    'cfg3': dict(N=1024, C=1, D=(128, 128), M=32, A=(15, 15),
                 text='large-batch 2-D shard: 1024 x 1x128x128 per GPU (8192 over 8), 32 atoms 1x15x15'),
    'cfg4': dict(N=2048, C=1, D=(4096,), M=64, A=(128,), text='1-D signals: 2048 x 1x4096 per GPU, 64 atoms x 128'),
    'cfg5': dict(N=16, C=1, D=(512, 512), M=8, A=(64, 64), text='large-atom 2-D: 16 x 1x512x512, 8 atoms 1x64x64'),
}
CPU_SAMPLE = {'cfg1': 100, 'cfg2': 4, 'cfg3': 16, 'cfg4': 64, 'cfg5': 1}   # samples of the bounded CPU run


def flops_per_sample_iteration(w):
    """12*M*C*prod(D)*prod(A): 2 reconstructions + 4 correlations at 2 flop per MAC (SURVEY 8d)."""
    return 12.0 * w['M'] * w['C'] * float(np.prod(w['D'])) * float(np.prod(w['A']))


def hbm_bytes_per_sample_iteration(w):
    """Staged plan of DESIGN.md: H read 4x / written 1x, V read 2x, R written 2x / read 2x (fp32)."""
    T = float(np.prod([d + a - 1 for d, a in zip(w['D'], w['A'])]))
    return 4.0 * (5.0 * w['M'] * T + 6.0 * w['C'] * float(np.prod(w['D'])))


# -------------------------------------------------------------------------------------------------------------
# clocks during the timed region (B200_PROFILING.md)
# -------------------------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
              'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
              'clocks_event_reasons.sw_power_cap')

    def __init__(self, index: int):
        self.index, self.proc, self.lines, self.thread = index, None, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), f'--query-gpu={self.FIELDS}',
                                          '--format=csv,noheader,nounits', '-lms', '25'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._pump, daemon=True)
        self.thread.start()

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def stop(self, t0=None, t1=None):
        if self.proc is None:
            return None
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        for t, line in self.lines:
            if t0 is not None and not (t0 <= t <= t1 + 0.2):
                continue
            parts = [x.strip() for x in line.split(',')]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                smax.append(float(parts[1]))
            except ValueError:
                continue
            for name, val in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), parts[3:7]):
                if val.lower().startswith('active'):
                    reasons.add(name)
        if not sm:
            return None
        return {'sm_mhz': float(np.median(sm)), 'sm_max_mhz': float(max(smax)), 'reasons': sorted(reasons),
                'samples': len(sm)}


# -------------------------------------------------------------------------------------------------------------
# CPU baseline: the oracle port of the reference's numpy backend on a bounded sample
# -------------------------------------------------------------------------------------------------------------
def cpu_oracle_run(w, n_sample, steps, warmup, kind='caching_fft'):
    """Times the MU iteration of the CPU oracle (oracle/tnmf_oracle.py) on `n_sample` samples of workload `w`:
    OracleNMF_CachingFFT / OracleNMF_FFT (Fourier-domain forms, scipy.fft on all host threads) or OracleNMF
    (coordinate-space form).  Returns (sample-iterations/s, seconds per step)."""
    from oracle import tnmf_oracle as orc
    rng = np.random.default_rng(0)
    V = rng.random((n_sample, w['C'], *w['D']), dtype=np.float32)
    cls = {'caching_fft': orc.OracleNMF_CachingFFT, 'fft': orc.OracleNMF_FFT, 'direct': orc.OracleNMF}[kind]
    nmf = cls(n_atoms=w['M'], atom_shape=w['A'])
    np.random.seed(0)
    nmf.initialize(V)
    for _ in range(warmup):
        nmf.update_H()
        nmf.update_W()
    t0 = time.perf_counter()
    for _ in range(steps):
        nmf.update_H()
        nmf.update_W()
    dt = time.perf_counter() - t0
    return n_sample * steps / dt, dt / steps


def import_reference():
    """The UNMODIFIED reference package, if it travelled with the repo: `baseline/_ref` (pip install --target of
    /root/reference, git-ignored) - with the two `opt_einsum` entry points it uses mapped onto numpy.einsum when that
    package is absent (tests/golden/_shim, the same shim the golden vectors were generated with).  None otherwise."""
    ref_dir = os.path.join(ROOT, 'baseline', '_ref')
    if not os.path.isdir(os.path.join(ref_dir, 'tnmf')):
        return None
    try:
        import opt_einsum  # noqa: F401
    except ImportError:
        sys.path.insert(0, os.path.join(ROOT, 'tests', 'golden', '_shim'))
    sys.path.insert(0, ref_dir)
    try:
        from tnmf.TransformInvariantNMF import TransformInvariantNMF as RefNMF
        return RefNMF
    except Exception as exc:                                            # pylint: disable=broad-except
        print(f'reference package present but not importable: {exc!r}', file=sys.stderr)
        return None


def reference_run(RefNMF, w, n_sample, steps, warmup, backend):
    """Times the reference's own `fit` (stock facade, stock backend) on `n_sample` samples: the iteration loop only,
    clocked by the progress callback (which also switches the per-iteration energy evaluation off,
    tnmf/TransformInvariantNMF.py:342-346).  Returns (sample-iterations/s, seconds per step)."""
    rng = np.random.default_rng(0)
    V = rng.random((n_sample, w['C'], *w['D']), dtype=np.float32)
    stamps = []
    np.random.seed(0)
    nmf = RefNMF(n_atoms=w['M'], atom_shape=w['A'], backend=backend)
    nmf.fit(V, n_iterations=warmup + steps, progress_callback=lambda *_: stamps.append(time.perf_counter()) or True)
    dt = stamps[warmup + steps - 1] - stamps[warmup - 1]
    return n_sample * steps / dt, dt / steps


def run_reference(args, w):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    n_sample = CPU_SAMPLE[args.workload]
    n_direct = max(1, n_sample // 2)
    RefNMF = import_reference()
    beside = {}
    if RefNMF is not None:
        kind = 'reference'
        value, s_per_step = reference_run(RefNMF, w, n_sample, args.steps, max(args.warmup, 1), 'numpy_caching_fft')
        what = ('unmodified emdgroup/tnmf (baseline/_ref): TransformInvariantNMF(backend="numpy_caching_fft").fit, '
                'iteration loop clocked by the progress callback, scipy.fft workers=-1 (all host threads)')
        try:
            nv, _ = reference_run(RefNMF, w, n_direct, 1, 1, 'numpy')
            beside['numpy'] = {'value': nv, 'unit': UNIT, 'sample': f'{n_direct} samples, 1 warm-up + 1 timed iteration',
                               'what': 'unmodified reference, backend="numpy" (im2col + BLAS)'}
        except Exception as exc:                                        # pylint: disable=broad-except
            beside['numpy'] = {'unavailable': repr(exc)}
        pv, _ = cpu_oracle_run(w, n_sample, args.steps, max(args.warmup, 1), 'caching_fft')
        beside['oracle_port'] = {'value': pv, 'unit': UNIT, 'what': 'oracle.OracleNMF_CachingFFT on the same sample '
                                 '(the port that stands in where the reference package is absent)'}
    else:
        kind = 'port'
        value, s_per_step = cpu_oracle_run(w, n_sample, args.steps, args.warmup, 'caching_fft')
        what = ('oracle.OracleNMF_CachingFFT: restatement of the reference numpy_caching_fft backend (spectra of V, W, H '
                'cached between uses), scipy.fft workers=-1 (all host threads); the reference package is not on this box')
        dv, _ = cpu_oracle_run(w, n_direct, 1, 1, 'direct')
        beside['numpy_direct'] = {'value': dv, 'unit': UNIT, 'cores': 1,
                                  'sample': f'{n_direct} samples, 1 warm-up + 1 timed iteration',
                                  'what': 'oracle.OracleNMF: coordinate-space restatement of the reference numpy '
                                          'backend (single-threaded shift-and-add)'}
    sample = f'{n_sample} of {w["N"]} samples of {args.workload}, every step one full MU iteration'
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': 1e3 * s_per_step, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': f'{args.workload}: {w["text"]}', 'algorithm': 'batch MU', 'cpu_sample': sample,
                   'threads': {v: os.environ.get(v) for v in ('OMP_NUM_THREADS', 'OPENBLAS_NUM_THREADS')}},
        'cpu_baseline': dict({'value': value, 'unit': UNIT, 'cores': os.cpu_count(), 'kind': kind, 'sample': sample,
                              'what': what}, **beside),
        'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line), flush=True)


# -------------------------------------------------------------------------------------------------------------
# own arm
# -------------------------------------------------------------------------------------------------------------
def measure_fp32_peak(lib, torch, device):
    """FP32-FMA pipe peak of this GPU in TFLOP/s, measured with the library's probe kernel (best of 5)."""
    import ctypes
    sink = torch.zeros(64, dtype=torch.float32, device=device)
    flops = ctypes.c_double(0.0)
    st = torch.cuda.current_stream(device).cuda_stream
    best = 0.0
    for i in range(7):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        rc = lib.tnmf_fp32_peak_probe(sink.data_ptr(), 4096, ctypes.byref(flops), st)
        b.record()
        torch.cuda.synchronize(device)
        if rc != 0:
            return None
        if i >= 2:
            best = max(best, flops.value / (a.elapsed_time(b) * 1e-3) / 1e12)
    return best


def time_steps(nmf_cls, w, n_local, device, args, steps, warmup, sharded, dist):
    """Device time (ms, max over ranks when sharded) of `steps` batch MU iterations on `n_local` resident samples per
    rank: the same `_batch_step` replay the headline number times."""
    import torch
    gen = torch.Generator(device=device)
    gen.manual_seed(4321 + int(os.environ.get('RANK', '0')))
    V = torch.rand((n_local, w['C'], *w['D']), dtype=torch.float32, device=device, generator=gen)
    nmf = nmf_cls(n_atoms=w['M'], atom_shape=w['A'], backend='b200', init='device', distributed=sharded,
                  input_is_local_shard=True, equal_shards=True, kernel_path=args.kernel_path,
                  cuda_graph=not args.no_cuda_graph)
    nmf._initialize_matrices(V, keep_W=False)                            # pylint: disable=protected-access
    step = nmf._batch_step()                                             # pylint: disable=protected-access
    for _ in range(warmup):
        step()
    torch.cuda.synchronize(device)
    if sharded:
        dist.barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(steps):
        step()
    ev1.record()
    torch.cuda.synchronize(device)
    ms = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device=device)
    if sharded:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    families = dict(nmf._backend.kernel_families(), kernels=nmf._backend.kernel_names())   # pylint: disable=protected-access
    finite = bool(torch.isfinite(nmf.energy_device()).item())
    del nmf, V, step
    torch.cuda.empty_cache()
    return float(ms.item()), families, finite


def measure_cfg3(nmf_cls, device, args, world, rank, dist):
    """BASELINE config 3 on the record of every run: 8192 samples of 1x128x128, 32 atoms 15x15, sharded over the ranks
    (STRONG scaling: 8192 / N samples per GPU, W-gradient all-reduce every iteration), and - on rank 0, the other ranks
    waiting - the same 8192 samples on one GPU, so that the line carries its own 1 -> N efficiency."""
    w3 = WORKLOADS['cfg3']
    total, steps, warmup = 8192, 5, 3
    if total % world:
        return {'skipped': f'{total} samples do not split evenly over {world} ranks'}
    ms_n, families, finite = time_steps(nmf_cls, w3, total // world, device, args, steps, warmup, world > 1, dist)
    out = {'workload': 'cfg3: 8192 x 1x128x128, 32 atoms 1x15x15, sample-sharded (strong scaling)', 'samples': total,
           'samples_per_gpu': total // world, 'steps': steps, 'warmup': warmup, 'ms_per_step': ms_n / steps,
           'value': total * steps / (ms_n * 1e-3), 'unit': UNIT, 'kernel_path': families, 'finite': finite}
    if world > 1:
        ms_1 = None
        if rank == 0:
            ms_1, _, _ = time_steps(nmf_cls, w3, total, device, args, 3, 2, False, dist)
        dist.barrier()
        if rank == 0:
            out['single_gpu'] = {'ms_per_step': ms_1 / 3, 'value': total * 3 / (ms_1 * 1e-3), 'steps': 3,
                                 'what': 'all 8192 samples on rank 0 alone, same run'}
            out['speedup'] = (ms_1 / 3) / (ms_n / steps)
            out['efficiency'] = out['speedup'] / world
    return out


DUMP_BYTES = 64 << 20           # most that --dump-outputs writes
H_SAMPLE = 1 << 22              # elements of H kept when all of it would not fit


def seed_start_values(nmf, device, rank):
    """Overwrite the library's random start values with ones drawn here (1 - U[0, 1), W normalised over its shift axes
    like the facade does): they then depend neither on how a build lays out H nor on the order it draws in.  W is the
    same on every rank, H differs per rank like the samples do."""
    import torch
    W, H = nmf.W_device, nmf.H_device
    gen = torch.Generator(device=device)
    gen.manual_seed(99)
    W0 = 1 - torch.rand(W.shape, dtype=W.dtype, device=device, generator=gen)
    W.copy_(W0 / W0.sum(dim=nmf._axes_W_normalization, keepdim=True))  # pylint: disable=protected-access
    gen.manual_seed(5678 + rank)
    H.copy_(1 - torch.rand(H.shape, dtype=H.dtype, device=device, generator=gen))
    torch.cuda.empty_cache()        # the buffers the steps allocate are then placed as if the temporaries never existed


def dump_outputs(out_dir, be, W, H):
    """W and H as .npy files in their own dtype.  An H whose bytes together with W's exceed DUMP_BYTES is written as
    H_sample.npy: its elements at the flat C-order indices sorted(numpy.random.default_rng(0).choice(H.numel(),
    H_SAMPLE, replace=False)), the same indices on every run with the same arguments."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for stale in ('H.npy', 'H_sample.npy'):           # a run with other arguments may have left the other form
        if os.path.exists(os.path.join(out_dir, stale)):
            os.remove(os.path.join(out_dir, stale))
    np.save(os.path.join(out_dir, 'W.npy'), be.to_ndarray(W))
    if (W.numel() + H.numel()) * H.element_size() <= DUMP_BYTES:
        np.save(os.path.join(out_dir, 'H.npy'), be.to_ndarray(H))
    else:
        idx = np.sort(np.random.default_rng(0).choice(H.numel(), H_SAMPLE, replace=False))
        np.save(os.path.join(out_dir, 'H_sample.npy'), be.to_ndarray(torch.take(H, torch.from_numpy(idx).to(H.device))))


def run_b200(args, w):
    import torch
    import torch.distributed as dist
    from tnmf_b200 import TransformInvariantNMF, _lib

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise RuntimeError('bench.py --impl b200 needs a CUDA device (tnmf_b200 has no CPU fallback)')
    torch.cuda.set_device(local_rank)
    device = torch.device('cuda', local_rank)
    if world > 1:
        dist.init_process_group('nccl', device_id=device)
    lib = _lib.load()

    n_local = w['N']
    gen = torch.Generator(device=device)
    gen.manual_seed(1234 + rank)
    V = torch.rand((n_local, w['C'], *w['D']), dtype=torch.float32, device=device, generator=gen)
    torch.manual_seed(99)       # the start values the library draws itself in the e2e and cfg3 legs below (those of
                                # the timed loop are replaced by seed_start_values)

    nmf = TransformInvariantNMF(n_atoms=w['M'], atom_shape=w['A'], backend='b200', init='device',
                                input_is_local_shard=True, kernel_path=args.kernel_path,
                                cuda_graph=not args.no_cuda_graph)
    be = nmf._backend                                                    # pylint: disable=protected-access
    nmf._initialize_matrices(V, keep_W=False)                            # pylint: disable=protected-access
    seed_start_values(nmf, device, rank)

    # one batch MU iteration exactly as fit_batch runs it: eager the first time, CUDA-graph replays afterwards
    step = nmf._batch_step()                                             # pylint: disable=protected-access

    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize(device)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(device)

    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    launches0 = be.launches
    peer_active = nmf._peer is not None                                  # pylint: disable=protected-access
    t_wall0 = time.perf_counter()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        step()
    ev1.record()
    torch.cuda.synchronize(device)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(device)
    t_wall1 = time.perf_counter()
    launches = be.launches - launches0
    clocks = sampler.stop(t_wall0, t_wall1) if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, be, nmf.W_device, nmf.H_device)
    # per-kernel durations: the same iteration launched eagerly with a CUDA-event pair around every hot-path call
    be.kernel_events = {}
    n_probe = min(args.steps, 5)
    for _ in range(n_probe):
        step()
    torch.cuda.synchronize(device)
    events, be.kernel_events = be.kernel_events, None

    ms = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = float(ms.item())
    value = world * n_local * args.steps / (ms_total * 1e-3)

    # per-kernel averages over the timed region (CUDA events on the launching stream)
    kern_ms = {k: float(np.mean([a.elapsed_time(b) for a, b in v])) for k, v in events.items()}
    kern_calls = {k: len(v) / n_probe for k, v in events.items()}
    energy = float(nmf._energy_function())                               # pylint: disable=protected-access
    if not np.isfinite(energy):
        raise RuntimeError('non-finite energy after the timed iterations')

    # ---- end to end through the public API: host batch -> fit() -> host results --------------------------------
    V_host = V.cpu().pin_memory()
    e2e_iters = args.steps
    nmf_e = TransformInvariantNMF(n_atoms=w['M'], atom_shape=w['A'], backend='b200', init='device',
                                  input_is_local_shard=True, equal_shards=True, kernel_path=args.kernel_path,
                                  cuda_graph=not args.no_cuda_graph)
    nmf_e.fit(V_host, n_iterations=3)                                    # warm-up (allocations, graph capture)
    torch.cuda.synchronize(device)
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    nmf_e.fit(V_host, n_iterations=e2e_iters)
    W_host = nmf_e.W
    e_host = nmf_e._energy_function()                                    # pylint: disable=protected-access
    torch.cuda.synchronize(device)
    dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    e2e_value = world * n_local * e2e_iters / float(dt.item())
    h2d = V_host.numel() * 4 / e2e_iters
    d2h = (W_host.size * 4 + 8) / e2e_iters
    assert np.isfinite(e_host)

    cfg3 = None
    if args.workload == 'cfg2' and not args.no_cfg3:
        del nmf_e, V_host
        torch.cuda.empty_cache()
        cfg3 = measure_cfg3(TransformInvariantNMF, device, args, world, rank, dist)

    if rank != 0:
        finish_ranks(world, dist)
        return

    # ---- roofline of the dominant kernel -------------------------------------------------------------------------
    fp32_peak = measure_fp32_peak(lib, torch, device)
    peaks = {}
    try:
        with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as f:
            peaks = json.load(f)
    except OSError:
        pass
    hbm_peak, hbm_src = (peaks['hbm_gbs'], 'measured') if 'hbm_gbs' in peaks else (6650.0, 'fallback')
    macs = w['M'] * w['C'] * float(np.prod(w['D'])) * float(np.prod(w['A'])) * n_local
    kernel_flops = {'reconstruct': 2 * macs, 'update_h': 4 * macs, 'gradient_w': 4 * macs}
    share = {k: kern_ms[k] * kern_calls[k] for k in kern_ms}
    dominant = max((k for k in share if k in kernel_flops), key=lambda k: share[k])
    achieved = kernel_flops[dominant] / (kern_ms[dominant] * 1e-3) / 1e12
    step_ms = ms_total / args.steps
    flops_step = flops_per_sample_iteration(w) * n_local
    bytes_step = hbm_bytes_per_sample_iteration(w) * n_local
    traffic, traffic_src = None, None
    try:
        with open(os.path.join(ROOT, 'profiles', 'ncu_traffic.json')) as f:
            entry = json.load(f).get(args.workload, {}).get(dominant)
        if entry and entry.get('family') == be.kernel_families().get(dominant):
            traffic, traffic_src = entry['bytes'], entry['source']
    except (OSError, ValueError):
        pass
    families = be.kernel_families()
    # tensor-pipe denominator of the 3xTF32 kernels: dense TF32 = half the measured dense bf16 rate, three MMAs per
    # product -> useful flops at most bf16/6
    bf16_peak, bf16_src = (peaks['bf16_tflops'], 'measured') if 'bf16_tflops' in peaks else (2250.0, 'nominal')
    tc_peak = bf16_peak / 6.0
    per_kernel = {}
    for k in kernel_flops:
        if k not in kern_ms:
            continue
        tf = kernel_flops[k] / (kern_ms[k] * 1e-3) / 1e12
        on_tc = families.get(k) == 'tc'
        pk = tc_peak if on_tc else fp32_peak
        per_kernel[k] = {'family': families.get(k), 'bound': 'tensor (3xTF32)' if on_tc else 'fp32', 'ms': kern_ms[k],
                         'launches_per_step': kern_calls[k], 'achieved_tflops': tf, 'peak_tflops': pk,
                         'frac': (tf / pk) if pk else None}
    dom = per_kernel[dominant]
    roofline = {
        'bound': 'tensor' if families.get(dominant) == 'tc' else 'fp32', 'kernel': dominant, 'achieved': achieved,
        'peak': dom['peak_tflops'], 'unit': 'TFLOP/s', 'frac': dom['frac'], 'traffic': traffic,
        'traffic_source': traffic_src, 'traffic_unit': 'bytes per launch (dram read + write, ncu)',
        'peak_source': 'fp32: FP32-FMA probe kernel of libtnmf_b200.so timed in this run (MEASURED_PEAKS.json holds no '
                       'FP32 figure; nominal 148 SM x 128 FMA x 2 x 1.965 GHz = 74.4).  tensor (3xTF32): '
                       f'{bf16_src} dense bf16 {bf16_peak:.0f} TFLOP/s / 2 (TF32) / 3 (MMAs per product)',
        'kernels': per_kernel,
        'kernel_ms': kern_ms, 'kernel_launches_per_step': kern_calls,
        'kernel_share_of_step': {k: share[k] / step_ms for k in share},
        'whole_step': {'tflops': flops_step / (step_ms * 1e-3) / 1e12,
                       'frac_of_fp32_peak': (flops_step / (step_ms * 1e-3) / 1e12 / fp32_peak) if fp32_peak else None,
                       'algorithmic_hbm_gbs': bytes_step / (step_ms * 1e-3) / 1e9,
                       'frac_of_hbm_peak': bytes_step / (step_ms * 1e-3) / 1e9 / hbm_peak,
                       'hbm_peak_gbs': hbm_peak, 'hbm_peak_source': hbm_src},
    }

    # ---- CPU baseline on this box's host cores (bounded sample) ------------------------------------------------
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        n_sample = CPU_SAMPLE[args.workload]
        RefNMF = import_reference()
        sample = f'{n_sample} of {w["N"]} samples of {args.workload}, 1 warm-up + 3 timed MU iterations'
        if RefNMF is not None:
            cpu_value, _ = reference_run(RefNMF, w, n_sample, 3, 1, 'numpy_caching_fft')
            cpu = {'value': cpu_value, 'unit': UNIT, 'cores': os.cpu_count(), 'kind': 'reference', 'sample': sample,
                   'what': 'unmodified emdgroup/tnmf (baseline/_ref), backend="numpy_caching_fft", all host threads'}
        else:
            cpu_value, _ = cpu_oracle_run(w, n_sample, 3, 1, 'caching_fft')
            n_direct = max(1, n_sample // 2)
            direct_value, _ = cpu_oracle_run(w, n_direct, 1, 1, 'direct')
            cpu = {'value': cpu_value, 'unit': UNIT, 'cores': os.cpu_count(), 'kind': 'port', 'sample': sample,
                   'what': 'oracle.OracleNMF_CachingFFT: restatement of the reference numpy_caching_fft backend, '
                           'scipy.fft workers=-1 (all host threads)',
                   'numpy_direct': {'value': direct_value, 'unit': UNIT, 'cores': 1,
                                    'sample': f'{n_direct} samples, 1 warm-up + 1 timed iteration',
                                    'what': 'oracle.OracleNMF: coordinate-space restatement of the reference numpy '
                                            'backend (single-threaded shift-and-add)'}}

    line = {
        'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': step_ms, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32',
        'data': 'synthetic',
        'config': {'workload': f'{args.workload}: {w["text"]}', 'algorithm': 'batch MU (H update, W update)',
                   'samples_per_gpu': n_local, 'global_samples': world * n_local,
                   'parallelism': (f'sample-sharded x{world}, W gradient summed over the ranks '
                                   + ('inside the W-update kernel over NVLink peer memory' if peer_active
                                      else 'by an NCCL all-reduce')) if world > 1 else 'single GPU',
                   'kernel_path': be.kernel_families(), 'kernels': be.kernel_names(), 'launch': 'CUDA graph replay of one iteration' if nmf._cuda_graph  # pylint: disable=protected-access
                   else 'eager launches',
                   'l2': 'working set (V, R, H) exceeds the 126 MB L2; no explicit flush'
                   if (bytes_step / 5 > 126e6) else 'working set fits L2; iterations overwrite H and R in between',
                   'final_energy': energy, 'cfg3': cfg3},
        'roofline': roofline, 'cpu_baseline': cpu,
        'e2e': {'value': e2e_value, 'unit': UNIT, 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
                'what': f'fit(V_host_pinned, n_iterations={e2e_iters}) + W and energy read back; upload, device init '
                        f'and download inside the timed region, bytes amortised over the iterations'},
        'gpu_launches': launches, 'clocks': clocks,
    }
    print(json.dumps(line), flush=True)
    finish_ranks(world, dist)


def finish_ranks(world, dist):
    """End of a multi-rank run.  The step graphs hold captured NCCL kernels; tearing the communicator down under them
    was seen to hang at interpreter exit (the JSON line already printed), so the ranks meet once more and leave without
    running the destructors."""
    if world > 1:
        import torch
        torch.cuda.synchronize()
        dist.barrier()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=50,
                    help='timed iterations of the headline loop and of the e2e leg; the cfg3 leg of a cfg2 run always '
                         'times 5 (see measure_cfg3)')
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--workload', default='cfg2', choices=sorted(WORKLOADS))
    ap.add_argument('--kernel-path', default='auto', choices=['auto', 'generic', 'tiled', 'tma', 'tc'])
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-cuda-graph', action='store_true')
    ap.add_argument('--no-cfg3', action='store_true', help='skip the cfg3 strong-scaling leg of the cfg2 run')
    ap.add_argument('--samples', type=int, default=0, help='samples per GPU instead of the workload default '
                    '(e.g. --workload cfg5 --samples 512: BASELINE config 5 at its full batch)')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write W and H after the last timed step as .npy files to DIR (own arm only)')
    args = ap.parse_args()
    if args.dump_outputs and args.impl != 'b200':
        ap.error('--dump-outputs applies to --impl b200')
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    args.warmup = max(args.warmup, 3) if args.impl == 'b200' else args.warmup
    w = dict(WORKLOADS[args.workload])
    if args.samples > 0:
        w['N'] = args.samples
        w['text'] = f"{w['text']} [--samples {args.samples}]"
    world = int(os.environ.get('WORLD_SIZE', '1'))
    if args.impl == 'b200' and args.gpus != world and world == 1 and args.gpus > 1:
        # convenience: relaunch under torchrun when asked for several GPUs from a plain `python bench.py`
        cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', f'--nproc-per-node={args.gpus}',
               '--master-addr', '127.0.0.1', '--master-port', os.environ.get('MASTER_PORT', '29511'),
               os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    if args.impl == 'reference':
        run_reference(args, w)
    else:
        run_b200(args, w)


if __name__ == '__main__':
    main()
