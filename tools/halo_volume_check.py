"""
Halo (row) sharding of ONE volume over the GPUs of a box, over NCCL (tnmf_b200.RowShardedNMF with three shift axes):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port 29513 \
        tools/halo_volume_check.py [--out FILE]

(a) correctness: 10 iterations on one 1x96^3 volume, 8 atoms of 7^3, cut into N bands of z-planes, against the same fit
    on rank 0 alone (tnmf_b200.TransformInvariantNMF, same seeded start): W / H max-relative differences;
(b) timing: one MU step of one 1x512^3 volume, 8 atoms of 7^3 (CUDA events around the timed steps, max over ranks);
(c) the same with the plane window off (the bands update their halo planes and correlate with a zero-haloed copy of H),
    so the window's gain is measured rather than estimated.
Compare the N = 1 run's step time with the others' for speedup and efficiency.  One JSON line on rank 0 (also written
to --out); the device name and power limit are part of it.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tnmf_b200 import RowShardedNMF, TransformInvariantNMF  # noqa: E402
from tnmf_b200.halo import B200Ops  # noqa: E402

ATOMS, ATOM = 8, (7, 7, 7)


def _power_limit():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader', '-i',
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        return q.stdout.strip() or None
    except (OSError, subprocess.SubprocessError):
        return None


def _time_steps(V, plane_window, warmup, steps, device):
    np.random.seed(12)
    nmf = RowShardedNMF(ATOMS, ATOM, ops=B200Ops(plane_window=plane_window))
    nmf.initialize(V)
    for _ in range(warmup):
        nmf.step(0.05)
    torch.cuda.synchronize(device)
    dist.barrier()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        nmf.step(0.05)
    b.record()
    torch.cuda.synchronize(device)
    dt = torch.tensor([a.elapsed_time(b) / steps], dtype=torch.float64, device=device)
    dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    band = [nmf.plan['t0'], nmf.plan['t1']]
    names = nmf.ops.be.kernel_names()
    del nmf
    torch.cuda.empty_cache()
    return float(dt.item()), band, names


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--size', type=int, default=512, help='edge of the timed volume')
    ap.add_argument('--check-size', type=int, default=96, help='edge of the volume of the correctness check')
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=2)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    world, rank, local = int(os.environ['WORLD_SIZE']), int(os.environ['RANK']), int(os.environ['LOCAL_RANK'])
    torch.cuda.set_device(local)
    device = torch.device('cuda', local)
    dist.init_process_group('nccl', device_id=device)
    out = {'world': world, 'device': torch.cuda.get_device_name(device), 'power_limit': _power_limit(),
           'atoms': f'{ATOMS} x {"x".join(map(str, ATOM))}'}

    # (a) correctness
    c = args.check_size
    V = np.random.default_rng(2).random((1, 1, c, c, c), dtype=np.float32)
    iters = 10
    np.random.seed(11)
    nmf = RowShardedNMF(ATOMS, ATOM)
    nmf.fit(V, n_iterations=iters, sparsity_H=0.05)
    H, W = nmf.gather_H(), nmf.W
    out['check_problem'] = f'1x{c}^3, {iters} iterations, sparsity 0.05'
    out['check_kernels'] = nmf.ops.be.kernel_names()
    del nmf
    torch.cuda.empty_cache()
    ok = True
    if rank == 0:
        np.random.seed(11)
        one = TransformInvariantNMF(n_atoms=ATOMS, atom_shape=ATOM, backend='b200', init='numpy', distributed=False)
        one.fit(V, n_iterations=iters, sparsity_H=0.05)
        out['W_max_rel'] = float(np.abs(W - one.W).max() / np.abs(one.W).max())
        out['H_max_rel'] = float(np.abs(H - one.H).max() / np.abs(one.H).max())
        ok = out['W_max_rel'] <= 1e-3 and out['H_max_rel'] <= 1e-3
        del one
        torch.cuda.empty_cache()
    dist.barrier()

    # (b), (c) timing
    s = args.size
    Vbig = np.random.default_rng(3).random((1, 1, s, s, s), dtype=np.float32)
    out['timing_problem'] = f'1x{s}^3, sparsity 0.05, {args.steps} steps after {args.warmup}'
    out['ms_per_step'], out['band'], out['kernels'] = _time_steps(Vbig, True, args.warmup, args.steps, device)
    out['ms_per_step_no_window'], _, _ = _time_steps(Vbig, False, args.warmup, args.steps, device)
    out['window_gain'] = out['ms_per_step_no_window'] / out['ms_per_step']
    T0 = s + ATOM[0] - 1
    flop = 12.0 * ATOMS * 1 * s ** 3 * float(np.prod(ATOM))        # 12 M C prod(D) prod(A) per MU step
    out['tflops_per_s'] = flop / (out['ms_per_step'] * 1e-3) / 1e12
    out['owned_planes_per_band'] = T0 / world
    out['ok'] = bool(ok)
    if rank == 0:
        line = json.dumps(out)
        print(line, flush=True)
        if args.out:
            with open(args.out, 'w') as f:
                f.write(line + '\n')
    torch.cuda.synchronize(device)
    dist.barrier()
    dist.destroy_process_group()
    sys.exit(0 if ok else 1)


if __name__ == '__main__':
    main()
