"""
Kullback-Leibler MU step against the Frobenius MU step on the B200, in the same run: cfg2 (64 x 3x256x256, 16 atoms
3x11x11) and one GPU's shard of cfg3 (1024 x 1x128x128, 32 atoms 15x15), float32, 'valid'.

Each step (H update, W gradient, W update) is captured into a CUDA graph; the two graphs are replayed in alternating
blocks of --steps and timed with CUDA events, for --reps rounds, so that both see the same state of the machine.  A run of
its own then records CUDA events around every library call (`B200_Backend.kernel_events`: reconstruction, quotient, H
update, W gradient, W update).  One JSON line with the GPU name and power limit goes to stdout and to --out.

    python tools/bench_kl.py [--steps 20] [--reps 5] [--warmup 3] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

WORKLOADS = {
    'cfg2': dict(N=64, C=3, D=(256, 256), M=16, A=(11, 11)),
    'cfg3_shard': dict(N=1024, C=1, D=(128, 128), M=32, A=(15, 15)),
}


def gpu_info():
    q = subprocess.run(['nvidia-smi', '-i', str(torch.cuda.current_device()),
                        '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return q.stdout.strip()


def setup(w, divergence, V):
    from tnmf_b200 import B200_Backend
    be = B200_Backend(reconstruction_mode='valid', init='device')      # (a host draw of the cfg3 H would be 5 GB)
    Wd, Hd = be.initialize(V, w['A'], w['M'], None, (-2, -1))
    g0 = torch.Generator(device='cuda').manual_seed(1)
    Wd.copy_(torch.rand(Wd.shape, generator=g0, device='cuda'))
    be.normalize(Wd, (-2, -1))
    Hd.copy_(torch.rand(Hd.shape, generator=g0, device='cuda'))
    grad = torch.empty((2, *Wd.shape), dtype=Wd.dtype, device=Wd.device)
    kw = {} if divergence == 'frobenius' else {'divergence': divergence}

    def step():
        be.update_H(V, Wd, Hd, **kw)
        be.apply_W_update(Wd, be.gradient_W(V, Wd, Hd, slice(None), grad, **kw))
    return be, step


def capture(step, warmup):
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(warmup):
            step()
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        step()
    g.replay()
    torch.cuda.synchronize()
    return g


def time_replays(g, steps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        g.replay()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / steps


def kernel_times(be, step, calls=10):
    be.kernel_events = {}
    for _ in range(calls):
        step()
    torch.cuda.synchronize()
    out = {k: round(float(np.mean([x.elapsed_time(y) for x, y in v])), 4) for k, v in be.kernel_events.items()}
    per_step = {k: len(v) / calls for k, v in be.kernel_events.items()}
    be.kernel_events = None
    return out, per_step


def run(name, w, steps, reps, warmup):
    g0 = torch.Generator(device='cuda').manual_seed(0)
    V = torch.rand((w['N'], w['C']) + w['D'], generator=g0, device='cuda')
    legs = {d: setup(w, d, V) for d in ('frobenius', 'kl')}
    graphs = {d: capture(step, warmup) for d, (_, step) in legs.items()}
    times = {d: [] for d in legs}
    for _ in range(reps):
        for d in ('frobenius', 'kl'):
            times[d].append(time_replays(graphs[d], steps))
    out = {'shape': f"{w['N']} x {w['C']}x{'x'.join(map(str, w['D']))}, {w['M']} atoms {'x'.join(map(str, w['A']))}",
           'kernel_names': legs['kl'][0].kernel_names(w['N'])}
    for d, (be, step) in legs.items():
        ms, per_step = kernel_times(be, step)
        out[d] = {'ms_per_step_median': round(float(np.median(times[d])), 4),
                  'ms_per_step_reps': [round(t, 4) for t in times[d]],
                  'kernel_ms': ms, 'calls_per_step': per_step}
    out['kl_over_frobenius'] = round(out['kl']['ms_per_step_median'] / out['frobenius']['ms_per_step_median'], 4)
    del legs, graphs
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--workloads', default=','.join(WORKLOADS))
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('bench_kl.py needs a CUDA device')
    res = {'tool': 'bench_kl', 'gpu': gpu_info(), 'steps': args.steps, 'reps': args.reps,
           'timing': 'CUDA events around graph replays, KL and Frobenius alternating',
           'workloads': {n: run(n, WORKLOADS[n], args.steps, args.reps, args.warmup) for n in args.workloads.split(',')}}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
