"""
Volumetric (3-D) MU step on the B200: 16 samples of 1 x 64^3, 8 atoms of 7 x 7 x 7, 'valid' (H = 176 MB, more than
the 126 MB of L2).  Prints one JSON line (and writes it to --out): GPU name and power limit, ms per MU step from CUDA
events over graph-replayed steps, per-kernel ms from `B200_Backend.kernel_events`, useful TFLOP/s (12 N M C prod(D)
prod(A) per step) and its share of the 277.2 TFLOP/s 3xTF32 ceiling (DESIGN.md §4).  For comparison it times
kernel_path='generic' and the same step written with torch conv3d (cuDNN, fp32, TF32 off), the formulation of the
reference's PyTorch backend, after checking that formulation against the oracle at a small size.

    python tools/bench_3d.py [--steps 50] [--warmup 5] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import tnmf_oracle as orc  # noqa: E402

N, C, M, D, A = 16, 1, 8, (64, 64, 64), (7, 7, 7)
CEILING_TFLOPS = 277.2
EPS = 1e-9


def gpu_info():
    q = subprocess.run(['nvidia-smi', '-i', '0', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return q.stdout.strip()


def flops_per_step(n):
    return 12.0 * n * M * C * np.prod(D) * np.prod(A)


def time_graph(step, steps, warmup):
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
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        g.replay()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / steps


def library_step(path, V, steps, warmup, kernels=False):
    from tnmf_b200 import B200_Backend
    be = B200_Backend(reconstruction_mode='valid', kernel_path=path)
    Wd, Hd = be.initialize(V, A, M, None, (-3, -2, -1))
    g0 = torch.Generator(device='cuda').manual_seed(1)
    Wd.copy_(torch.rand(Wd.shape, generator=g0, device='cuda'))
    Hd.copy_(torch.rand(Hd.shape, generator=g0, device='cuda'))
    grad = torch.empty((2, *Wd.shape), dtype=Wd.dtype, device=Wd.device)

    def step():
        be.update_H(V, Wd, Hd)
        be.apply_W_update(Wd, be.gradient_W(V, Wd, Hd, slice(None), grad))

    out = {'kernel_names': be.kernel_names(N)}
    if path == 'generic':                                   # seconds per step: eager, no graph
        step()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(steps):
            step()
        b.record()
        b.synchronize()
        out['ms_per_step'] = a.elapsed_time(b) / steps
        out['steps'] = steps
        return out
    out['ms_per_step'] = time_graph(step, steps, warmup)
    out['steps'] = steps
    if kernels:                                             # a run of its own: events around every library call
        be.kernel_events = {}
        for _ in range(10):
            step()
        torch.cuda.synchronize()
        out['kernel_ms'] = {k: float(np.mean([x.elapsed_time(y) for x, y in v])) for k, v in be.kernel_events.items()}
        out['kernel_calls_per_step'] = {k: len(v) / 10 for k, v in be.kernel_events.items()}
        be.kernel_events = None
    return out


# ---- the reference's PyTorch formulation (conv3d; cuDNN) ----------------------------------------------------------
def conv_R(W, H):
    return F.conv3d(H, W.flip((2, 3, 4)).transpose(0, 1))


def conv_grad_H(X, W):
    return F.conv3d(X, W, padding=tuple(a - 1 for a in A))


def conv_grad_W(X, H):
    return F.conv3d(H.transpose(0, 1), X.transpose(0, 1)).flip((2, 3, 4))


def check_conv_against_oracle():
    rng = np.random.default_rng(4)
    V = rng.random((2, C, 9, 10, 11))
    W = rng.random((3, C) + A)
    H = rng.random((2, 3) + orc.transform_shape('valid', V.shape[2:], A))
    t = lambda x: torch.from_numpy(x).cuda()
    err = lambda a, b: float(np.abs(a.cpu().numpy() - b).max() / np.abs(b).max())
    R = conv_R(t(W), t(H))
    nh, _ = orc.reconstruction_gradient_H(V, W, H)
    nw, _ = orc.reconstruction_gradient_W(V, W, H)
    e = max(err(R, orc.reconstruct(W, H)), err(conv_grad_H(t(V), t(W)), nh), err(conv_grad_W(t(V), t(H)), nw))
    assert e < 1e-10, e
    return e


def cudnn_step(V, steps, warmup):
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    Vd = torch.as_tensor(V).cuda()
    g0 = torch.Generator(device='cuda').manual_seed(1)
    W = torch.rand((M, C) + A, generator=g0, device='cuda')
    H = torch.rand((N, M) + tuple(d + a - 1 for d, a in zip(D, A)), generator=g0, device='cuda')

    def step():
        R = conv_R(W, H)
        H.mul_(conv_grad_H(Vd, W)).div_(conv_grad_H(R, W).add_(EPS))
        R = conv_R(W, H)
        W.mul_(conv_grad_W(Vd, H)).div_(conv_grad_W(R, H).add_(EPS))
        W.div_(W.sum(dim=(2, 3, 4), keepdim=True))

    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        step()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / steps


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n\n')[0])
    ap.add_argument('--steps', type=int, default=50)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--generic-steps', type=int, default=3)
    ap.add_argument('--cudnn-steps', type=int, default=10)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('bench_3d.py needs a CUDA device')
    V = np.random.default_rng(0).random((N, C) + D).astype(np.float32)
    res = {'gpu': gpu_info(), 'problem': {'N': N, 'C': C, 'M': M, 'D': D, 'A': A, 'mode': 'valid'},
           'flops_per_step': flops_per_step(N)}
    tc = library_step('auto', V, args.steps, args.warmup, kernels=True)
    tc['tflops'] = flops_per_step(N) / tc['ms_per_step'] / 1e9
    tc['fraction_of_3xtf32_ceiling'] = tc['tflops'] / CEILING_TFLOPS
    res['auto'] = tc
    res['generic'] = library_step('generic', V, args.generic_steps, 0)
    res['cudnn_conv3d'] = {'oracle_check_max_rel_err': check_conv_against_oracle(),
                           'ms_per_step': cudnn_step(V, args.cudnn_steps, 2), 'steps': args.cudnn_steps}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
