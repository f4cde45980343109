#!/usr/bin/env python
"""Time what a per-weight Gaussian prior costs.

1. The captured train step (GraphedTrainStep: sample_elbo[_lr] + backward + FusedAdam in one CUDA graph) with the
   model_params prior against the same net after posterior_to_prior(), at two shapes:
     cfg2: 784-1200-1200-10, weight sampling, TF32, B = 128, S = 2, mixture prior (the network-level route);
     cfg3: 784-1200-1200-10, local reparameterisation, fp32, B = 128, S = 2.
   The configurations alternate inside every round; each timed sample is ONE replay between CUDA events after a write
   of 256 MB that evicts the 126 MB L2 (outside the events).  Median and 10th / 90th percentile in microseconds.
2. Each new kernel alone at the cfg2 parameter count (one launch over the 6 tensors of the net, Philox eps), L2
   flushed before every launch: median time, and the bytes it must move (16 B per weight or bias forward: mu, rho and
   the prior's two values; 32 B backward: those plus both gradients read and written) over that time against the
   7.7 TB/s HBM3e peak of the B200 data sheet.
The device name and its power limit are printed with the times.
usage: python tools/time_gauss_prior.py [--rounds 300]"""
import argparse
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bnn_b200  # noqa: E402
from bnn_b200 import _lib as L  # noqa: E402
from bnn_b200 import functional as F  # noqa: E402

B, S, DIMS = 128, 2, (784, 1200, 1200, 10)
HBM_PEAK = 7.7e12


def device_info():
    name = torch.cuda.get_device_name()
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader',
                            f'--id={torch.cuda.current_device()}'], capture_output=True, text=True, timeout=30)
        power = q.stdout.strip() or 'unknown'
    except (OSError, subprocess.SubprocessError):
        power = 'unknown'
    return name, power


def make_net(lr):
    mp = dict(input_shape=DIMS[0], classes=DIMS[-1], batch_size=B, hidden_units=list(DIMS[1:-1]),
              mode='classification', mu_init=[-0.2, 0.2], rho_init=[-5, -4],
              prior_init=[1.0] if lr else [0.5, 0, -6], mixture_prior=not lr, local_reparam=lr, tf32=not lr)
    torch.manual_seed(0)
    return bnn_b200.BayesianNetwork(mp).cuda().train()


def make_step(lr, prior, x, y):
    net = make_net(lr)
    if prior:
        net.posterior_to_prior()
    opt = bnn_b200.FusedAdam(net.parameters(), lr=1e-3)
    bnn_b200.manual_seed(1)
    return bnn_b200.GraphedTrainStep(net, opt, x, y, S, beta=0.01, warmup=3), net


def time_it(fn, flush, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t = []
    for _ in range(n):
        flush.zero_()
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        t.append(e0.elapsed_time(e1) * 1e3)
    return np.asarray(t)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--rounds', type=int, default=300)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('time_gauss_prior.py needs a CUDA device')
    name, power = device_info()
    print(f'device: {name}, power limit: {power}; {"-".join(map(str, DIMS))}, B={B}, S={S}')
    g = torch.Generator().manual_seed(2)
    x = torch.rand(B, DIMS[0], generator=g).cuda()
    y = torch.randint(0, DIMS[-1], (B,), generator=g).cuda()
    configs = [(lr, prior) for lr in (False, True) for prior in (False, True)]
    steps = {c: make_step(c[0], c[1], x, y)[0] for c in configs}
    flush = torch.empty(64 << 20, dtype=torch.float32, device='cuda')     # 256 MB > the 126 MB L2
    for c in configs:
        for _ in range(10):
            steps[c]()
    torch.cuda.synchronize()
    times = {c: [] for c in configs}
    for r in range(a.rounds):
        for c in (configs if r % 2 == 0 else configs[::-1]):
            times[c].append(time_it(steps[c], flush, 1)[0])
    label = {False: 'cfg2 (WS, TF32, network-level)', True: 'cfg3 (LR, fp32)'}
    for c in configs:
        t = np.asarray(times[c])
        print(f'{label[c[0]]:>32s} {"per-weight prior" if c[1] else "model_params prior":>18s}: median '
              f'{np.median(t):7.1f} us  (p10 {np.percentile(t, 10):7.1f}, p90 {np.percentile(t, 90):7.1f}, n={len(t)})')
    for lr in (False, True):
        d = np.median(times[(lr, True)]) - np.median(times[(lr, False)])
        print(f'{label[lr]}: per-weight - model_params prior: {d:+.1f} us per step (medians)')

    # the kernels alone, at the cfg2 parameter count
    net = make_net(False)
    net.posterior_to_prior()
    params = [l.params() for l in net.layers()]
    gauss = [bnn_b200.layers.gauss_prior(l) for l in net.layers()]
    n_par = sum(l[0].numel() + l[2].numel() for l in params)          # weights and biases, each a (mu, rho) pair
    grads = [[torch.zeros_like(p) for p in l] for l in params]
    bnn_b200.manual_seed(3)
    eps = F.plan_eps([((1,), (1,))] * len(params), S, 'cuda')
    tab, nt, _ = F._gauss_prior_table(params, gauss, eps, True, S, grads)
    rng = eps.rng(0)
    acc = torch.zeros(2 * S + 1, dtype=torch.float64, device='cuda')
    st = L.stream()
    lib = L.lib()
    kernels = {
        'bbb_gauss_prior_logprob': (lambda: lib.bbb_gauss_prior_logprob(tab, nt, S, C.byref(rng), acc[:S].data_ptr(),
                                                                         acc[S:2 * S].data_ptr(), st), 16),
        'bbb_gauss_prior_logprob_bwd': (lambda: lib.bbb_gauss_prior_logprob_bwd(tab, nt, S, C.byref(rng), -0.5, 0.5,
                                                                                None, None, 0, None, st), 32),
        'bbb_gauss_prior_kl': (lambda: lib.bbb_gauss_prior_kl(tab, nt, acc[2 * S:].data_ptr(), st), 16),
        'bbb_gauss_prior_kl_bwd': (lambda: lib.bbb_gauss_prior_kl_bwd(tab, nt, 1.0, None, None, st), 32),
    }
    for k, (fn, bpp) in kernels.items():
        for _ in range(20):
            L.check(fn(), k)
        t = time_it(lambda: L.check(fn(), k), flush, 500)
        med = np.median(t)
        bw = bpp * n_par / (med * 1e-6)
        print(f'{k:>28s}: median {med:6.1f} us (p10 {np.percentile(t, 10):6.1f}, p90 {np.percentile(t, 90):6.1f}); '
              f'{bpp * n_par / 1e6:5.1f} MB -> {bw / 1e12:5.2f} TB/s = {100 * bw / HBM_PEAK:4.1f} % of 7.7 TB/s '
              f'({n_par} weights and biases, S={S})')


if __name__ == '__main__':
    main()
