#!/usr/bin/env python
"""Time the captured train step (GraphedTrainStep: sample_elbo + backward + FusedAdam in one CUDA graph) of the
heteroscedastic regression net against the homoscedastic one, at the BASELINE config-1 shape: 1-400-400-2
(likelihood='heteroscedastic', D = 1) against 1-400-400-1 (the fixed-sigma Gaussian), B = 128, S = 5, mixture prior,
in exact fp32 and in TF32 mode.

The four configurations alternate inside every round so that drift of the shared machine hits all of them alike.  Each
timed sample is ONE graph replay between CUDA events, after a write of 256 MB that evicts the 126 MB L2 (outside the
events), so the step starts from HBM as it does in a training loop that touches data between steps.  Reported: median
and 10th / 90th percentile in microseconds.  The device name and its power limit are printed with the times.
--profile DIR instead runs one replay of each step under torch.profiler and writes the kernel table to
DIR/heteroscedastic_kernels.txt (a separate run: tracing slows the host), checking that the heteroscedastic step runs
nll_gauss_het_kernel and elbo_finalize_kernel and the Gaussian step, whose fused head does both, neither.
usage: python tools/time_heteroscedastic.py [--rounds 400] [--profile DIR]"""
import argparse
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bnn_b200  # noqa: E402

B, S, HIDDEN = 128, 5, 400


def device_info():
    name = torch.cuda.get_device_name()
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader',
                            f'--id={torch.cuda.current_device()}'], capture_output=True, text=True, timeout=30)
        power = q.stdout.strip() or 'unknown'
    except (OSError, subprocess.SubprocessError):
        power = 'unknown'
    return name, power


def make_step(likelihood, tf32, x, y):
    mp = dict(input_shape=1, classes=1, batch_size=B, hidden_units=HIDDEN, mode='regression', mu_init=[-0.2, 0.2],
              rho_init=[-5, -4], prior_init=[0.5, 0, -6], mixture_prior=True, tf32=tf32, likelihood=likelihood)
    torch.manual_seed(0)
    net = bnn_b200.BayesianNetwork(mp).cuda().train()
    opt = bnn_b200.FusedAdam(net.parameters(), lr=1e-3)
    sigma = 1.0 if likelihood == 'heteroscedastic' else 0.1
    bnn_b200.manual_seed(1)
    return bnn_b200.GraphedTrainStep(net, opt, x, y, S, sigma=sigma, beta=0.01, warmup=3)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--rounds', type=int, default=400)
    ap.add_argument('--profile', default=None, help='directory for the torch.profiler kernel table')
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('time_heteroscedastic.py needs a CUDA device')
    name, power = device_info()
    g = torch.Generator().manual_seed(2)
    x = (2 * torch.rand(B, 1, generator=g) - 1).cuda()
    y = torch.sin(3 * x) + 0.1 * torch.randn(B, 1, generator=g).cuda()
    configs = [(lik, tf32) for tf32 in (False, True) for lik in ('heteroscedastic', 'gaussian')]
    steps = {c: make_step(c[0], c[1], x, y) for c in configs}
    head = (f'device: {name}, power limit: {power}; captured train step (GraphedTrainStep + FusedAdam), 1-{HIDDEN}-'
            f'{HIDDEN}-(2 heteroscedastic | 1 gaussian), B={B}, S={S}')
    print(head)
    if a.profile:
        from torch.profiler import ProfilerActivity, profile
        os.makedirs(a.profile, exist_ok=True)
        with open(os.path.join(a.profile, 'heteroscedastic_kernels.txt'), 'w') as f:
            f.write(head + '\n')
            for c in configs:
                step = steps[c]
                step()
                torch.cuda.synchronize()
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    step()
                    torch.cuda.synchronize()
                kernels = [e.key for e in prof.key_averages() if e.device_type == torch.autograd.DeviceType.CUDA]
                tag = f'== {c[0]} {"tf32" if c[1] else "fp32"}'
                table = prof.key_averages().table(sort_by='cuda_time_total', row_limit=30)
                f.write(f'{tag}\n{table}\n')
                print(tag)
                print(table)
                # the heteroscedastic step runs the likelihood and the assembly as kernels of their own; the Gaussian
                # step does both inside its fused head (head_fwd_kernel also serves the plain forward of a narrow layer)
                het = c[0] == 'heteroscedastic'
                for kname in ('nll_gauss_het_kernel', 'elbo_finalize_kernel'):
                    assert any(kname in k for k in kernels) == het, (kname, kernels)
        return
    flush = torch.empty(64 << 20, dtype=torch.float32, device='cuda')     # 256 MB > the 126 MB L2
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in configs]
    times = {c: [] for c in configs}
    for c in configs:                                                     # warm-up replays
        for _ in range(10):
            steps[c]()
    torch.cuda.synchronize()
    for r in range(a.rounds):
        order = configs if r % 2 == 0 else configs[::-1]
        for c in order:
            flush.zero_()
            e0, e1 = ev[configs.index(c)]
            e0.record()
            steps[c]()
            e1.record()
            e1.synchronize()
            times[c].append(e0.elapsed_time(e1) * 1e3)
    for c in configs:
        t = np.asarray(times[c])
        print(f'{c[0]:>15s} {"tf32" if c[1] else "fp32"}: median {np.median(t):7.1f} us  '
              f'(p10 {np.percentile(t, 10):7.1f}, p90 {np.percentile(t, 90):7.1f}, n={len(t)})')
    for tf32 in (False, True):
        d = np.median(times[('heteroscedastic', tf32)]) - np.median(times[('gaussian', tf32)])
        print(f'heteroscedastic - gaussian, {"tf32" if tf32 else "fp32"}: {d:+.1f} us per step (medians)')


if __name__ == '__main__':
    main()
