#!/usr/bin/env python
"""Time posterior-predictive evaluation of a test set: the MNIST-shape net (784-1200-1200-10, mixture prior), N = 10 000
rows, S = 10 samples, in exact fp32 and TF32 mode, weight sampling and local reparameterisation.

  (a) what a user writes without BayesianNetwork.predictive: S calls of net(x, sample=True), the softmax mean on the
      device (bbb_softmax_mean), then the sampled logits and the mean copied to the host and the entropy, mutual
      information and ECE computed with numpy;
  (b) net.predictive(x, S, target=y).metrics();
  (c) bbb_predictive_stats alone on the [S, N, C] outputs (CUDA events, mean over many launches; the 4 MB input stays
      in L2 between launches).
(a) and (b) are host-clock times of calls that end with host values (median of --reps).  The device name and its
power limit are printed with the times.  --profile DIR instead runs (b) once per mode under torch.profiler and writes
the kernel table to DIR/predictive_kernels.txt (a separate run: tracing slows the host).
usage: python tools/time_predictive.py [--reps 5] [--profile DIR]"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bnn_b200  # noqa: E402
from bnn_b200 import functional as F  # noqa: E402

N, S, DIMS, N_BINS = 10000, 10, (784, 1200, 1200, 10), 15


def device_info():
    name = torch.cuda.get_device_name()
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader',
                            f'--id={torch.cuda.current_device()}'], capture_output=True, text=True, timeout=30)
        power = q.stdout.strip() or 'unknown'
    except (OSError, subprocess.SubprocessError):
        power = 'unknown'
    return name, power


def make_net(tf32, lr):
    mp = dict(input_shape=DIMS[0], classes=DIMS[-1], batch_size=128, hidden_units=list(DIMS[1:-1]),
              mode='classification', mu_init=[-0.2, 0.2], rho_init=[-5, -4],
              prior_init=[1.0] if lr else [0.5, 0, -8], mixture_prior=not lr, local_reparam=lr, tf32=tf32)
    torch.manual_seed(0)
    return bnn_b200.BayesianNetwork(mp).cuda().eval()


def host_metrics(logits, pbar, y, n_bins=N_BINS):
    """(a)'s host side: entropy, expected entropy, mutual information and ECE in numpy."""
    z = logits.astype(np.float64)
    p = np.exp(z - z.max(-1, keepdims=True))
    p /= p.sum(-1, keepdims=True)
    pb = pbar.astype(np.float64)
    with np.errstate(divide='ignore', invalid='ignore'):
        ent = -np.nansum(pb * np.log(pb), -1)
        exp_ent = -np.nansum(p * np.log(p), -1).mean(0)
    mi = np.maximum(ent - exp_ent, 0.0)
    conf, pred = pb.max(-1), pb.argmax(-1)
    cor = (pred == y).astype(np.float64)
    m = np.clip(np.ceil(conf * n_bins) - 1, 0, n_bins - 1).astype(np.int64)
    ece = np.abs(np.bincount(m, cor, n_bins) - np.bincount(m, conf, n_bins)).sum() / len(y)
    return dict(accuracy=cor.mean(), ece=ece, mi=mi.mean())


def leg_a(net, x, y_host):
    with torch.no_grad():
        logits = torch.stack([net(x, sample=True) for _ in range(S)])
        pbar = F.softmax_mean(logits)
    return host_metrics(logits.cpu().numpy(), pbar.cpu().numpy(), y_host)


def leg_b(net, x, y):
    return net.predictive(x, S, target=y).metrics()


def host_time(fn, reps):
    fn()                                         # warm-up: module loads, allocator, every shape of the timed calls
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()                                     # ends with host values: the device work is complete
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts)) * 1e3


def kernel_time(outs, y, launches=200):
    mean, rs, pred, acc = F.predictive_stats(outs, y, n_bins=N_BINS)

    def launch():
        F._predictive_launch(outs, y, 'classification', 1.0, N_BINS, mean, rs, pred, acc)
    for _ in range(5):
        launch()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(launches):
        launch()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / launches


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--profile', default=None, help='directory for the torch.profiler kernel table of (b)')
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('time_predictive.py needs a CUDA device')
    name, power = device_info()
    print(f'device: {name}, power limit: {power}; N={N} S={S} net {"-".join(map(str, DIMS))}')
    g = torch.Generator().manual_seed(1)
    x = torch.rand(N, DIMS[0], generator=g).cuda()
    y_cpu = torch.randint(0, DIMS[-1], (N,), generator=g)
    y, y_host = y_cpu.cuda(), y_cpu.numpy()
    bnn_b200.manual_seed(7)
    modes = [(tf32, lr) for lr in (False, True) for tf32 in (False, True)]
    if a.profile:
        from torch.profiler import ProfilerActivity, profile
        os.makedirs(a.profile, exist_ok=True)
        with open(os.path.join(a.profile, 'predictive_kernels.txt'), 'w') as f:
            f.write(f'device: {name}, power limit: {power}\n')
            for tf32, lr in modes:
                net = make_net(tf32, lr)
                leg_b(net, x, y)
                torch.cuda.synchronize()
                with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
                    leg_b(net, x, y)
                    torch.cuda.synchronize()
                table = prof.key_averages().table(sort_by='cuda_time_total', row_limit=20)
                head = f'== (b) {"tf32" if tf32 else "fp32"} {"lr" if lr else "ws"}'
                f.write(f'{head}\n{table}\n')
                print(head)
                print(table)
        return
    for tf32, lr in modes:
        net = make_net(tf32, lr)
        ta = host_time(lambda: leg_a(net, x, y_host), a.reps)
        tb = host_time(lambda: leg_b(net, x, y), a.reps)
        with torch.no_grad():
            outs = net.sample_predict(x, S)
        tc = kernel_time(outs, y)
        ma, mb = leg_a(net, x, y_host), leg_b(net, x, y)
        print(f'{"tf32" if tf32 else "fp32"} {"lr" if lr else "ws"}: (a) loop + host numpy {ta:.2f} ms | '
              f'(b) predictive + metrics {tb:.2f} ms | (c) bbb_predictive_stats {tc:.1f} us | '
              f'accuracy (a) {ma["accuracy"]:.4f} (b) {mb["accuracy"]:.4f}, ece (a) {ma["ece"]:.4f} (b) {mb["ece"]:.4f}')


if __name__ == '__main__':
    main()
