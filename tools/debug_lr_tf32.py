#!/usr/bin/env python
"""Where does the TF32 path of the local-reparameterisation estimator lose accuracy?  Runs the forward and the backward of
the MNIST-shape LR net on the exact fp32 kernels and on the tcgen05 kernels with the SAME Philox eps, and prints the
max-norm relative difference of every intermediate (y, delta per layer; dx and the four gradients per layer).
usage: python tools/debug_lr_tf32.py"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bnn_b200  # noqa: E402,F401
from bnn_b200 import functional as F, rng as R  # noqa: E402

dev = 'cuda'
torch.manual_seed(0)
dims, B, S = (784, 1200, 1200, 10), 128, 2
params = []
for i, o in zip(dims[:-1], dims[1:]):
    params.append((torch.empty(i, o, device=dev).uniform_(-0.2, 0.2), torch.empty(i, o, device=dev).uniform_(-5, -4),
                   torch.empty(o, device=dev).uniform_(-0.2, 0.2), torch.empty(o, device=dev).uniform_(-5, -4)))
x = torch.rand(B, dims[0], device=dev)
d_out = torch.randn(S, B, dims[-1], device=dev) / B


def rel(a, b):
    return float((a.double() - b.double()).abs().max() / b.double().abs().max())


def run(est, params, tf32, beta):
    """forward + backward of one estimator with the same Philox eps -> (ys, deltas, grads, log-prob accumulators)"""
    R.manual_seed(7, 0)
    eps = F.plan_eps(est.eps_shapes(params, B), S, x.device, True)
    acc = torch.zeros(est.acc_len(S), dtype=torch.float64, device=dev)
    ys, deltas = F._forward(est, x, params, S, eps, True, True, tf32, est.lp(acc, S))
    ys, deltas = [t.clone() for t in ys], [None if t is None else t.clone() for t in deltas]
    _, grads = backward(est, params, eps, ys, deltas, tf32, beta)
    return ys, deltas, grads, acc


def backward(est, params, eps, ys, deltas, tf32, beta):
    _, grads = F._backward(est, x, [t.clone() for t in ys], [None if t is None else t.clone() for t in deltas],
                           d_out.clone(), params, S, eps, True, tf32, est.elbo_grad_args(beta, None, S), None, False)
    return None, [[g.clone() for g in lg] for lg in grads]


lr = F._LocalReparam(1.0)
res = {}
for tf32 in (False, True):
    ys, deltas, grads, kl = run(lr, params, tf32, 0.1)
    res[tf32] = (ys, deltas, grads, float(kl))
(y0, d0, g0, k0), (y1, d1, g1, k1) = res[False], res[True]
print('kl', k0, k1)
for l in range(len(params)):
    print(f'layer {l}: y {rel(y1[l], y0[l]):.2e}  delta {rel(d1[l], d0[l]):.2e}  '
          + '  '.join(f'{n} {rel(a, b):.2e}' for n, a, b in zip(('g_w_mu', 'g_w_rho', 'g_b_mu', 'g_b_rho'), g1[l], g0[l])))

# ---- backward kernels alone: both modes on the SAME stored forward (the TF32 one), so the ReLU masks are identical ----
R.manual_seed(7, 0)
eps = F.plan_eps(lr.eps_shapes(params, B), S, x.device, True)
gb = {tf32: backward(lr, params, eps, y1, d1, tf32, 0.1)[1] for tf32 in (False, True)}
print('backward kernels on identical forward state:')
for l in range(len(params)):
    print(f'layer {l}: ' + '  '.join(f'{n} {rel(a, b):.2e}' for n, a, b in zip(('g_w_mu', 'g_w_rho', 'g_b_mu', 'g_b_rho'), gb[True][l], gb[False][l])))
flips = [float(((a > 0) != (b > 0)).float().mean()) for a, b in zip(y1[:-1], y0[:-1])]
print('fraction of hidden units whose ReLU mask differs between the two forwards:', flips)

# ---- the same experiment on the weight-sampling estimator (same shapes, [out, in] weights) --------------------------
ws = F._WeightSampling(F.make_prior([0.5, 0, -8], True))
wparams = [tuple(t.t().contiguous() if t.dim() == 2 else t for t in p) for p in params]
wres = {}
for tf32 in (False, True):
    ys, _, grads, _ = run(ws, wparams, tf32, 0.0)
    wres[tf32] = (ys, grads)
print('weight-sampling estimator, fp32 kernels vs tcgen05 kernels:')
for l in range(len(wparams)):
    print(f'layer {l}: y {rel(wres[True][0][l], wres[False][0][l]):.2e}  '
          + '  '.join(f'{n} {rel(a, b):.2e}' for n, a, b in zip(('g_w_mu', 'g_w_rho', 'g_b_mu', 'g_b_rho'), wres[True][1][l], wres[False][1][l])))
print('mask flips:', [float(((a > 0) != (b > 0)).float().mean()) for a, b in zip(wres[True][0][:-1], wres[False][0][:-1])])
