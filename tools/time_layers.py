#!/usr/bin/env python
"""Warm and cold (L2-flushed) CUDA-event timings of the layer kernels through the C ABI, one layer at a time, with the
flags the per-layer host path (functional._forward / _backward with weight sampling) passes in TF32 mode.
usage: python tools/time_layers.py [B S [d0 d1 ... dn]]
The widths d0 .. dn name a network (default: the MNIST shape 784 1200 1200 10); its first layer reads the shared network
input and hands no dx down, the others read the stored pre-activation of the layer below.  BBB_LIB selects the library."""
import ctypes as C
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bnn_b200  # noqa: E402
from bnn_b200 import _lib as L, functional as F  # noqa: E402

B = int(sys.argv[1]) if len(sys.argv) > 1 else 128
S = int(sys.argv[2]) if len(sys.argv) > 2 else 2
dims = [int(d) for d in sys.argv[3:]] or [784, 1200, 1200, 10]
dev = 'cuda'
prior = F.make_prior([0.5, 0, -8], True)
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)


def timeit(fn, n=30, cold=False):
    for _ in range(3):
        fn()
    ts = []
    for _ in range(n):
        if cold:
            flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e3)
    ts.sort()
    return ts[len(ts) // 2]


for l, (inn, out) in enumerate(zip(dims[:-1], dims[1:])):
    first = l == 0
    torch.manual_seed(0)
    wm = torch.empty(out, inn, device=dev).uniform_(-0.2, 0.2); wr = torch.empty(out, inn, device=dev).uniform_(-5, -4)
    bm = torch.empty(out, device=dev).uniform_(-0.2, 0.2); br = torch.empty(out, device=dev).uniform_(-5, -4)
    x = torch.randn(1 if first else S, B, inn, device=dev)
    y = torch.zeros(S, B, out, device=dev); dy = torch.randn(S, B, out, device=dev)
    dx = torch.zeros(S, B, inn, device=dev)
    g = [torch.empty_like(t) for t in (wm, wr, bm, br)]
    acc = torch.zeros(2 * S, dtype=torch.float64, device=dev)
    rng = L.Rng(1, 0, 0, 0, None)
    st = torch.cuda.current_stream().cuda_stream
    base = L.F_SAMPLE | L.F_TF32 | L.F_OUT_ZEROED | (0 if first else L.F_RELU_IN)
    xs = 0 if first else B * inn

    def fwd():
        L.check(L.lib().bbb_linear_fwd(x.data_ptr(), xs, wm.data_ptr(), wr.data_ptr(), bm.data_ptr(), br.data_ptr(), None,
                                       None, C.byref(rng), C.byref(prior), S, B, inn, out, base | L.F_LOGPROB, y.data_ptr(),
                                       acc[:S].data_ptr(), acc[S:].data_ptr(), st), 'fwd')

    def bwd(extra=0):
        fl = base | extra | (L.F_NO_DX if first else L.F_DX_PREACT)
        L.check(L.lib().bbb_linear_bwd(dy.data_ptr(), None, x.data_ptr(), xs, wm.data_ptr(), wr.data_ptr(), bm.data_ptr(),
                                       br.data_ptr(), None, None, C.byref(rng), C.byref(prior), S, B, inn, out, fl, -0.25,
                                       0.25, None, None, 0, None, None if first else dx.data_ptr(), g[0].data_ptr(),
                                       g[1].data_ptr(), g[2].data_ptr(), g[3].data_ptr(), st), 'bwd')

    print(f'[{inn}x{out}] B={B} S={S}  fwd warm {timeit(fwd):6.1f} us  cold {timeit(fwd, cold=True):6.1f} us   '
          f'bwd warm {timeit(bwd):6.1f} us  cold {timeit(bwd, cold=True):6.1f} us', flush=True)

cnt = torch.zeros(1, dtype=torch.int32, device=dev)
st = torch.cuda.current_stream().cuda_stream
print('tiny kernel (launch floor, events around one launch):', timeit(lambda: L.lib().bbb_counter_add(cnt.data_ptr(), 0, st)), 'us')
