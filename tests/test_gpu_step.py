"""GPU tests of the step-level pieces: FusedAdam (SURVEY 8f-1) and the CUDA-graph train step."""
import numpy as np
import pytest
import torch

import bnn_b200
from tests import parity_cases as PC
from tests.golden_util import Case

pytestmark = pytest.mark.gpu
DEV = 'cuda'


def test_fused_adam_matches_torch_adam_on_gpu():
    torch.manual_seed(0)
    shapes = [(1200, 784), (1200,), (10, 1200), (10,), (3, 5), (7,)]     # includes unaligned tails
    ps = [torch.nn.Parameter(torch.randn(s, device=DEV)) for s in shapes]
    qs = [torch.nn.Parameter(p.detach().clone()) for p in ps]
    ref = torch.optim.Adam(ps, lr=1e-3)
    opt = bnn_b200.FusedAdam(qs, lr=1e-3)
    for it in range(5):
        for p, q in zip(ps, qs):
            g = torch.randn(p.shape, device=DEV)
            p.grad, q.grad = g.clone(), g.clone()
        ref.step()
        opt.step()
    for p, q in zip(ps, qs):
        assert torch.allclose(p, q, rtol=2e-6, atol=1e-7), float((p - q).abs().max())
        assert torch.allclose(ref.state[p]['exp_avg_sq'], opt.state[q]['exp_avg_sq'], rtol=1e-6, atol=1e-12)


@pytest.mark.parametrize('name,tf32', [('cfg4_bandit', False), ('small_cls_mix', False), ('cfg2_mnist_mix', True),
                                       ('small_lr_cls', False)])
def test_graphed_step_equals_eager_steps(name, tf32):
    """3 replays of the captured step == 3 eager steps with the same Philox coordinates and FusedAdam;
    capture/warm-up must leave the model untouched."""
    c = Case(name)
    x = c.x.to(DEV)
    y = c.y.to(DEV) if c.mode == 'classification' else torch.randn(c.B, c.dims[-1], device=DEV)
    seed, step0, warm = 321, 100, 2

    net_g = PC.build_net(c, DEV, tf32=tf32).train()
    opt_g = bnn_b200.FusedAdam(net_g.parameters(), lr=1e-3)
    bnn_b200.manual_seed(seed, step0)
    before = [p.detach().clone() for p in net_g.parameters()]
    gs = bnn_b200.GraphedTrainStep(net_g, opt_g, x, y, c.S, sigma=c.sigma, beta=c.beta, warmup=warm)
    for p, b in zip(net_g.parameters(), before):
        assert torch.equal(p, b)
    losses_g = []
    for k in range(3):
        info = gs(x, y, beta=c.beta)
        losses_g.append(float(info[0]))

    def eager_run():
        net_e = PC.build_net(c, DEV, tf32=tf32).train()
        opt_e = bnn_b200.FusedAdam(net_e.parameters(), lr=1e-3)
        bnn_b200.manual_seed(seed, step0 + warm)      # the capture consumed `warm` + 1 host steps; it baked step0 + warm
        losses = []
        elbo = net_e.sample_elbo_lr if c.lr else net_e.sample_elbo
        for k in range(3):
            net_e.zero_grad()
            info = elbo(x, y, c.beta, c.S, sigma=c.sigma)
            info[0].backward()
            opt_e.step()
            losses.append(float(info[0].detach()))
        return net_e, losses

    net_e, losses_e = eager_run()
    # (TF32: the third loss already sees two Adam steps whose sign-flipped weights differ between any two runs)
    np.testing.assert_allclose(losses_g, losses_e, rtol=1e-5 if not tf32 else 5e-4)
    if not tf32:
        for p, q in zip(net_g.parameters(), net_e.parameters()):
            assert torch.allclose(p, q, rtol=1e-4, atol=2e-6), float((p - q).abs().max())
    else:
        # The tensor-core kernels combine split-K partial tiles with fp32 red.add, whose order varies from run
        # to run (~1e-7), and the next TF32 rounding of those activations turns a fraction of that into ~1e-5
        # relative differences (measured eager-vs-eager with identical seeds, tools/debug_graph.py).  Adam's
        # first steps move a weight by +-lr whatever its gradient's size, so weights with a tiny gradient can
        # step the other way.  Two runs of this path agree statistically, not bit for bit -- so the bound on
        # graph-vs-eager is set by the eager-vs-eager disagreement measured here, in the same process.
        net_e2, _ = eager_run()

        def mismatch(pa, pb):
            return float((~torch.isclose(pa, pb, rtol=1e-4, atol=2e-6)).float().mean())
        for p, q, q2 in zip(net_g.parameters(), net_e.parameters(), net_e2.parameters()):
            floor = mismatch(q, q2)
            got = mismatch(p, q)
            # the floor itself moves from run to run (one failure in ~10 full-suite runs at 3 * floor + 0.01): the count
            # bound is loose, the size bound below is exact (3 steps of at most 2 lr)
            assert got <= max(0.05, 5 * floor + 0.02), (got, floor)
            assert float((p - q).abs().max()) <= 3 * 2 * 1e-3 * 1.05
    assert losses_g[0] != losses_g[1]                   # fresh eps every replay


def test_graphed_step_follows_a_step_lr_scheduler():
    """reg_task.py:53-54 / class_task.py:60-61 drive the optimiser with torch's StepLR.  The captured Adam launch has the
    initial lr baked in; GraphedTrainStep scales it by a device scalar it refreshes when the host lr has moved.  Four
    steps with the lr halved after every step: graph == eager (exact fp32 kernels)."""
    c = Case('small_cls_mix')
    x, y = c.x.to(DEV), c.y.to(DEV)
    out = []
    for graphed in (False, True):
        net = PC.build_net(c, DEV, tf32=False).train()
        opt = bnn_b200.FusedAdam(net.parameters(), lr=1e-2)
        sched = torch.optim.lr_scheduler.StepLR(opt, step_size=1, gamma=0.5)
        if graphed:
            bnn_b200.manual_seed(9, 50)
            gs = bnn_b200.GraphedTrainStep(net, opt, x, y, c.S, sigma=c.sigma, beta=c.beta, warmup=2)
        else:
            bnn_b200.manual_seed(9, 52)       # the capture consumed warmup + 1 host steps and baked step 52
        for k in range(4):
            if graphed:
                gs(x, y)
            else:
                net.zero_grad()
                net.sample_elbo(x, y, c.beta, c.S, sigma=c.sigma)[0].backward()
                opt.step()
            sched.step()
        out.append([p.detach().clone() for p in net.parameters()])
    assert opt.param_groups[0]['lr'] == pytest.approx(1e-2 / 16)
    for p, q in zip(*out):
        assert torch.allclose(p, q, rtol=1e-4, atol=2e-6), float((p - q).abs().max())


@pytest.mark.parametrize('tf32', [False, True])
def test_row_sharded_step_equals_full_batch(tf32):
    """The minibatch-row axis (parallel.ShardPlan / sharded_elbo) on the real kernels: two row shards computed one after
    the other with the same Philox stream, gradients averaged = the full-batch step's gradients."""
    from bnn_b200 import parallel
    c = Case('cfg2_mnist_mix')
    x, y = c.x.to(DEV), c.y.to(DEV)
    net = PC.build_net(c, DEV, tf32=tf32).train()
    bnn_b200.manual_seed(11, 3)
    net.zero_grad()
    full = net.sample_elbo(x, y, c.beta, c.S)
    full[0].backward()
    want = [p.grad.clone() for p in net.parameters()]
    acc, loss = [torch.zeros_like(p) for p in net.parameters()], 0.0
    for r in range(2):
        plan = parallel.ShardPlan(r, 2, c.S, x.shape[0], row_shards=2)
        bnn_b200.manual_seed(11, 3)
        net.zero_grad()
        info = parallel.sharded_elbo(net, *plan.rows(x, y), c.beta, plan)
        info[0].backward()
        loss += float(info[0].detach()) / 2
        for a, p in zip(acc, net.parameters()):
            a += p.grad / 2
    rtol = 5e-3 if tf32 else 2e-5
    assert abs(loss - float(full[0].detach())) <= rtol * abs(float(full[0].detach()))
    for a, b in zip(acc, want):
        assert float((a - b).abs().max()) <= rtol * float(b.abs().max())


def test_peer_adam_kernel_two_ranks_on_one_device():
    """bbb_adam_step_peer with two 'ranks' whose buffers live on this one GPU, launched on two streams: the flag
    barriers in (peer) memory let them meet, each reduces its slice of BOTH gradient buckets, updates with its own
    m / v and writes the new parameters into both parameter buffers.  Result == Adam on the mean gradient."""
    import ctypes as C
    L = bnn_b200._lib
    lib = L.lib()
    torch.manual_seed(0)
    n, W = 100003, 2                                   # n % 4 != 0: the tail belongs to the last rank
    npad = (n + 3) // 4 * 4
    p0 = torch.randn(npad, device=DEV)
    ps = [p0.clone(), p0.clone()]
    gs = [torch.randn(npad, device=DEV), torch.randn(npad, device=DEV)]
    ms = [torch.zeros(npad, device=DEV) for _ in range(W)]
    vs = [torch.zeros(npad, device=DEV) for _ in range(W)]
    flags = [torch.zeros(16, dtype=torch.int32, device=DEV) for _ in range(W)]
    words = [torch.zeros(2, dtype=torch.int32, device=DEV) for _ in range(W)]
    ref_p = torch.nn.Parameter(p0[:n].clone())
    ref = torch.optim.Adam([ref_p], lr=1e-2)
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    torch.cuda.synchronize()
    for step in (1, 2, 3):
        for g in gs:
            g.normal_()
        torch.cuda.synchronize()
        for r in range(W):
            comm = L.PeerComm()
            comm.world, comm.rank = W, r
            for k in range(W):
                comm.grads[k], comm.params[k], comm.flags[k] = gs[k].data_ptr(), ps[k].data_ptr(), flags[k].data_ptr()
            comm.epoch, comm.done_blocks = words[r][0:1].data_ptr(), words[r][1:2].data_ptr()
            with torch.cuda.stream(streams[r]):
                L.check(lib.bbb_adam_step_peer(C.byref(comm), ms[r].data_ptr(), vs[r].data_ptr(), n, 1e-2, 0.9, 0.999,
                                               1e-8, step, None, None, streams[r].cuda_stream), 'bbb_adam_step_peer')
        torch.cuda.synchronize()
        ref_p.grad = (0.5 * (gs[0] + gs[1]))[:n].clone()
        ref.step()
        assert int(words[0][0]) == step and int(words[1][0]) == step and int(words[0][1]) == 0
    assert torch.equal(ps[0][:n], ps[1][:n])                                  # both ranks hold the same parameters
    assert torch.allclose(ps[0][:n], ref_p.detach(), rtol=2e-6, atol=1e-7), float((ps[0][:n] - ref_p).abs().max())
    half = (n // 4) // 2 * 4
    assert float(ms[0][half:].abs().max()) == 0.0 and float(ms[1][:half].abs().max()) == 0.0   # state is sharded


def test_peer_sharded_adam_single_gpu_equals_fused_adam():
    """One rank: PeerShardedAdam (flat re-homed parameters, bucket gradients) == FusedAdam on the same Philox steps."""
    from bnn_b200 import functional as F
    c = Case('cfg4_bandit')
    x, y = c.x.to(DEV), torch.randn(c.B, 1, device=DEV)
    res = []
    try:
        for peer in (False, True):
            F.grad_buckets.clear()
            net = PC.build_net(c, DEV).train()
            opt = (bnn_b200.PeerShardedAdam if peer else bnn_b200.FusedAdam)(net.parameters(), lr=1e-3)
            bnn_b200.manual_seed(3, 0)
            for _ in range(3):
                net.zero_grad()
                net.sample_elbo(x, y, c.beta, c.S)[0].backward()
                opt.step()
            res.append([p.detach().clone() for p in net.parameters()])
    finally:
        F.grad_buckets.clear()
    for a, b in zip(*res):
        assert torch.allclose(a, b, rtol=1e-5, atol=1e-7), float((a - b).abs().max())
