"""CPU tests of the Python host (nn.Module mirror + autograd glue) against the golden fixtures, with
the C ABI replaced by the test double in tests/fake_bbb.py.  No GPU, no product CPU path: the double
is test infrastructure.  The same checks run against the real library in tests/test_gpu_parity.py."""
import ctypes
import os
import re

import pytest
import torch

import bnn_b200
from tests import fake_bbb, parity_cases as PC
from tests.golden_util import Case, SMALL, SMALL_LR, DEEP_SMALL

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture
def fake(monkeypatch):
    return fake_bbb.install(monkeypatch)


@pytest.mark.parametrize('name', SMALL + SMALL_LR + DEEP_SMALL + ['cfg4_bandit'])
@pytest.mark.parametrize('fused', [True, False])
def test_train_step_network_level(fake, name, fused):
    PC.check_train_step(Case(name), 'cpu', fused=fused)
    fused_used = ('nll_ce' in fake.calls) or ('nll_gauss' in fake.calls) or ('head_fwd' in fake.calls)
    case = Case(name)
    expect_fused = fused and not case.meta.get('flat_target', False)
    assert fused_used == expect_fused        # [B] vs [B,1] broadcast targets (SURVEY B-3) take the general path


@pytest.mark.parametrize('name', ['small_cls_mix', 'small_cls_gauss', 'deep5_small_mix'])
def test_tf32_train_step_takes_the_network_level_call_when_supported(fake, name):
    """tf32=True routes sample_elbo through ONE bbb_mlp_fwd call when bbb_mlp_supported says so (hidden widths that are
    multiples of 4, a head on top), otherwise through the per-layer calls; same results either way."""
    case = Case(name)
    PC.check_train_step(case, 'cpu', fused=True, tf32=True)
    expect = all(d % 4 == 0 for d in case.dims[:-1])
    assert ('mlp_fwd' in fake.calls) == expect
    assert ('linear_fwd' in fake.calls) == (not expect)


@pytest.mark.parametrize('name', SMALL + SMALL_LR)
def test_train_step_layer_level(fake, name):
    PC.check_layerwise_train_step(Case(name), 'cpu')


@pytest.mark.parametrize('name', SMALL + SMALL_LR)
def test_eval_modes(fake, name):
    PC.check_eval_modes(Case(name), 'cpu')


@pytest.mark.parametrize('name', ['small_cls_mix', 'small_lr_cls', 'deep5_small_mix'])
def test_state_dict_layout(fake, name):
    PC.check_state_dict(Case(name), 'cpu')


def test_wrong_estimator_asserts(fake):
    c, clr = Case('small_cls_mix'), Case('small_lr_cls')
    with pytest.raises(AssertionError):
        PC.build_net(c, 'cpu').sample_elbo_lr(c.x, c.y, 0.5, 1)
    with pytest.raises(AssertionError):
        PC.build_net(clr, 'cpu').sample_elbo(clr.x, clr.y, 0.5, 1)


def test_local_reparam_defaults_to_false(fake):
    """bandits.py:24-34 omits 'local_reparam'; the reference raises KeyError (SURVEY App. B-1)."""
    mp = Case('small_bandit_bcast').model_params()
    del mp['local_reparam']
    net = bnn_b200.BayesianNetwork(mp)
    assert net.local_reparam is False and isinstance(net.l1, bnn_b200.BayesianLinear)


def test_deeper_network_extension(fake):
    mp = Case('small_cls_mix').model_params()
    mp['hidden_units'] = [12, 8, 8, 6]
    net = bnn_b200.BayesianNetwork(mp)
    assert net.n_layers == 5 and hasattr(net, 'l5') and hasattr(net, 'l4_act') and not hasattr(net, 'l5_act')


def test_no_cpu_fallback():
    """Without the double, CPU tensors are refused loudly (the CUDA path is the only path)."""
    c = Case('small_cls_mix')
    net = PC.build_net(c, 'cpu')
    with pytest.raises(RuntimeError, match='CUDA'):
        net(c.x, sample=True)


def test_library_matches_the_header():
    """libbbb.so loads and exports every function include/bbb.h declares (no compute calls)."""
    hdr = open(os.path.join(ROOT, 'include', 'bbb.h')).read()
    declared = set(re.findall(r'\b(bbb_[a-z0-9_]+)\s*\(', hdr))
    assert declared == set(bnn_b200._lib.EXPORTS), declared ^ set(bnn_b200._lib.EXPORTS)
    lib = ctypes.CDLL(bnn_b200._lib.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), name
    assert bnn_b200._lib.lib().bbb_version() == 101


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, 'bayesian-neural-network_b200')
    for fn in os.listdir(pkg) + ['../networks.py', '../config.py', '../bnn_b200.py']:
        p = os.path.join(pkg, fn)
        if p.endswith('.py'):
            src = open(p).read()
            assert 'import oracle' not in src and 'from oracle' not in src, fn


def test_fused_adam_matches_torch_adam(fake):
    """FusedAdam (host logic + ABI semantics through the double) == torch.optim.Adam over several steps."""
    torch.manual_seed(0)
    shapes = [(7, 5), (5,), (3, 4), (10,)]
    ps = [torch.nn.Parameter(torch.randn(s)) for s in shapes]
    qs = [torch.nn.Parameter(p.detach().clone()) for p in ps]
    ref = torch.optim.Adam(ps, lr=3e-3)
    opt = bnn_b200.FusedAdam(qs, lr=3e-3)
    for it in range(4):
        for p, q in zip(ps, qs):
            g = torch.randn(p.shape)
            p.grad, q.grad = g.clone(), g.clone()
        ref.step()
        opt.step()
    for p, q in zip(ps, qs):
        assert torch.allclose(p, q, rtol=1e-5, atol=1e-7)


def test_peer_sharded_adam_single_rank_is_adam(fake):
    """PeerShardedAdam with one rank: parameters re-homed into one flat buffer (same values, views), gradients land in
    the flat bucket the network-level backward writes, the update equals torch.optim.Adam, state names are torch's."""
    from bnn_b200 import functional as F
    c = Case('small_cls_mix')
    ref_net = PC.build_net(c, 'cpu').train()
    net = PC.build_net(c, 'cpu').train()
    ref = torch.optim.Adam(ref_net.parameters(), lr=3e-3)
    try:
        opt = bnn_b200.PeerShardedAdam(net.parameters(), lr=3e-3)
        assert opt.world == 1 and opt.reduces_gradients
        for p, q in zip(ref_net.parameters(), net.parameters()):
            assert torch.equal(p, q) and q.data_ptr() >= opt.flat_p.data_ptr()
        with bnn_b200.eps_mode('reference'):
            for it in range(3):
                for n_, o_ in ((ref_net, ref), (net, opt)):
                    torch.manual_seed(5 + it)
                    n_.zero_grad()
                    n_.sample_elbo(c.x, c.y, c.beta, c.S)[0].backward()
                    o_.step()
                assert net.l1.weight_mu.grad.data_ptr() == opt.flat_g.data_ptr()      # the bucket, not a copy
        for p, q in zip(ref_net.parameters(), net.parameters()):
            assert torch.allclose(p, q, rtol=1e-5, atol=1e-7), float((p - q).abs().max())
            assert torch.allclose(ref.state[p]['exp_avg_sq'], opt.state[q]['exp_avg_sq'], rtol=1e-5, atol=1e-12)
    finally:
        F.grad_buckets.clear()


def test_gradient_bucket_is_not_used_while_a_grad_is_alive(fake):
    """A p.grad kept alive across steps (zero_grad(set_to_none=False), gradient accumulation) must not alias the
    persistent bucket the next backward writes into: accumulating two backwards gives exactly twice the gradient."""
    from bnn_b200 import functional as F
    c = Case('small_cls_mix')
    net = PC.build_net(c, 'cpu').train()
    try:
        opt = bnn_b200.PeerShardedAdam(net.parameters(), lr=1e-3)
        grads = []
        with bnn_b200.eps_mode('reference'):
            for it in range(2):                      # two backwards, no zero_grad in between: accumulation
                torch.manual_seed(5)
                net.sample_elbo(c.x, c.y, c.beta, c.S)[0].backward()
                grads.append(net.l1.weight_mu.grad.detach().clone())
        assert torch.allclose(grads[1], 2 * grads[0], rtol=1e-6, atol=1e-9)
        torch.nn.Module.zero_grad(net, set_to_none=False)             # grads stay alive, zero-filled
        with bnn_b200.eps_mode('reference'):
            torch.manual_seed(5)
            net.sample_elbo(c.x, c.y, c.beta, c.S)[0].backward()
        assert torch.allclose(net.l1.weight_mu.grad, grads[0], rtol=1e-6, atol=1e-9)
    finally:
        F.grad_buckets.clear()


def test_fused_step_above_128_rows_uses_uninitialised_workspace(fake):
    """Batches above 128 rows: no kernel adds into a pre-zeroed output there, so the per-step workspace is allocated
    uninitialised (functional._prezero) and BBB_F_OUT_ZEROED is not passed; the step still equals the oracle's."""
    from bnn_b200 import functional as F
    from oracle import bbb_oracle as O
    torch.manual_seed(3)
    dims, B, S = (6, 9, 4), 150, 2
    layers = O.init_layers(dims, [-0.2, 0.2], [-5, -4])
    x, y = torch.randn(B, dims[0]), torch.randint(0, dims[-1], (B,))
    eps = O.draw_eps(dims, S)
    ref = [tuple(p.clone().requires_grad_(True) for p in layer) for layer in layers]
    want = O.train_step(x, y, ref, O.make_prior([0.5, 0, -6], True), eps, 0.4, 'classification', 1.0)
    assert not F._prezero(B) and F._prezero(128)
    mine = [tuple(p.clone().requires_grad_(True) for p in layer) for layer in layers]
    bnn_b200.rng.set_injected_eps([t for per in eps for pair in per for t in pair])
    with bnn_b200.eps_mode('injected'):
        got = F.fused_elbo(x, y, 0.4, S, 1.0, 'classification', F.make_prior([0.5, 0, -6], True), mine)
    got[0].backward()
    for a, b in zip(got, want):
        assert abs(float(a.detach().reshape(-1)[0]) - float(b.detach().reshape(-1)[0])) <= 1e-5 * abs(float(b.detach().reshape(-1)[0])) + 1e-6
    for la, lb in zip(mine, ref):
        for p, q in zip(la, lb):
            assert (p.grad - q.grad).abs().max() <= 2e-5 * q.grad.abs().max() + 1e-7


def test_large_batch_tf32_step_stores_post_activations(fake):
    """TF32 mode, >= 384 rows: the hidden layers the library can do it for are asked to store max(y, 0)
    (BBB_F_RELU_OUT) and their consumers -- next forward, wgrad, the (x > 0) mask of dgrad, the head -- are called
    without BBB_F_RELU_IN; the step still equals the oracle's."""
    from bnn_b200 import functional as F
    from oracle import bbb_oracle as O
    torch.manual_seed(4)
    dims, B, S = (32, 40, 36, 4), 400, 2
    layers = O.init_layers(dims, [-0.2, 0.2], [-5, -4])
    x, y = torch.randn(B, dims[0]), torch.randint(0, dims[-1], (B,))
    eps = O.draw_eps(dims, S)
    ref = [tuple(p.clone().requires_grad_(True) for p in layer) for layer in layers]
    want = O.train_step(x, y, ref, O.make_prior([0.5, 0, -6], True), eps, 0.4, 'classification', 1.0)
    mine = [tuple(p.clone().requires_grad_(True) for p in layer) for layer in layers]
    assert F._relu_out_layers(mine, B, True) == [True, True, False] and not any(F._relu_out_layers(mine, B, False))
    assert F._relu_out_layers(mine, 128, True) == [False] * 3
    bnn_b200.rng.set_injected_eps([t for per in eps for pair in per for t in pair])
    with bnn_b200.eps_mode('injected'):
        got = F.fused_elbo(x, y, 0.4, S, 1.0, 'classification', F.make_prior([0.5, 0, -6], True), mine, tf32=True)
    got[0].backward()
    for a, b in zip(got, want):
        assert abs(float(a.detach().reshape(-1)[0]) - float(b.detach().reshape(-1)[0])) <= 1e-5 * abs(float(b.detach().reshape(-1)[0])) + 1e-6
    for la, lb in zip(mine, ref):
        for p, q in zip(la, lb):
            assert (p.grad - q.grad).abs().max() <= 2e-5 * q.grad.abs().max() + 1e-7


def test_second_backward_over_a_fused_graph_is_refused(fake):
    """The fused ELBO's backward workspace is single-use (zero-filled by the forward, added into by the kernels), and the
    TF32 LR backward overwrites its saved delta: retain_graph=True + a second backward raises instead of returning wrong
    gradients.  The exact fp32 LR path keeps nothing single-use and may be differentiated twice."""
    c = Case('small_cls_mix')
    net = PC.build_net(c, 'cpu').train()
    with bnn_b200.eps_mode('reference'):
        torch.manual_seed(5)
        loss = net.sample_elbo(c.x, c.y, c.beta, c.S)[0]
    loss.backward(retain_graph=True)
    with pytest.raises(RuntimeError, match='already differentiated'):
        loss.backward()
    c = Case('small_lr_cls')
    for tf32 in (True, False):
        net = PC.build_net(c, 'cpu', tf32=tf32).train()
        with bnn_b200.eps_mode('reference'):
            torch.manual_seed(5)
            loss = net.sample_elbo_lr(c.x, c.y, c.beta, c.S)[0]
        loss.backward(retain_graph=True)
        g1 = net.l1.weight_mu.grad.clone()
        if tf32:
            with pytest.raises(RuntimeError, match='already differentiated'):
                loss.backward()
        else:
            net.zero_grad()
            loss.backward()
            assert torch.allclose(net.l1.weight_mu.grad, g1)


def test_beta_may_be_a_tensor(fake):
    c = Case('small_cls_mix')
    outs = []
    for beta in (c.beta, torch.tensor([c.beta])):
        net = PC.build_net(c, 'cpu').train()
        with bnn_b200.eps_mode('reference'):
            torch.manual_seed(5)
            info = net.sample_elbo(c.x, c.y, beta, c.S)
        info[0].backward()
        outs.append((float(info[0].detach()), net.l2.weight_rho.grad.clone()))
    assert outs[0][0] == outs[1][0] and torch.allclose(outs[0][1], outs[1][1], rtol=1e-6, atol=1e-9)


def test_graphed_step_refuses_the_removed_fused_optimizer():
    """fuse_optimizer is kept as a keyword for existing callers; asking for the removed path fails before anything is
    allocated or captured, whatever the device"""
    c = Case('small_cls_mix')
    net = PC.build_net(c, 'cpu')
    with pytest.raises(ValueError, match='DESIGN.md §4.6'):
        bnn_b200.GraphedTrainStep(net, bnn_b200.FusedAdam(net.parameters()), c.x, c.y, c.S, fuse_optimizer=True)


@pytest.mark.parametrize('name', SMALL + SMALL_LR)
def test_batched_prediction(fake, name):
    PC.check_batched_prediction(Case(name), 'cpu')


@pytest.mark.parametrize('name', ['small_cls_mix', 'deep5_small_mix'])
def test_snr_pruning(fake, name):
    PC.check_snr_pruning(Case(name), 'cpu')


def test_peer_comm_struct_matches_header():
    """ctypes mirror of struct bbb_peer_comm: array lengths follow BBB_MAX_PEERS, field order follows include/bbb.h."""
    import ctypes as C
    hdr = open(os.path.join(ROOT, 'include', 'bbb.h')).read()
    n = int(re.search(r'#define BBB_MAX_PEERS (\d+)', hdr).group(1))
    L = bnn_b200._lib
    fields = dict(L.PeerComm._fields_)
    assert fields['grads']._length_ == n and fields['params']._length_ == n and fields['flags']._length_ == n
    body = re.search(r'typedef struct bbb_peer_comm \{(.*?)\} bbb_peer_comm;', hdr, re.S).group(1)
    body = re.sub(r'/\*.*?\*/', '', body, flags=re.S)                     # declarations only
    order = re.findall(r'\*?(\w+)(?:\[\w+\])?\s*[;,]', body)
    assert order == [f for f, _ in L.PeerComm._fields_]
    assert C.sizeof(L.PeerComm) == 8 + 3 * 8 * n + 32
