"""Per-weight Gaussian priors p(w_i) = N(m_i, softplus(r_i)^2): the bbb_gauss_prior_* kernels and their routing in
BayesianNetwork (posterior_to_prior, set_prior, clear_prior), for both estimators.

CPU: the oracle (oracle/gauss_prior.py) against torch autograd, the host's routing on the CPU double of the C ABI
(extended here by the four new entry points, evaluated with the oracle), the unchanged call sequence of a net without a
per-weight prior, set_prior's errors and the real library's argument checks.  GPU: the kernels against the oracle,
the same eps as the layer kernels, whole steps against float64 autograd, graph replay, row sharding, and sequential
Bayesian updating of a conjugate model."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

import bnn_b200
from bnn_b200 import _lib as L
from bnn_b200 import functional as F
from oracle import bbb_oracle as O
from oracle import gauss_prior as GP
from tests import fake_bbb
from tests.golden_util import PNAMES
from tests.test_heteroscedastic import HetFake

EINVAL = -1
MU_INIT, RHO_INIT = [-0.2, 0.2], [-5, -4]


# ---------------------------------------------------------------------------------------------------------------------
# CPU double of the four new entry points, and a log of every layer call's flags and prior-gradient arguments
# ---------------------------------------------------------------------------------------------------------------------
def _t64(ptr, *shape):
    return torch.from_numpy(fake_bbb._f(ptr, *shape).astype(np.float64))


class PriorFake(HetFake):
    """The double (with bbb_nll_gauss_het) plus the four prior entry points, evaluated with the oracle."""
    log = []

    @staticmethod
    def _tensors(t, nt, bwd):
        if nt < 0 or nt > 64 or (nt and t is None):
            return None
        out = []
        for k in range(nt):
            x = t[k]
            if x.n < 0:
                return None
            if x.n == 0:
                continue
            if not (x.mu and x.rho and x.prior_mu and x.prior_rho) or (bwd and not (x.grad_mu and x.grad_rho)):
                return None
            out.append(x)
        return out

    @staticmethod
    def _vals(x, grad=False):
        mu, rho = (_t64(p, x.n).requires_grad_(grad) for p in (x.mu, x.rho))
        return mu, rho, _t64(x.prior_mu, x.n), _t64(x.prior_rho, x.n)

    @staticmethod
    def _add(x, gm, gr, c):
        for ptr, g in ((x.grad_mu, gm), (x.grad_rho, gr)):
            G = fake_bbb._f(ptr, x.n)
            G[...] = (G + c * g.numpy()).astype(np.float32)

    def bbb_gauss_prior_logprob(self, t, nt, S, rng, logp, logq, st):
        ts = self._tensors(t, nt, False)
        if ts is None or S <= 0 or not (rng and logp and logq):
            return EINVAL
        self.calls.append('gauss_prior_logprob')
        LP, LQ = fake_bbb._d(logp, S), fake_bbb._d(logq, S)
        for x in ts:
            assert x.eps, 'fake lib: inject eps'
            lp, lq = GP.logprob(*self._vals(x), _t64(x.eps, S, x.n))
            LP += lp.numpy()
            LQ += lq.numpy()
        return 0

    def bbb_gauss_prior_logprob_bwd(self, t, nt, S, rng, gp, gq, gp_dev, gq_dev, gstride, oscale, st):
        ts = self._tensors(t, nt, True)
        if ts is None or S <= 0 or not rng or gstride < 0:
            return EINVAL
        self.calls.append('gauss_prior_logprob_bwd')
        PriorFake.log.append(('gauss_prior_logprob_bwd', gp, gq, bool(gp_dev), bool(gq_dev)))
        GPD, GQD = fake_bbb._f(gp_dev, max(1, S * gstride)), fake_bbb._f(gq_dev, max(1, S * gstride))
        gps = torch.tensor([gp * (float(GPD[s * gstride]) if gp_dev else 1.0) for s in range(S)], dtype=torch.float64)
        gqs = torch.tensor([gq * (float(GQD[s * gstride]) if gq_dev else 1.0) for s in range(S)], dtype=torch.float64)
        osc = float(fake_bbb._f(oscale, 1)[0]) if oscale else 1.0
        for x in ts:
            with torch.enable_grad():           # (called from inside autograd's backward)
                mu, rho, m, r = self._vals(x, True)
                lp, lq = GP.logprob(mu, rho, m, r, _t64(x.eps, S, x.n))
                gm, gr = torch.autograd.grad((gps * lp + gqs * lq).sum(), (mu, rho))
            self._add(x, gm, gr, osc)
        return 0

    def bbb_gauss_prior_kl(self, t, nt, kl, st):
        ts = self._tensors(t, nt, False)
        if ts is None or not kl:
            return EINVAL
        self.calls.append('gauss_prior_kl')
        fake_bbb._d(kl, 1)[0] += sum(float(GP.kl(*self._vals(x))) for x in ts)
        return 0

    def bbb_gauss_prior_kl_bwd(self, t, nt, g_kl, g_kl_dev, oscale, st):
        ts = self._tensors(t, nt, True)
        if ts is None:
            return EINVAL
        self.calls.append('gauss_prior_kl_bwd')
        c = g_kl * (float(fake_bbb._f(g_kl_dev, 1)[0]) if g_kl_dev else 1.0)
        c *= float(fake_bbb._f(oscale, 1)[0]) if oscale else 1.0
        for x in ts:
            with torch.enable_grad():
                mu, rho, m, r = self._vals(x, True)
                gm, gr = torch.autograd.grad(GP.kl(mu, rho, m, r), (mu, rho))
            self._add(x, gm, gr, c)
        return 0

    # the flags (and prior-gradient scalars) of every layer-level call
    def bbb_linear_fwd(self, *a):
        PriorFake.log.append(('linear_fwd', a[14]))
        return super().bbb_linear_fwd(*a)

    def bbb_linear_bwd(self, *a):
        PriorFake.log.append(('linear_bwd', a[16], a[17], a[18], bool(a[19]), bool(a[20])))
        return super().bbb_linear_bwd(*a)

    def bbb_head_fwd(self, *a):
        PriorFake.log.append(('head_fwd', a[14]))
        return super().bbb_head_fwd(*a)

    def bbb_lr_linear_fwd(self, *a):
        PriorFake.log.append(('lr_fwd', a[14]))
        return super().bbb_lr_linear_fwd(*a)

    def bbb_lr_linear_bwd(self, *a):
        PriorFake.log.append(('lr_bwd', a[17]))
        return super().bbb_lr_linear_bwd(*a)

    def bbb_mlp_fwd(self, *a):
        PriorFake.log.append(('mlp_fwd', a[7]))
        n = len(PriorFake.log)
        st = super().bbb_mlp_fwd(*a)
        del PriorFake.log[n:]
        return st

    def bbb_mlp_bwd(self, *a):
        PriorFake.log.append(('mlp_bwd', a[7], a[8], a[9], bool(a[10]), bool(a[11])))
        n = len(PriorFake.log)
        st = super().bbb_mlp_bwd(*a)
        del PriorFake.log[n:]
        return st


@pytest.fixture
def fake(monkeypatch):
    lib = PriorFake()
    fake_bbb.FakeLib.calls = []
    PriorFake.log = []
    monkeypatch.setattr(bnn_b200._lib, 'lib', lambda: lib)
    monkeypatch.setattr(bnn_b200._lib, 'require_cuda', lambda *a: None)
    monkeypatch.setattr(bnn_b200._lib, 'stream', lambda: None)
    return lib


# ---------------------------------------------------------------------------------------------------------------------
# shared helpers
# ---------------------------------------------------------------------------------------------------------------------
def _model_params(dims, D, lr=False, mixture=None, **extra):
    mixture = (not lr) if mixture is None else mixture
    mp = dict(input_shape=dims[0], classes=D, batch_size=128, hidden_units=list(dims[1:]), mode='regression',
              mu_init=MU_INIT, rho_init=RHO_INIT, prior_init=[0.5, 0, -6] if mixture else [0.3], mixture_prior=mixture,
              local_reparam=lr)
    mp.update(extra)
    return mp


def _make_net(dims, D, device, seed=0, **kw):
    torch.manual_seed(seed)
    return bnn_b200.BayesianNetwork(_model_params(dims, D, **kw)).to(device)


def _data(B, n_in, D, seed=1):
    g = torch.Generator().manual_seed(seed)
    x = 2 * torch.rand(B, n_in, generator=g) - 1
    v = torch.randn(n_in, D, generator=g) / math.sqrt(n_in)
    return x, torch.sin(3 * x @ v) + 0.1 * torch.randn(B, D, generator=g)


def _random_prior(net, seed=3):
    """A non-trivial per-weight prior: m ~ 0.1 N(0, 1), sigma ~ U[0.05, 0.5], per weight and bias."""
    g = torch.Generator().manual_seed(seed)
    dev = net.l1.weight_mu.device
    entries = []
    for l in net.layers():
        e = []
        for ref in (l.weight_mu, l.bias_mu):
            e += [(0.1 * torch.randn(ref.shape, generator=g)).to(dev),
                  (0.05 + 0.45 * torch.rand(ref.shape, generator=g)).to(dev)]
        entries.append(tuple(e))
    net.set_prior(entries)
    return entries


def _maxnorm_err(got, want):
    g, w = torch.as_tensor(got).double().cpu(), torch.as_tensor(want).double().cpu()
    return float((g - w).abs().max()) / max(float(w.abs().max()), 1e-300)


def _het_nll(out, y, sigma_min):
    D = out.shape[-1] // 2
    f, r = out[..., :D], out[..., D:]
    s = sigma_min + torch.clamp(r, min=0) + torch.log1p(torch.exp(-r.abs()))
    return (0.5 * ((y - f) / s) ** 2 + torch.log(s) + 0.5 * math.log(2 * math.pi)).sum()


def _oracle_step(net, x, y, S, beta, eps, lr, sigma):
    """float64 sample_elbo[_lr] with the net's per-weight prior, the given draws and autograd gradients"""
    layers = [tuple(t.detach().cpu().double().requires_grad_() for t in l.params()) for l in net.layers()]
    priors = [tuple(t.detach().cpu().double() for t in bnn_b200.layers.gauss_prior(l)) for l in net.layers()]
    x64, y64 = x.detach().cpu().double(), y.detach().cpu().double()
    nll = torch.zeros((), dtype=torch.float64)
    terms = []
    for s in range(S):
        h = x64
        lp = lq = kl = 0
        for li, (layer, pr) in enumerate(zip(layers, priors)):
            e1, e2 = (t.double() for t in eps[s][li])
            if lr:
                h, _ = O.lr_linear(h, layer, 1.0, e1, e2, calc_kl=False)
                kl = kl + GP.kl(layer[0], layer[1], pr[0], pr[1]) + GP.kl(layer[2], layer[3], pr[2], pr[3])
            else:
                h, _, _ = O.bayes_linear(h, layer, ('gaussian', 1.0), e1, e2, calc_log_probs=False)
                for a, b in ((0, 0), (2, 2)):
                    p_, q_ = GP.logprob(layer[a], layer[a + 1], pr[b], pr[b + 1], (e1 if a == 0 else e2)[None])
                    lp, lq = lp + p_[0], lq + q_[0]
            if li + 1 < len(layers):
                h = torch.relu(h)
        terms.append(kl if lr else (lp, lq))
        nll = nll + (_het_nll(h, y64, net.sigma_min) if net._het else O.nll(h, y64, 'regression', sigma))
    nll = nll / S
    if lr:
        k = torch.stack(terms).mean()
        loss = beta * k + nll
        scalars = (loss, k, nll)
    else:
        lps = torch.stack([t[0] for t in terms]).mean()
        lqs = torch.stack([t[1] for t in terms]).mean()
        loss = beta * lqs - beta * lps + nll
        scalars = (loss, lps, lqs, nll)
    loss.backward()
    return [float(v.detach()) for v in scalars], [[t.grad for t in l] for l in layers]


def _net_step(net, x, y, S, beta, seed, sigma=1.0):
    net.train()
    net.zero_grad()
    with bnn_b200.eps_mode('reference'):
        torch.manual_seed(seed)
        info = (net.sample_elbo_lr if net.local_reparam else net.sample_elbo)(x, y, beta, S, sigma)
    info[0].backward()
    return [float(v.detach().reshape(-1)[0]) for v in info], [[p.grad for p in l.params()] for l in net.layers()]


def check_step(dims, D, B, S, device, lr=False, tf32=False, rtol=1e-5, rtol_gemm=None, seed=5, **kw):
    """sample_elbo[_lr] with a non-trivial per-weight prior in the reference eps mode against float64 autograd of the
    oracle under the same draws; rtol bounds the prior scalars, rtol_gemm everything downstream of a contraction."""
    rg = rtol if rtol_gemm is None else rtol_gemm
    net = _make_net(dims, D, device, lr=lr, tf32=tf32, **kw)
    _random_prior(net)
    x, y = _data(B, dims[0], D)
    sigma = 1.0 if net._het else 0.5
    out_w = D * (2 if net._het else 1)
    with torch.random.fork_rng():
        torch.manual_seed(seed)
        eps = O.draw_eps(list(dims) + [out_w], S, batch=B, local_reparam=lr)
    want_s, want_g = _oracle_step(net, x, y, S, 0.3, eps, lr, sigma)
    got_s, got_g = _net_step(net, x.to(device), y.to(device), S, 0.3, seed, sigma)
    scale = sum(abs(v) for v in want_s[1:])
    assert abs(got_s[0] - want_s[0]) <= rg * scale, ('loss', got_s[0], want_s[0])
    for k in range(1, len(want_s) - 1):
        assert abs(got_s[k] - want_s[k]) <= rtol * abs(want_s[k]), (k, got_s[k], want_s[k])
    assert abs(got_s[-1] - want_s[-1]) <= rg * abs(want_s[-1]), ('nll', got_s[-1], want_s[-1])
    worst = 0.0
    for li, (gl, wl) in enumerate(zip(got_g, want_g)):
        for pn, g, w in zip(PNAMES, gl, wl):
            err = _maxnorm_err(g, w)
            assert err <= rg, f'l{li + 1}.{pn}: max-norm relative error {err:.3e} > {rg:.1e}'
            worst = max(worst, err)
    return worst


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the oracle
# ---------------------------------------------------------------------------------------------------------------------
def _rand_layer(n, seed):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(n, generator=g, dtype=torch.float64), torch.rand(n, generator=g, dtype=torch.float64) * 4 - 6,
            0.3 * torch.randn(n, generator=g, dtype=torch.float64), torch.rand(n, generator=g, dtype=torch.float64) - 2)


def test_oracle_matches_torch_distributions_and_the_header_gradients():
    """log p, log q against torch.distributions; the KL against torch.distributions.kl_divergence; the gradients of
    both by autograd against the closed forms bbb.h states."""
    mu, rho, m, r = _rand_layer(37, 0)
    mu.requires_grad_()
    rho.requires_grad_()
    eps = torch.randn(3, 37, dtype=torch.float64, generator=torch.Generator().manual_seed(1))
    sg, sp = GP.softplus(rho), GP.softplus(r)
    lp, lq = GP.logprob(mu, rho, m, r, eps)
    w = mu + sg * eps
    N = torch.distributions.Normal
    torch.testing.assert_close(lp, N(m, sp).log_prob(w).sum(1), rtol=1e-12, atol=1e-12)
    torch.testing.assert_close(lq, N(mu, sg).log_prob(w).sum(1), rtol=1e-12, atol=1e-12)
    gp, gq = torch.tensor([0.3, -1.2, 2.0], dtype=torch.float64), torch.tensor([-0.7, 0.4, 1.1], dtype=torch.float64)
    gm, gr = torch.autograd.grad((gp * lp + gq * lq).sum(), (mu, rho))
    with torch.no_grad():
        t = -gp[:, None] * (w - m) / sp ** 2
        torch.testing.assert_close(gm, t.sum(0), rtol=1e-12, atol=1e-12)
        torch.testing.assert_close(gr, torch.sigmoid(rho) * (t * eps - gq[:, None] / sg).sum(0), rtol=1e-12, atol=1e-12)
    kl = GP.kl(mu, rho, m, r)
    want = torch.distributions.kl_divergence(N(mu, sg), N(m, sp)).sum()
    assert abs(float(kl.detach()) - float(want.detach())) <= 1e-12 * abs(float(want.detach()))
    gm, gr = torch.autograd.grad(kl, (mu, rho))
    with torch.no_grad():
        torch.testing.assert_close(gm, (mu - m) / sp ** 2, rtol=1e-12, atol=1e-12)
        torch.testing.assert_close(gr, torch.sigmoid(rho) * (sg / sp ** 2 - 1 / sg), rtol=1e-12, atol=1e-12)
    assert float(GP.kl(mu, rho, mu, rho).detach()) == pytest.approx(0.0, abs=1e-12)
    torch.testing.assert_close(GP.softplus(GP.sigma_to_rho(sp)), sp, rtol=1e-12, atol=0)


# ---------------------------------------------------------------------------------------------------------------------
# CPU: routing on the double
# ---------------------------------------------------------------------------------------------------------------------
def _routing(dims, D, lr=False, tf32=False, prior=True, fused=True, B=16, **kw):
    net = _make_net(dims, D, 'cpu', lr=lr, tf32=tf32, fused=fused, **kw)
    if prior:
        _random_prior(net)
    x, y = _data(B, dims[0], D)
    fake_bbb.FakeLib.calls = []
    PriorFake.log = []
    with bnn_b200.eps_mode('reference'):
        info = (net.sample_elbo_lr if lr else net.sample_elbo)(x, y, 0.5, 2)
    fwd, nlog = list(fake_bbb.FakeLib.calls), len(PriorFake.log)
    info[0].backward()
    return fwd, fake_bbb.FakeLib.calls[len(fwd):], PriorFake.log[:nlog], PriorFake.log[nlog:]


NOLP = ~L.F_LOGPROB


@pytest.mark.parametrize('fused', [True, False])
def test_weight_sampling_routing(fake, fused):
    """The prior kernel runs once before the layers, which run without BBB_F_LOGPROB, and once after the layer
    backward, which gets gp = gq = 0 and no device multipliers."""
    fwd, bwd, flog, blog = _routing((8, 16, 16), 1, fused=fused)
    assert fwd[0] == 'gauss_prior_logprob' and fwd.count('gauss_prior_logprob') == 1
    assert fwd[1:4] == ['linear_fwd', 'linear_fwd', 'head_fwd' if fused else 'linear_fwd']
    assert all(not e[1] & L.F_LOGPROB for e in flog)
    assert bwd == ['linear_bwd'] * 3 + ['gauss_prior_logprob_bwd']
    assert all(e[2:] == (0.0, 0.0, False, False) for e in blog if e[0] == 'linear_bwd')
    gp, gq = blog[-1][1:3]
    if fused:
        assert (gp, gq) == (pytest.approx(-0.25), pytest.approx(0.25))         # -beta / S, beta / S
    else:
        assert blog[-1][3:] == (True, True)                                   # per-sample device multipliers


def test_network_level_routing(fake):
    fwd, bwd, flog, blog = _routing((8, 16, 16), 1, tf32=True)
    assert fwd == ['gauss_prior_logprob', 'mlp_fwd', 'head_fwd']
    assert flog == [('mlp_fwd', L.F_SAMPLE | L.F_TF32)]
    assert bwd == ['mlp_bwd', 'gauss_prior_logprob_bwd']
    assert blog[0] == ('mlp_bwd', L.F_SAMPLE | L.F_TF32, 0.0, 0.0, False, False)


@pytest.mark.parametrize('het', [False, True])
def test_lr_and_heteroscedastic_routing(fake, het):
    kw = dict(likelihood='heteroscedastic') if het else {}
    fwd, bwd, flog, blog = _routing((8, 16, 16), 2, lr=True, **kw)
    assert fwd[:4] == ['gauss_prior_kl', 'lr_fwd', 'lr_fwd', 'lr_fwd']
    assert fwd[4] == ('nll_gauss_het' if het else 'nll_gauss')
    assert all(not e[1] & L.F_LOGPROB for e in flog + blog)
    assert bwd == ['lr_bwd'] * 3 + ['gauss_prior_kl_bwd']
    if het:
        fwd, bwd, _, _ = _routing((8, 16, 16), 2, **kw)
        assert fwd[:4] == ['gauss_prior_logprob', 'linear_fwd', 'linear_fwd', 'linear_fwd']
        assert bwd == ['linear_bwd'] * 3 + ['gauss_prior_logprob_bwd']


@pytest.mark.parametrize('lr,tf32,fused', [(False, False, True), (False, True, True), (False, False, False),
                                           (True, False, True), (True, False, False)])
def test_without_a_prior_the_calls_are_unchanged(fake, lr, tf32, fused):
    """No per-weight prior (never set, or cleared): exactly the calls, flags and prior-gradient arguments of a net
    built without the feature."""
    base = _routing((8, 16, 16), 1, lr=lr, tf32=tf32, fused=fused, prior=False)
    net_calls = [c for c in base[0] + base[1]]
    assert not any('gauss_prior' in c for c in net_calls)
    assert any(e[1] & L.F_LOGPROB for e in base[2])
    # a net whose prior was set and then cleared makes the same calls as one that never had one
    net = _make_net((8, 16, 16), 1, 'cpu', lr=lr, tf32=tf32, fused=fused)
    _random_prior(net)
    net.clear_prior()
    x, y = _data(16, 8, 1)
    fake_bbb.FakeLib.calls = []
    PriorFake.log = []
    with bnn_b200.eps_mode('reference'):
        info = (net.sample_elbo_lr if lr else net.sample_elbo)(x, y, 0.5, 2)
    info[0].backward()
    assert fake_bbb.FakeLib.calls == base[0] + base[1]
    assert PriorFake.log == base[2] + base[3]


@pytest.mark.parametrize('lr', [False, True])
@pytest.mark.parametrize('kw', [{}, dict(fused=False), dict(likelihood='heteroscedastic')], ids=['fused', 'unfused',
                                                                                               'het'])
def test_step_on_the_double_matches_the_oracle(fake, lr, kw):
    check_step((3, 16, 16), 2, 12, 3, 'cpu', lr=lr, **kw)


@pytest.mark.parametrize('lr', [False, True])
def test_layer_log_probs_reflect_the_prior(fake, lr):
    """net.log_prior() / log_variational_posterior() / kl_cost() after a training-mode forward use the per-weight
    prior (the single-layer autograd function), and their gradients flow."""
    net = _make_net((3, 8), 2, 'cpu', lr=lr)
    _random_prior(net)
    x, _ = _data(5, 3, 2)
    net.train()
    with bnn_b200.eps_mode('reference'):
        torch.manual_seed(4)
        net(x)
        torch.manual_seed(4)
        eps = O.draw_eps([3, 8, 2], 1, batch=5, local_reparam=lr)[0]
    pr = [tuple(t.double() for t in bnn_b200.layers.gauss_prior(l)) for l in net.layers()]
    layers = [tuple(t.detach().double() for t in l.params()) for l in net.layers()]
    if lr:
        want = sum(float(GP.kl(p[0], p[1], q[0], q[1]) + GP.kl(p[2], p[3], q[2], q[3])) for p, q in zip(layers, pr))
        assert float(net.kl_cost()) == pytest.approx(want, rel=1e-6)
        net.kl_cost().backward()
    else:
        lp = lq = 0.0
        for p, q, (ew, eb) in zip(layers, pr, eps):
            for a, e in ((0, ew), (2, eb)):
                u, v = GP.logprob(p[a], p[a + 1], q[a], q[a + 1], e.double()[None])
                lp, lq = lp + float(u), lq + float(v)
        assert float(net.log_prior()) == pytest.approx(lp, rel=1e-6)
        assert float(net.log_variational_posterior()) == pytest.approx(lq, rel=1e-6)
        (net.log_variational_posterior() - net.log_prior()).backward()
    assert fake_bbb.FakeLib.calls.count('gauss_prior_kl_bwd' if lr else 'gauss_prior_logprob_bwd') == 2
    assert all(p.grad is not None and bool(torch.isfinite(p.grad).all()) for p in net.parameters())


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the public API
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('lr', [False, True])
def test_posterior_to_prior_set_prior_clear_prior(lr):
    net = _make_net((3, 16, 16), 2, 'cpu', lr=lr)
    keys = list(net.state_dict().keys())
    assert all(bnn_b200.layers.gauss_prior(l) is None for l in net.layers())
    net.posterior_to_prior()
    for l in net.layers():
        for b, p in zip(bnn_b200.layers.gauss_prior(l), l.params()):
            assert torch.equal(b, p.detach()) and b.data_ptr() != p.data_ptr() and not b.requires_grad
    assert list(net.state_dict().keys()) == keys                    # the prior is not part of the state_dict
    ptrs = [b.data_ptr() for l in net.layers() for b in bnn_b200.layers.gauss_prior(l)]
    with torch.no_grad():
        net.l1.weight_mu.add_(1.0)
    net.posterior_to_prior()                                        # in place: a captured graph keeps reading them
    assert [b.data_ptr() for l in net.layers() for b in bnn_b200.layers.gauss_prior(l)] == ptrs
    assert torch.equal(net.l1.prior_weight_mu, net.l1.weight_mu.detach())
    net.set_prior([(0.0, 0.2, 0.1, 1e-5)] * 3)
    assert [b.data_ptr() for l in net.layers() for b in bnn_b200.layers.gauss_prior(l)] == ptrs
    sp = torch.log1p(torch.exp(net.l2.prior_weight_rho.double()))
    assert torch.allclose(sp, torch.full_like(sp, 0.2), rtol=1e-6)
    sp = torch.log1p(torch.exp(net.l2.prior_bias_rho.double()))
    assert torch.allclose(sp, torch.full_like(sp, 1e-5), rtol=1e-5)
    assert bool((net.l3.prior_bias_mu == 0.1).all())
    net.clear_prior()
    assert all(bnn_b200.layers.gauss_prior(l) is None for l in net.layers())
    assert list(net.state_dict().keys()) == keys


def test_set_prior_errors():
    net = _make_net((3, 16, 4), 2, 'cpu')
    good = [(torch.zeros(l.weight_mu.shape), torch.ones(l.weight_mu.shape), torch.zeros(l.bias_mu.shape),
             torch.ones(l.bias_mu.shape)) for l in net.layers()]
    bad = []
    bad.append((good[:2], 'per layer'))
    bad.append(([good[0][:3]] + good[1:], 'expected'))
    bad.append(([(good[0][0].t(),) + good[0][1:]] + good[1:], 'shape'))
    bad.append(([good[0][:3] + (torch.ones(5),)] + good[1:], 'shape'))
    for s in (0.0, -1.0, float('nan'), float('inf')):
        bad.append(([(0.0, s, 0.0, 1.0)] * 3, 'sigma'))
        w = good[1][1].clone()
        w[0, 0] = s
        bad.append(([good[0], (good[1][0], w) + good[1][2:], good[2]], 'sigma'))
    bad.append(([(torch.zeros(good[0][0].shape, device='meta'),) + good[0][1:]] + good[1:], 'device'))
    for entries, msg in bad:
        with pytest.raises(ValueError, match=msg):
            net.set_prior(entries)
        assert all(bnn_b200.layers.gauss_prior(l) is None for l in net.layers())   # nothing changed
    net.set_prior(good)
    net.l2.prior_weight_mu = None                                   # a prior on some layers only
    x, y = _data(4, 3, 2)
    with pytest.raises(ValueError, match='every layer'):
        net.sample_elbo(x, y, 1.0, 1)


def test_abi_rejects_bad_arguments():
    """The real library's argument checks (they return before any device work, so they run without a GPU)."""
    lib = L.lib()
    buf = 16                          # never dereferenced: every call below is refused first
    rng = L.Rng(0, 0, 0, 0, None)

    def table(**change):
        t = (L.GaussPriorTensor * 2)()
        for x in t:
            x.mu = x.rho = x.prior_mu = x.prior_rho = x.grad_mu = x.grad_rho = buf
            x.n = 8
        for k, v in change.items():
            setattr(t[1], k, v)
        return t

    ok = table()
    for t, n in ((ok, -1), (ok, 65), (None, 2)):
        assert lib.bbb_gauss_prior_logprob(t, n, 2, C.byref(rng), buf, buf, None) == EINVAL
        assert lib.bbb_gauss_prior_logprob_bwd(t, n, 2, C.byref(rng), 1.0, 1.0, None, None, 0, None, None) == EINVAL
        assert lib.bbb_gauss_prior_kl(t, n, buf, None) == EINVAL
        assert lib.bbb_gauss_prior_kl_bwd(t, n, 1.0, None, None, None) == EINVAL
    for change in (dict(n=-1), dict(mu=None), dict(rho=None), dict(prior_mu=None), dict(prior_rho=None)):
        t = table(**change)
        assert lib.bbb_gauss_prior_logprob(t, 2, 2, C.byref(rng), buf, buf, None) == EINVAL, change
        assert lib.bbb_gauss_prior_logprob_bwd(t, 2, 2, C.byref(rng), 1.0, 1.0, None, None, 0, None, None) == EINVAL
        assert lib.bbb_gauss_prior_kl(t, 2, buf, None) == EINVAL, change
        assert lib.bbb_gauss_prior_kl_bwd(t, 2, 1.0, None, None, None) == EINVAL, change
    for change in (dict(grad_mu=None), dict(grad_rho=None)):
        t = table(**change)
        assert lib.bbb_gauss_prior_logprob_bwd(t, 2, 2, C.byref(rng), 1.0, 1.0, None, None, 0, None, None) == EINVAL
        assert lib.bbb_gauss_prior_kl_bwd(t, 2, 1.0, None, None, None) == EINVAL
    for S in (0, -3):
        assert lib.bbb_gauss_prior_logprob(ok, 2, S, C.byref(rng), buf, buf, None) == EINVAL
        assert lib.bbb_gauss_prior_logprob_bwd(ok, 2, S, C.byref(rng), 1.0, 1.0, None, None, 0, None, None) == EINVAL
    assert lib.bbb_gauss_prior_logprob(ok, 2, 2, None, buf, buf, None) == EINVAL
    assert lib.bbb_gauss_prior_logprob(ok, 2, 2, C.byref(rng), None, buf, None) == EINVAL
    assert lib.bbb_gauss_prior_logprob(ok, 2, 2, C.byref(rng), buf, None, None) == EINVAL
    assert lib.bbb_gauss_prior_logprob_bwd(ok, 2, 2, None, 1.0, 1.0, None, None, 0, None, None) == EINVAL
    assert lib.bbb_gauss_prior_kl(ok, 2, None, None) == EINVAL
    # empty tensors (null pointers allowed) and an empty table launch nothing
    empty = table(n=0, mu=None, rho=None, prior_mu=None, prior_rho=None, grad_mu=None, grad_rho=None)
    empty[0].n = 0
    assert lib.bbb_gauss_prior_logprob(empty, 2, 2, C.byref(rng), buf, buf, None) == 0
    assert lib.bbb_gauss_prior_logprob_bwd(empty, 2, 2, C.byref(rng), 1.0, 1.0, None, None, 0, None, None) == 0
    assert lib.bbb_gauss_prior_kl(empty, 2, buf, None) == 0
    assert lib.bbb_gauss_prior_kl_bwd(None, 0, 1.0, None, None, None) == 0


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the kernels against the oracle
# ---------------------------------------------------------------------------------------------------------------------
SIZES = (1, 3, 4, 5, 7, 64, 1001, 4099)


def _kernel_tensors(offset, seed=0):
    """Tensors of every size in SIZES as views of one flat buffer per role, starting `offset` elements in (offset 1:
    none is 16-byte aligned), with a non-trivial prior."""
    g = torch.Generator().manual_seed(seed)
    total = sum(SIZES) + offset
    flat = {k: torch.empty(total, dtype=torch.float32, device='cuda') for k in ('mu', 'rho', 'pm', 'pr', 'gm', 'gr')}
    vals = dict(mu=torch.randn(total, generator=g), rho=torch.rand(total, generator=g) * 4 - 6,
                pm=0.3 * torch.randn(total, generator=g), pr=torch.rand(total, generator=g) - 2,
                gm=torch.randn(total, generator=g), gr=torch.randn(total, generator=g))
    for k in flat:
        flat[k].copy_(vals[k])
    out, off = [], offset
    for n in SIZES:
        out.append({k: flat[k][off:off + n] for k in flat})
        off += n
    return out


def _table(ts, eps=None, ids=None):
    tab = (L.GaussPriorTensor * len(ts))()
    for i, t in enumerate(ts):
        x = tab[i]
        x.mu, x.rho, x.prior_mu, x.prior_rho = (t[k].data_ptr() for k in ('mu', 'rho', 'pm', 'pr'))
        x.grad_mu, x.grad_rho = t['gm'].data_ptr(), t['gr'].data_ptr()
        x.eps = None if eps is None else eps[i].data_ptr()
        x.n, x.tensor_id = t['mu'].numel(), (ids[i] if ids else i)
    return tab


def _d64(t):
    return t.detach().cpu().double()


@pytest.mark.gpu
@pytest.mark.parametrize('S', [1, 3, 8, 11])
@pytest.mark.parametrize('offset', [0, 1], ids=['aligned', 'unaligned'])
@pytest.mark.parametrize('injected', [False, True], ids=['philox', 'injected'])
def test_gpu_logprob_kernels_match_the_oracle(S, offset, injected):
    """bbb_gauss_prior_logprob and its backward against the oracle: every size of SIZES in one launch, aligned and
    unaligned views, injected eps or Philox (the oracle then takes the stream bbb_philox_fill_normal writes), per-sample
    device multipliers.  Values and gradients within 1e-5 relative."""
    ts = _kernel_tensors(offset)
    seed, step, base = 1234, 7, 3
    ids = [2 * i + (i % 2) for i in range(len(ts))]
    if injected:
        eps = [torch.randn(S, t['mu'].numel(), generator=torch.Generator().manual_seed(i)).cuda()
               for i, t in enumerate(ts)]
        if offset:                                                       # unaligned eps rows too
            eps = [torch.cat([torch.zeros(1, device='cuda'), e.reshape(-1)])[1:].view_as(e) for e in eps]
    else:
        eps = [torch.stack([F.philox_normal(t['mu'].numel(), 'cuda', seed, step, base + s, ids[i]) for s in range(S)])
               for i, t in enumerate(ts)]
    tab = _table(ts, eps if injected else None, ids)
    rng = L.Rng(seed, step, base, 0, None)
    acc = torch.zeros(2 * S, dtype=torch.float64, device='cuda')
    st = L.stream()
    L.check(L.lib().bbb_gauss_prior_logprob(tab, len(ts), S, C.byref(rng), acc[:S].data_ptr(), acc[S:].data_ptr(),
                                            st), 'logprob')
    gpd = torch.linspace(-1.0, 2.0, S, device='cuda')
    gqd = torch.linspace(0.5, -0.7, S, device='cuda')
    oscale = torch.tensor([0.75], device='cuda')
    before = [(_d64(t['gm']), _d64(t['gr'])) for t in ts]
    L.check(L.lib().bbb_gauss_prior_logprob_bwd(tab, len(ts), S, C.byref(rng), 0.4, -1.5, gpd.data_ptr(),
                                                gqd.data_ptr(), 1, oscale.data_ptr(), st), 'logprob_bwd')
    torch.cuda.synchronize()
    lp = lq = 0
    gp = 0.4 * _d64(gpd)
    gq = -1.5 * _d64(gqd)
    for t, e, (gm0, gr0) in zip(ts, eps, before):
        mu, rho = _d64(t['mu']).requires_grad_(), _d64(t['rho']).requires_grad_()
        u, v = GP.logprob(mu, rho, _d64(t['pm']), _d64(t['pr']), _d64(e))
        lp, lq = lp + u.detach(), lq + v.detach()
        gm, gr = torch.autograd.grad((gp * u + gq * v).sum(), (mu, rho))
        for got, g0, w in ((t['gm'], gm0, gm), (t['gr'], gr0, gr)):
            d = _d64(got) - g0
            assert _maxnorm_err(d, 0.75 * w) <= 1e-5, (t['mu'].numel(), _maxnorm_err(d, 0.75 * w))
    for got, want in ((acc[:S], lp), (acc[S:], lq)):
        np.testing.assert_allclose(got.cpu().numpy(), want.numpy(), rtol=1e-5)


@pytest.mark.gpu
@pytest.mark.parametrize('offset', [0, 1], ids=['aligned', 'unaligned'])
def test_gpu_kl_kernels_match_the_oracle(offset):
    ts = _kernel_tensors(offset, seed=4)
    tab = _table(ts)
    kl = torch.zeros(1, dtype=torch.float64, device='cuda')
    gk = torch.tensor([2.0], device='cuda')
    osc = torch.tensor([0.5], device='cuda')
    before = [(_d64(t['gm']), _d64(t['gr'])) for t in ts]
    st = L.stream()
    L.check(L.lib().bbb_gauss_prior_kl(tab, len(ts), kl.data_ptr(), st), 'kl')
    L.check(L.lib().bbb_gauss_prior_kl_bwd(tab, len(ts), 0.3, gk.data_ptr(), osc.data_ptr(), st), 'kl_bwd')
    torch.cuda.synchronize()
    want = 0
    for t, (gm0, gr0) in zip(ts, before):
        mu, rho = _d64(t['mu']).requires_grad_(), _d64(t['rho']).requires_grad_()
        k = GP.kl(mu, rho, _d64(t['pm']), _d64(t['pr']))
        want = want + float(k)
        gm, gr = torch.autograd.grad(k, (mu, rho))
        for got, g0, w in ((t['gm'], gm0, gm), (t['gr'], gr0, gr)):
            assert _maxnorm_err(_d64(got) - g0, 0.3 * w) <= 1e-5
    assert float(kl) == pytest.approx(want, rel=1e-5)


@pytest.mark.gpu
@pytest.mark.parametrize('lr', [False, True])
def test_gpu_kl_is_exactly_zero_after_posterior_to_prior(lr):
    """q == p, including trained-posterior scales sigma ~ 1e-5: the KL is exactly 0 (every element's term is 0 in fp32)
    and so are its gradients; the Monte Carlo log p - log q of weight sampling is 0 up to round-off."""
    net = _make_net((9, 33, 5), 3, 'cuda', lr=True)
    with torch.no_grad():
        net.l1.weight_rho[:4] = -11.5                                      # sigma ~ 1e-5
    net.posterior_to_prior()
    params = [l.params() for l in net.layers()]
    gauss = [bnn_b200.layers.gauss_prior(l) for l in net.layers()]
    grads = [[torch.zeros_like(p) for p in l] for l in params]
    tab, n, _ = F._gauss_prior_table(params, gauss, F._EpsPlan(), True, 1, grads)
    kl = torch.zeros(1, dtype=torch.float64, device='cuda')
    L.check(L.lib().bbb_gauss_prior_kl(tab, n, kl.data_ptr(), L.stream()), 'kl')
    L.check(L.lib().bbb_gauss_prior_kl_bwd(tab, n, 1.0, None, None, L.stream()), 'kl_bwd')
    assert float(kl) == 0.0
    assert all(bool((g == 0).all()) for l in grads for g in l)
    net.train()
    info = net.sample_elbo_lr(torch.randn(4, 9, device='cuda'), torch.randn(4, 3, device='cuda'), 1.0, 2)
    assert float(info[1]) == 0.0


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the same eps as the layer kernels, whole steps, graphs, sharding
# ---------------------------------------------------------------------------------------------------------------------
def _philox_step(net, x, y, S, seed):
    net.train()
    net.zero_grad()
    bnn_b200.manual_seed(seed, 4)
    info = (net.sample_elbo_lr if net.local_reparam else net.sample_elbo)(x, y, 0.2, S, 0.5)
    info[0].backward()
    return [float(v.detach().reshape(-1)[0]) for v in info], [p.grad.clone() for p in net.parameters()]


@pytest.mark.gpu
@pytest.mark.parametrize('B', [128, 640])
@pytest.mark.parametrize('lr', [False, True], ids=['ws', 'lr'])
@pytest.mark.parametrize('tf32', [False, True], ids=['fp32', 'tf32'])
def test_gpu_scalar_prior_as_a_per_weight_prior_reproduces_the_scalar_path(B, lr, tf32):
    """Every weight's prior set to N(0, sigma1): the step reproduces the scalar-Gaussian path (mixture_prior=False) on
    the same Philox stream, loss, every returned scalar and every gradient within 1e-5, on the network-level route (TF32,
    B = 128) and the per-layer ones.  So the prior kernel regenerates the very eps the layer kernels drew."""
    dims, D, S = (16, 64, 64), 2, 3
    x, y = _data(B, dims[0], D, seed=2)
    x, y = x.cuda(), y.cuda()
    res = []
    for prior in (False, True):
        net = _make_net(dims, D, 'cuda', lr=lr, tf32=tf32, mixture=False)
        if prior:
            net.set_prior([(0.0, 0.3, 0.0, 0.3)] * net.n_layers)
        res.append(_philox_step(net, x, y, S, 21))
    (sa, ga), (sb, gb) = res
    np.testing.assert_allclose(sb, sa, rtol=1e-5, atol=0)
    for a, b in zip(ga, gb):
        assert _maxnorm_err(b, a) <= 1e-5, _maxnorm_err(b, a)


CFG = ((16, 64, 64), 2, 128, 3)
DEEP = ((16, 128, 128, 128), 2, 640, 3)


@pytest.mark.gpu
@pytest.mark.parametrize('cfg', [CFG, DEEP], ids=['b128', 'deep4_b640'])
@pytest.mark.parametrize('lr', [False, True], ids=['ws', 'lr'])
@pytest.mark.parametrize('tf32', [False, True], ids=['fp32', 'tf32'])
def test_gpu_step_matches_float64_autograd(cfg, lr, tf32):
    """A whole step with a non-trivial per-weight prior (m != 0, per-weight sp) in the reference eps mode against
    float64 autograd of the oracle: fp32 within 1e-5, TF32 at the bounds of DESIGN §2 (5e-3 downstream of a contraction,
    local reparameterisation 2e-2, 1e-5 on the prior scalars).  Weight sampling on the 4-layer batch-640 net measured
    1.07e-2 on a B200, in the last layer's bias_rho gradient: the fp32 prior terms cancel most of the TF32 data term
    there, so the kernels' TF32 rounding is large against the max-norm (DESIGN §4.4c has the same family at 5.1e-3
    without a prior); that case is held to 2e-2 (DESIGN §4.4d)."""
    dims, D, B, S = cfg
    rg = (2e-2 if lr or cfg is DEEP else 5e-3) if tf32 else 1e-5
    check_step(dims, D, B, S, 'cuda', lr=lr, tf32=tf32, rtol_gemm=rg)


@pytest.mark.gpu
@pytest.mark.parametrize('lr', [False, True], ids=['ws', 'lr'])
@pytest.mark.parametrize('kw', [dict(likelihood='heteroscedastic'), dict(fused=False)], ids=['het', 'unfused'])
def test_gpu_het_and_unfused_steps_match_float64_autograd(lr, kw):
    dims, D, B, S = CFG
    check_step(dims, D, B, S, 'cuda', lr=lr, **kw)


@pytest.mark.gpu
@pytest.mark.parametrize('lr', [False, True], ids=['ws', 'lr'])
def test_gpu_graphed_step_follows_an_in_place_prior(lr):
    """Replays of a captured step with a per-weight prior equal eager steps, including after posterior_to_prior()
    refreshed the prior in place between replays."""
    dims, D, B, S = (16, 64, 64), 2, 128, 3
    x, y = _data(B, dims[0], D, seed=3)
    x, y = x.cuda(), y.cuda()
    seed, step0, warm = 77, 10, 2

    def run(graphed):
        net = _make_net(dims, D, 'cuda', lr=lr, tf32=True).train()
        _random_prior(net)
        opt = bnn_b200.FusedAdam(net.parameters(), lr=1e-3)
        losses = []
        if graphed:
            bnn_b200.manual_seed(seed, step0)
            gs = bnn_b200.GraphedTrainStep(net, opt, x, y, S, beta=0.1, warmup=warm)
            step = lambda: float(gs(x, y)[0].detach())
        else:
            bnn_b200.manual_seed(seed, step0 + warm)

            def step():
                net.zero_grad()
                info = (net.sample_elbo_lr if lr else net.sample_elbo)(x, y, 0.1, S)
                info[0].backward()
                opt.step()
                return float(info[0].detach())
        for k in range(5):
            if k == 3:
                net.posterior_to_prior()
            losses.append(step())
        return losses, [p.detach().clone() for p in net.parameters()]

    (lg, pg), (le, pe) = run(True), run(False)
    np.testing.assert_allclose(lg, le, rtol=1e-5)
    for p, q in zip(pg, pe):
        assert torch.allclose(p, q, rtol=1e-4, atol=2e-6), float((p - q).abs().max())


@pytest.mark.gpu
def test_gpu_row_sharded_step_equals_full_batch():
    from bnn_b200 import parallel
    dims, D, B, S = (16, 64, 64), 2, 128, 3
    x, y = _data(B, dims[0], D, seed=6)
    x, y = x.cuda(), y.cuda()
    net = _make_net(dims, D, 'cuda').train()
    _random_prior(net)
    bnn_b200.manual_seed(11, 3)
    net.zero_grad()
    full = net.sample_elbo(x, y, 0.2, S)
    full[0].backward()
    want = [p.grad.clone() for p in net.parameters()]
    acc, loss = [torch.zeros_like(p) for p in net.parameters()], 0.0
    for r in range(2):
        plan = parallel.ShardPlan(r, 2, S, B, row_shards=2)
        bnn_b200.manual_seed(11, 3)
        net.zero_grad()
        info = parallel.sharded_elbo(net, *plan.rows(x, y), 0.2, plan)
        info[0].backward()
        loss += float(info[0].detach()) / 2
        for a, p in zip(acc, net.parameters()):
            a += p.grad / 2
    assert abs(loss - float(full[0].detach())) <= 2e-5 * abs(float(full[0].detach()))
    for a, b in zip(acc, want):
        assert float((a - b).abs().max()) <= 2e-5 * float(b.abs().max())


# ---------------------------------------------------------------------------------------------------------------------
# GPU: sequential Bayesian updating of a conjugate model
# ---------------------------------------------------------------------------------------------------------------------
K, NOISE, S0, BIAS_S = 8, 0.5, 1.0, 1e-3


def _onehot_data(n_per, theta, seed):
    g = torch.Generator().manual_seed(seed)
    k = torch.arange(K).repeat(n_per)
    x = torch.nn.functional.one_hot(k, K).float()
    y = theta[k] + NOISE * torch.randn(k.shape, generator=g)
    return x, y.view(-1, 1), k


def _train(net, x, y, steps=3000):
    """Full-batch ELBO (beta = 1: the whole data set is the batch, whose NLL sample_elbo_lr sums), Adam with a
    learning rate decaying from 1e-2 to 1e-4."""
    opt = torch.optim.Adam(net.parameters(), lr=1e-2)
    sched = torch.optim.lr_scheduler.LambdaLR(opt, lambda i: 0.01 ** (i / steps))
    net.train()
    for _ in range(steps):
        opt.zero_grad()
        net.sample_elbo_lr(x, y, 1.0, 8, NOISE)[0].backward()
        opt.step()
        sched.step()
    w_mu = net.l1.weight_mu.detach().cpu().double().view(-1)
    w_sg = torch.log1p(torch.exp(net.l1.weight_rho.detach().cpu().double())).view(-1)
    return w_mu, w_sg


def _conjugate(ys, ks):
    """The exact posterior of w_k under N(0, S0^2) and N(y; w_k, NOISE^2) (the bias pinned at 0)."""
    prec = torch.full((K,), 1 / S0 ** 2, dtype=torch.float64)
    lin = torch.zeros(K, dtype=torch.float64)
    for y, k in zip(ys, ks):
        prec += torch.bincount(k, minlength=K).double() / NOISE ** 2
        lin += torch.zeros(K, dtype=torch.float64).index_add_(0, k, y.view(-1).double()) / NOISE ** 2
    return lin / prec, prec.rsqrt()


@pytest.mark.gpu
def test_gpu_sequential_update_matches_the_batch_posterior():
    """One Bayesian linear layer on one-hot inputs (hidden_units=[], 8 inputs) with a Gaussian likelihood: its exact
    posterior factorises, so the mean-field family contains it.  The bias is pinned by a N(0, 1e-3) prior.  Trained on
    D1, then posterior_to_prior(), then trained on D2, the weights match the conjugate posterior of D1 u D2: every mean
    within 0.1 sigma and every sigma within 5 %.  Trained on D2 under the original prior instead (the control), they
    miss it: some sigma is off by more than 25 % (the D2-only posterior is sqrt(2) wider).  Measured on a B200: the
    sequential update 0.027 sigma and 1.1 %, the control 3.1 sigma and 42 %."""
    torch.manual_seed(0)
    theta = torch.randn(K)
    x1, y1, k1 = _onehot_data(16, theta, 1)
    x2, y2, k2 = _onehot_data(16, theta + 0.3, 2)
    mp = dict(input_shape=K, classes=1, batch_size=128, hidden_units=[], mode='regression', mu_init=[-0.2, 0.2],
              rho_init=[-5, -4], prior_init=[S0], mixture_prior=False, local_reparam=True)
    prior0 = [(0.0, S0, 0.0, BIAS_S)]

    def fresh():
        torch.manual_seed(1)
        net = bnn_b200.BayesianNetwork(mp).cuda()
        net.set_prior(prior0)
        bnn_b200.manual_seed(5)
        return net

    net = fresh()
    _train(net, x1.cuda(), y1.cuda())
    net.posterior_to_prior()
    mu, sg = _train(net, x2.cuda(), y2.cuda())
    want_mu, want_sg = _conjugate([y1, y2], [k1, k2])
    mean_err = float(((mu - want_mu) / want_sg).abs().max())
    sigma_err = float((sg / want_sg - 1).abs().max())
    print(f'sequential: max |mean error| / sigma = {mean_err:.4f}, max |sigma error| = {sigma_err:.4f}')
    assert mean_err <= 0.1 and sigma_err <= 0.05, (mean_err, sigma_err)
    ctl = fresh()
    cmu, csg = _train(ctl, x2.cuda(), y2.cuda())
    ctl_mean = float(((cmu - want_mu) / want_sg).abs().max())
    ctl_sigma = float((csg / want_sg - 1).abs().max())
    print(f'control: max |mean error| / sigma = {ctl_mean:.4f}, max |sigma error| = {ctl_sigma:.4f}')
    assert ctl_sigma > 0.25, (ctl_mean, ctl_sigma)
