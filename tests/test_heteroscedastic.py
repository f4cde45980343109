"""Heteroscedastic regression: a learned per-input noise sigma(x) = sigma_min + softplus(r) trained through the ELBO
(bbb_nll_gauss_het) and its posterior predictive split into epistemic and aleatoric variance (bbb_predictive_stats kind
BBB_NLL_GAUSS_HET), from the C ABI up to BayesianNetwork.

The float64 restatement below (het_*) is the reference the kernels and the host are held to; it is itself checked
against float64 torch autograd.  CPU: the oracle, the host's routing and result assembly on the CPU double of the C ABI
(extended here by the two new entry points), the model's parameter layout and every argument error, and the real
library's argument checks (they return before anything touches a device).  GPU: the kernels against the oracle,
whole train steps against float64 autograd, graph replay and row sharding, the predictive, and a fit that learns
sigma(x)."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

import bnn_b200
from bnn_b200 import functional as F
from oracle import bbb_oracle as O
from tests import fake_bbb
from tests.golden_util import PNAMES

EINVAL = -1
NAN = float('nan')
HALF_LOG_2PI = 0.5 * math.log(2 * math.pi)
MU_INIT, RHO_INIT = [-0.2, 0.2], [-5, -4]


# ---------------------------------------------------------------------------------------------------------------------
# float64 oracle: out [.., 2D] = [f | r], sigma = sigma_min + softplus(r)
# ---------------------------------------------------------------------------------------------------------------------
def het_sigma(r, sigma_min):
    r = torch.as_tensor(r).double()
    return sigma_min + torch.clamp(r, min=0) + torch.log1p(torch.exp(-r.abs()))


def het_nll(out, y, sigma_min):
    """sum over (s, b, d) of (y - f)^2 / (2 sigma^2) + log sigma + log(2 pi) / 2; y [B,D] against out [S,B,2D]"""
    z = torch.as_tensor(out).double()
    D = z.shape[-1] // 2
    f, s = z[..., :D], het_sigma(z[..., D:], sigma_min)
    a = (torch.as_tensor(y).double() - f) / s
    return (0.5 * a * a + torch.log(s) + HALF_LOG_2PI).sum()


def het_nll_grad(out, y, sigma_min, g=1.0):
    """closed-form g d nll / d out: g (f - y) / sigma^2 and g sigmoid(r) (1/sigma - (y - f)^2 / sigma^3)"""
    z = torch.as_tensor(out).double()
    D = z.shape[-1] // 2
    f, r = z[..., :D], z[..., D:]
    s = het_sigma(r, sigma_min)
    a = (torch.as_tensor(y).double() - f) / s
    return torch.cat([-g * a / s, g * torch.sigmoid(r) / s * (1 - a * a)], -1)


def het_predictive(out, y=None, sigma_min=1e-3):
    """the mixture (1/S) sum_s N(f_s, sigma_s^2) per row: mean, variance (epistemic), aleatoric, total (the mixture's
    own second moment minus the squared mean), with y: log_pred = log (1/S) sum_s prod_d N(y_d; f_s,d, sigma_s,d^2) and
    sq_err = sum_d (mean_d - y_d)^2"""
    z = torch.as_tensor(out).double()
    S, B, C2 = z.shape
    D = C2 // 2
    f, s = z[..., :D], het_sigma(z[..., D:], sigma_min)
    mean = f.mean(0)
    r = dict(mean=mean, variance=f.var(0, unbiased=False), aleatoric=(s * s).mean(0),
             total=(f * f + s * s).mean(0) - mean * mean)
    if y is not None:
        yy = torch.as_tensor(y).double().reshape(B, D)
        ll = torch.distributions.Normal(f, s).log_prob(yy).sum(-1)           # [S,B]
        r.update(log_pred=torch.logsumexp(ll, 0) - math.log(S), sq_err=((mean - yy) ** 2).sum(-1))
    return r


def het_metrics(out, y, sigma_min):
    r = het_predictive(out, y, sigma_min)
    n, D = r['mean'].shape
    return dict(n=n, nll=float(-r['log_pred'].mean()), rmse=math.sqrt(float(r['sq_err'].sum()) / (n * D)))


# ---------------------------------------------------------------------------------------------------------------------
# CPU double of the two new entry points
# ---------------------------------------------------------------------------------------------------------------------
class HetFake(fake_bbb.FakeLib):
    """The CPU double plus bbb_nll_gauss_het and bbb_predictive_stats kind BBB_NLL_GAUSS_HET, evaluated with the oracle
    above (argument checks as bbb.h).  bbb_elbo_finalize calls are counted apart from `calls`, so the call lists of the
    existing likelihoods read as the base double records them."""
    finalized = 0

    def bbb_nll_gauss_het(self, out, target, sigma_min, S, B, D, scale, nll, dout, st):
        if not (out and target and nll) or min(S, B, D) < 0 or (D == 0 and S * B > 0) or not sigma_min > 0:
            return EINVAL
        self.calls.append('nll_gauss_het')
        if S * B * D == 0:
            return 0
        Z = fake_bbb._f(out, S, B, 2 * D)
        T = fake_bbb._f(target, B, D)
        fake_bbb._d(nll, 1)[0] += float(het_nll(Z, T, sigma_min))
        if dout:
            fake_bbb._f(dout, S, B, 2 * D)[...] = (scale * het_nll_grad(Z, T, sigma_min)).numpy().astype(np.float32)
        return 0

    def bbb_predictive_stats(self, out, target, S, B, Cc, kind, sigma, n_bins, mean, row_stats, pred, acc, st):
        assert kind == 3, 'HetFake: the heteroscedastic predictive only'
        if (S < 1 or B < 0 or not 2 <= Cc <= 1024 or Cc % 2 or not sigma > 0 or (target and not acc)
                or (B and not (out and mean and row_stats))):
            return EINVAL
        if B == 0:
            return 0
        self.calls.append('predictive_stats')
        D = Cc // 2
        T = fake_bbb._f(target, B, D) if target else None
        r = het_predictive(fake_bbb._f(out, S, B, Cc), T, sigma)
        fake_bbb._f(mean, B, D)[...] = r['mean'].numpy()
        RS = fake_bbb._f(row_stats, B, Cc + 1)
        RS[:, :D], RS[:, D:Cc] = r['variance'].numpy(), r['aleatoric'].numpy()
        RS[:, Cc] = r['log_pred'].numpy() if T is not None else NAN
        if T is not None:
            A = fake_bbb._d(acc, 4)
            A[0] += B
            A[2] -= r['log_pred'].sum().item()
            A[3] += r['sq_err'].sum().item()
        return 0

    def bbb_elbo_finalize(self, *a):
        HetFake.finalized += 1
        return super().bbb_elbo_finalize(*a)


@pytest.fixture
def fake(monkeypatch):
    lib = HetFake()
    fake_bbb.FakeLib.calls = []
    HetFake.finalized = 0
    monkeypatch.setattr(bnn_b200._lib, 'lib', lambda: lib)
    monkeypatch.setattr(bnn_b200._lib, 'require_cuda', lambda *a: None)
    monkeypatch.setattr(bnn_b200._lib, 'stream', lambda: None)
    return lib


# ---------------------------------------------------------------------------------------------------------------------
# shared helpers
# ---------------------------------------------------------------------------------------------------------------------
def _model_params(dims, D, likelihood='heteroscedastic', lr=False, **extra):
    mp = dict(input_shape=dims[0], classes=D, batch_size=128, hidden_units=list(dims[1:]), mode='regression',
              mu_init=MU_INIT, rho_init=RHO_INIT, prior_init=[1.0] if lr else [0.5, 0, -6], mixture_prior=not lr,
              local_reparam=lr, likelihood=likelihood)
    mp.update(extra)
    return mp


def _make_net(dims, D, device, seed=0, **kw):
    torch.manual_seed(seed)
    return bnn_b200.BayesianNetwork(_model_params(dims, D, **kw)).to(device)


def _data(B, n_in, D, seed=1):
    """x ~ U[-1, 1]; targets a smooth function of x plus noise, y = sin(3 x V) + 0.1 eps, as a regression target is.
    (With targets independent of x the first layer's weight gradient is a sum of terms of random sign, and its
    cancellation amplifies TF32's relative rounding beyond the stated bound: 8.8e-3 measured at 4 layers, batch 640.)"""
    g = torch.Generator().manual_seed(seed)
    x = 2 * torch.rand(B, n_in, generator=g) - 1
    v = torch.randn(n_in, D, generator=g) / math.sqrt(n_in)
    return x, torch.sin(3 * x @ v) + 0.1 * torch.randn(B, D, generator=g)


def _maxnorm_err(got, want):
    g, w = torch.as_tensor(got).double().cpu(), torch.as_tensor(want).double().cpu()
    return float((g - w).abs().max()) / max(float(w.abs().max()), 1e-300)


def _oracle_step(net, x, y, S, beta, eps, lr):
    """The float64 oracle of sample_elbo[_lr] with the net's parameters and the given draws: the returned tuple and
    the gradients (autograd of the oracle layers plus het_nll)."""
    layers = [tuple(t.detach().cpu().double().requires_grad_() for t in l.params()) for l in net.layers()]
    x64 = x.detach().cpu().double()
    y64 = y.detach().cpu().double().reshape(x64.shape[0], net.classes)
    nll = torch.zeros((), dtype=torch.float64)
    terms = []
    for s in range(S):
        e = [tuple(t.double() for t in pair) for pair in eps[s]]
        if lr:
            out, kl = O.mlp_forward_lr(x64, layers, float(net.prior_init[0]), e, 'regression')
            terms.append(kl)
        else:
            out, lp, lq = O.mlp_forward(x64, layers, O.make_prior(net.prior_init, net.mixture_prior), e, 'regression')
            terms.append((lp, lq))
        nll = nll + het_nll(out, y64, net.sigma_min)
    nll = nll / S
    if lr:
        kl = torch.stack(terms).mean()
        loss = beta * kl + nll
        scalars = (loss, kl, nll)
    else:
        lp = torch.stack([t[0] for t in terms]).mean()
        lq = torch.stack([t[1] for t in terms]).mean()
        loss = beta * lq - beta * lp + nll
        scalars = (loss, lp, lq, nll)
    loss.backward()
    return [float(v.detach()) for v in scalars], [[t.grad for t in l] for l in layers]


def _net_step(net, x, y, S, beta, seed):
    net.train()
    net.zero_grad()
    with bnn_b200.eps_mode('reference'):
        torch.manual_seed(seed)
        info = (net.sample_elbo_lr if net.local_reparam else net.sample_elbo)(x, y, beta, S)
    info[0].backward()
    return [float(v.detach().reshape(-1)[0]) for v in info], [[p.grad for p in l.params()] for l in net.layers()]


def check_step_against_oracle(dims, D, B, S, device, lr=False, tf32=False, rtol=1e-5, rtol_gemm=None, y_flat=False,
                              seed=5):
    """sample_elbo[_lr] in the reference eps mode against float64 autograd of the oracle under the same draws.
    rtol bounds the log-prob / KL scalars, rtol_gemm everything downstream of a contraction."""
    rg = rtol if rtol_gemm is None else rtol_gemm
    net = _make_net(dims, D, device, lr=lr, tf32=tf32)
    x, y = _data(B, dims[0], D)
    y_in = y[:, 0] if y_flat else y
    with torch.random.fork_rng():
        torch.manual_seed(seed)
        eps = O.draw_eps(list(dims) + [2 * D], S, batch=B, local_reparam=lr)
    want_s, want_g = _oracle_step(net, x, y, S, 0.3, eps, lr)
    got_s, got_g = _net_step(net, x.to(device), y_in.to(device), S, 0.3, seed)
    assert len(got_s) == (3 if lr else 4)
    scale = sum(abs(v) for v in want_s[1:])          # the loss is a signed sum of the other scalars
    assert abs(got_s[0] - want_s[0]) <= rg * scale, ('loss', got_s[0], want_s[0])
    for k in range(1, len(want_s) - 1):
        assert abs(got_s[k] - want_s[k]) <= rtol * abs(want_s[k]), (k, got_s[k], want_s[k])
    assert abs(got_s[-1] - want_s[-1]) <= rg * abs(want_s[-1]), ('nll', got_s[-1], want_s[-1])
    worst = 0.0
    for li, (gl, wl) in enumerate(zip(got_g, want_g)):
        for pn, g, w in zip(PNAMES, gl, wl):
            assert bool(torch.isfinite(g).all()), (li, pn)
            err = _maxnorm_err(g, w)
            assert err <= rg, f'l{li + 1}.{pn}: max-norm relative error {err:.3e} > {rg:.1e}'
            worst = max(worst, err)
    return worst


# ---------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------
def _extreme_outputs(S, B, D, seed=0, res_scale=1.0):
    """[S,B,2D] outputs with r spanning [-40, 40] (both ends included) and targets with residuals up to res_scale"""
    g = torch.Generator().manual_seed(seed)
    f = torch.randn(S, B, D, generator=g)
    r = 80 * torch.rand(S, B, D, generator=g) - 40
    r.view(-1)[:4] = torch.tensor([-40.0, 40.0, 0.0, -40.0])
    y = res_scale * torch.randn(B, D, generator=g)
    return torch.cat([f, r], -1), y


@pytest.mark.parametrize('sigma_min,res', [(1e-3, 1.0), (1e-6, 1e3), (0.5, 10.0)])
def test_oracle_nll_and_gradient_equal_autograd(sigma_min, res):
    out, y = _extreme_outputs(3, 7, 2, res_scale=res)
    z = out.double().requires_grad_()
    D = 2
    s = sigma_min + torch.nn.functional.softplus(z[..., D:], threshold=1000.0)
    auto = -torch.distributions.Normal(z[..., :D], s).log_prob(y.double()).sum()
    (grad,) = torch.autograd.grad(auto, z)
    nll = het_nll(out, y, sigma_min)
    assert abs(float(nll) - float(auto.detach())) <= 1e-12 * abs(float(auto.detach()))
    mine = het_nll_grad(out, y, sigma_min)
    assert bool(torch.isfinite(mine).all())
    for half in (slice(0, D), slice(D, 2 * D)):
        assert _maxnorm_err(mine[..., half], grad[..., half]) <= 1e-12


def test_oracle_mixture_variance_is_epistemic_plus_aleatoric():
    out, y = _extreme_outputs(6, 9, 3, seed=2)
    out[..., 3:] = out[..., 3:] / 10
    r = het_predictive(out, y, 1e-2)
    assert torch.allclose(r['variance'] + r['aleatoric'], r['total'], rtol=1e-10, atol=1e-12)


def _routing(device_lib, dims, D, tf32, likelihood, lr=False):
    fake_bbb.FakeLib.calls = []
    HetFake.finalized = 0
    net = _make_net(dims, D, 'cpu', lr=lr, tf32=tf32, likelihood=likelihood)
    x, y = _data(16, dims[0], D)
    with bnn_b200.eps_mode('reference'):
        info = (net.sample_elbo_lr if lr else net.sample_elbo)(x, y, 0.5, 2)
    fwd = list(device_lib.calls)
    info[0].backward()
    return fwd, device_lib.calls[len(fwd):], HetFake.finalized, info


@pytest.mark.parametrize('tf32', [False, True])
def test_heteroscedastic_step_takes_the_per_layer_calls(fake, tf32):
    """A heteroscedastic sample_elbo runs every layer as a plain layer call, then bbb_nll_gauss_het and
    bbb_elbo_finalize, and the per-layer backward; neither the fused head nor the network-level call (which this
    Gaussian net takes in TF32 mode) appears.  The Gaussian net's call lists are what they were."""
    dims = (8, 16, 16)
    fwd, bwd, fin, info = _routing(fake, dims, 1, tf32, 'heteroscedastic')
    assert fwd == ['linear_fwd'] * 3 + ['nll_gauss_het'] and fin == 1
    assert bwd == ['linear_bwd'] * 3
    assert len(info) == 4
    fwd, bwd, _, _ = _routing(fake, dims, 1, tf32, 'gaussian')
    if tf32:
        assert fwd == ['mlp_fwd', 'head_fwd'] and bwd == ['mlp_bwd']
    else:
        assert fwd == ['linear_fwd'] * 2 + ['head_fwd'] and bwd == ['linear_bwd'] * 3


def test_heteroscedastic_lr_step_routing(fake):
    fwd, bwd, fin, info = _routing(fake, (8, 16, 16), 2, False, 'heteroscedastic', lr=True)
    assert fwd == ['lr_fwd'] * 3 + ['nll_gauss_het'] and fin == 1 and bwd == ['lr_bwd'] * 3
    assert len(info) == 3
    fwd, _, _, _ = _routing(fake, (8, 16, 16), 2, False, 'gaussian', lr=True)
    assert fwd == ['lr_fwd'] * 3 + ['nll_gauss']


@pytest.mark.parametrize('lr', [False, True])
def test_step_on_the_double_matches_the_oracle(fake, lr):
    """The host's plumbing (eps order, target layout, scaling of the likelihood gradient, tuple assembly) on the
    float64 double against the oracle; a [B] target with D = 1 is taken row for row."""
    check_step_against_oracle((3, 16, 16), 1, 12, 3, 'cpu', lr=lr, y_flat=True)
    check_step_against_oracle((3, 16, 16), 2, 12, 2, 'cpu', lr=lr)


def test_non_contiguous_target(fake):
    """A strided [B] target (D = 1) is copied to a contiguous buffer that outlives the likelihood call."""
    x, y = _data(12, 3, 2)
    res = []
    for tgt in (y[:, 0], y[:, 0].contiguous()):
        assert tgt.is_contiguous() == (len(res) == 1)
        res.append(_net_step(_make_net((3, 8, 8), 1, 'cpu'), x, tgt, 2, 0.4, 9))
    assert res[0][0] == res[1][0]


@pytest.mark.parametrize('lr', [False, True])
def test_fused_equals_unfused_on_the_double(fake, lr):
    """fused=False runs BayesianNetwork.get_nll in torch: the same numbers as bbb_nll_gauss_het's double."""
    x, y = _data(10, 3, 2)
    res = []
    for fused in (True, False):
        net = _make_net((3, 8, 8), 2, 'cpu', lr=lr, fused=fused)
        res.append(_net_step(net, x, y, 2, 0.4, 9))
    (sa, ga), (sb, gb) = res
    np.testing.assert_allclose(sa, sb, rtol=1e-6)
    for la, lb in zip(ga, gb):
        for a, b in zip(la, lb):
            assert _maxnorm_err(a, b) <= 1e-5


@pytest.mark.parametrize('lr', [False, True])
def test_parameter_shapes_and_state_dict(lr):
    net = bnn_b200.BayesianNetwork(_model_params((3, 16, 16), 2, lr=lr))
    assert net.likelihood == 'heteroscedastic' and net.sigma_min == 1e-3 and net.classes == 2
    want = (16, 4) if lr else (4, 16)
    assert tuple(net.l3.weight_mu.shape) == want and tuple(net.l3.bias_rho.shape) == (4,)
    assert list(net.state_dict().keys()) == [f'l{i + 1}.{pn}' for i in range(3) for pn in PNAMES]
    g = bnn_b200.BayesianNetwork(_model_params((3, 16, 16), 2, likelihood='gaussian', lr=lr))
    assert g.likelihood == 'gaussian' and tuple(g.l3.bias_mu.shape) == (2,)
    assert bnn_b200.BayesianNetwork(_model_params((3, 16, 16), 1, sigma_min=0.05)).sigma_min == 0.05


def test_value_errors(fake):
    with pytest.raises(ValueError, match='regression'):
        bnn_b200.BayesianNetwork(_model_params((3, 8), 2, mode='classification'))
    for bad in (0.0, -1e-3):
        with pytest.raises(ValueError, match='sigma_min'):
            bnn_b200.BayesianNetwork(_model_params((3, 8), 2, sigma_min=bad))
    with pytest.raises(ValueError, match='likelihood'):
        bnn_b200.BayesianNetwork(_model_params((3, 8), 2, likelihood='student'))
    x, y = _data(6, 3, 2)
    for lr in (False, True):
        net = _make_net((3, 8), 2, 'cpu', lr=lr)
        elbo = net.sample_elbo_lr if lr else net.sample_elbo
        with bnn_b200.eps_mode('reference'):
            for sigma in (0.5, torch.tensor(1.0)):
                with pytest.raises(ValueError, match='learns sigma'):
                    elbo(x, y, 1.0, 2, sigma=sigma)
                with pytest.raises(ValueError, match='learns sigma'):
                    elbo(x, y, 1.0, 2, sigma)
            for bad_y in (y[:, 0], y[:3], y[:1].expand(6, 2).contiguous()[:, :1], torch.zeros(6, 3), y[None]):
                with pytest.raises(ValueError, match='heteroscedastic target'):
                    elbo(x, bad_y, 1.0, 2)
        with pytest.raises(ValueError, match='learns sigma'):
            net.predictive(x, 2, target=y, sigma=0.3)
        with pytest.raises(ValueError, match='heteroscedastic target'):
            net.get_nll(torch.zeros(6, 4), y[:, 0])
    net1 = _make_net((3, 8), 1, 'cpu')
    with bnn_b200.eps_mode('reference'):
        net1.sample_elbo(x, y[:, 0], 1.0, 2)                    # D = 1: [B] and [B, 1] targets are accepted
        net1.sample_elbo(x, y[:, :1], 1.0, 2)
        with pytest.raises(ValueError, match='heteroscedastic target'):
            net1.sample_elbo(x, y[:1, 0], 1.0, 2)                # no broadcast of a single row
    with pytest.raises(ValueError, match='even width'):
        F.predictive_stats(torch.zeros(2, 3, 5), mode='heteroscedastic')


@pytest.mark.parametrize('lr', [False, True])
def test_predictive_result_on_the_double(fake, lr):
    """BayesianNetwork.predictive of a heteroscedastic net: variance is the epistemic part, aleatoric_variance the
    mean sigma(x)^2, both against the oracle applied to sample_predict's outputs under the same draws."""
    net = _make_net((3, 16, 16), 2, 'cpu', lr=lr, sigma_min=0.01).eval()
    with torch.no_grad():
        net.l3.bias_mu[2:] = torch.tensor([-1.0, 0.5])
    x, y = _data(9, 3, 2, seed=4)
    with bnn_b200.eps_mode('reference'):
        torch.manual_seed(3)
        outs = net.sample_predict(x, 4)
        torch.manual_seed(3)
        res = net.predictive(x, 4, target=y)
    assert tuple(outs.shape) == (4, 9, 4)
    want = het_predictive(outs, y, 0.01)
    for k, v in (('mean', res.mean), ('variance', res.variance), ('aleatoric', res.aleatoric_variance),
                 ('log_pred', res.log_pred)):
        np.testing.assert_allclose(v.double().numpy(), want[k].numpy(), rtol=1e-5, atol=1e-7, err_msg=k)
    m, wm = res.metrics(), het_metrics(outs, y, 0.01)
    assert m['n'] == 9 and m['nll'] == pytest.approx(wm['nll'], rel=1e-6) and m['rmse'] == pytest.approx(wm['rmse'])
    assert res.pred is None and res.entropy is None
    g = _make_net((3, 16, 16), 2, 'cpu', likelihood='gaussian')
    assert bnn_b200.PredictiveResult(torch.zeros(1, 2)).aleatoric_variance is None
    assert g.likelihood == 'gaussian'


def test_abi_rejects_bad_arguments():
    """The real library's argument checks (they return before any device work, so they run without a GPU)."""
    lib = bnn_b200._lib.lib()
    buf = C.c_void_p(16)            # never dereferenced: every call below is refused first
    ok = dict(out=buf, target=buf, sigma_min=1e-3, S=2, B=4, D=3, nll=buf)
    bad = [dict(sigma_min=0.0), dict(sigma_min=-1.0), dict(sigma_min=NAN), dict(out=None), dict(target=None),
           dict(nll=None), dict(S=-1), dict(B=-1), dict(D=-1), dict(D=0)]
    for change in bad:
        a = dict(ok, **change)
        st = lib.bbb_nll_gauss_het(a['out'], a['target'], a['sigma_min'], a['S'], a['B'], a['D'], 1.0, a['nll'], None,
                                   None)
        assert st == EINVAL, change
    # an empty call launches nothing
    assert lib.bbb_nll_gauss_het(buf, buf, 1e-3, 0, 4, 3, 1.0, buf, None, None) == 0
    assert lib.bbb_nll_gauss_het(buf, buf, 1e-3, 2, 0, 0, 1.0, buf, None, None) == 0
    # predictive kind BBB_NLL_GAUSS_HET: C = 2D even, sigma_min > 0
    okp = dict(out=buf, target=None, S=2, B=4, C=4, sigma=1e-3, mean=buf, rs=buf, acc=None)
    for change in (dict(C=3), dict(C=1), dict(C=0), dict(C=1026), dict(S=0), dict(B=-1), dict(sigma=0.0),
                   dict(target=buf), dict(out=None), dict(mean=None), dict(rs=None)):
        a = dict(okp, **change)
        st = lib.bbb_predictive_stats(a['out'], a['target'], a['S'], a['B'], a['C'], 3, a['sigma'], 0, a['mean'],
                                      a['rs'], None, a['acc'], None)
        assert st == EINVAL, change
    assert lib.bbb_predictive_stats(None, None, 2, 0, 4, 3, 1e-3, 0, None, None, None, None, None) == 0
    # the fused head does not implement the heteroscedastic likelihood
    st = lib.bbb_head_fwd(buf, 0, buf, buf, buf, buf, None, None, None, None, 2, 4, 8, 2, 0, 3, buf, 1.0, 1.0, buf,
                          None, None, None, buf, 1.0, None, None, None, None)
    assert st == EINVAL


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
def _kernel_call(out, y, sigma_min, grad_scale=0.25):
    S, B, C2 = out.shape
    nll = torch.zeros(1, dtype=torch.float64, device='cuda')
    dout = torch.full_like(out, NAN)
    bnn_b200._lib.check(bnn_b200._lib.lib().bbb_nll_gauss_het(out.data_ptr(), y.data_ptr(), sigma_min, S, B, C2 // 2,
                                                               grad_scale, nll.data_ptr(), dout.data_ptr(),
                                                               torch.cuda.current_stream().cuda_stream),
                        'bbb_nll_gauss_het')
    return float(nll), dout


@pytest.mark.gpu
@pytest.mark.parametrize('sigma_min,res,D', [(1e-3, 1.0, 1), (1e-3, 1.0, 3), (1e-6, 1e3, 2), (0.5, 10.0, 5)])
def test_gpu_nll_kernel_matches_the_oracle(sigma_min, res, D):
    """bbb_nll_gauss_het against the float64 oracle: nll to 1e-6 relative, each half of dout to 1e-5 of its max-norm,
    every output finite, for r in [-40, 40], sigma_min down to 1e-6 and residuals up to 1e3."""
    out, y = _extreme_outputs(3, 257, D, seed=D, res_scale=res)
    nll, dout = _kernel_call(out.cuda(), y.cuda(), sigma_min)
    sm = float(np.float32(sigma_min))
    want = float(het_nll(out, y, sm))
    assert math.isfinite(nll) and abs(nll - want) <= 1e-6 * abs(want), (nll, want)
    gw = het_nll_grad(out, y, sm, 0.25)
    dout = dout.cpu()
    assert bool(torch.isfinite(dout).all())
    for half in (slice(0, D), slice(D, 2 * D)):
        assert _maxnorm_err(dout[..., half], gw[..., half]) <= 1e-5


@pytest.mark.gpu
def test_gpu_nll_kernel_moderate_range_elementwise():
    """Ordinary values: every element of dout within 1e-5 relative of the oracle (not only the max-norm)."""
    g = torch.Generator().manual_seed(7)
    out = torch.cat([torch.randn(5, 128, 1, generator=g), 3 * torch.randn(5, 128, 1, generator=g)], -1)
    y = torch.randn(128, 1, generator=g)
    nll, dout = _kernel_call(out.cuda(), y.cuda(), 1e-3, 1.0 / 5)
    want = het_nll_grad(out, y, float(np.float32(1e-3)), 0.2)
    np.testing.assert_allclose(dout.cpu().double().numpy(), want.numpy(), rtol=1e-5, atol=1e-7)
    assert nll == pytest.approx(float(het_nll(out, y, float(np.float32(1e-3)))), rel=1e-6)


CFG1 = ((1, 400, 400), 1, 128, 5)          # 1-400-400-2, B = 128, S = 5
DEEP = ((16, 256, 256, 256), 2, 640, 3)    # 4 layers, batch 640: the large-batch kernel families


@pytest.mark.gpu
@pytest.mark.parametrize('cfg', [CFG1, DEEP], ids=['cfg1', 'deep4_b640'])
@pytest.mark.parametrize('lr', [False, True], ids=['ws', 'lr'])
@pytest.mark.parametrize('tf32', [False, True], ids=['fp32', 'tf32'])
def test_gpu_step_matches_float64_autograd(cfg, lr, tf32):
    """Whole train step in the reference eps mode against float64 autograd of the oracle layers + het_nll: the
    returned tuple and every gradient.  fp32 <= 1e-5; TF32 at the bounds of DESIGN §2 (5e-3, local
    reparameterisation 2e-2), except weight sampling on the 4-layer batch-640 net: its first layer's weight gradient
    (16 inputs, a sum over 1 920 rows of the TF32 backward) measured 5.1e-3 of its max-norm on a B200, so that case is
    held to 1e-2 (DESIGN §4.4c)."""
    dims, D, B, S = cfg
    rg = (2e-2 if lr else (1e-2 if cfg is DEEP else 5e-3)) if tf32 else 1e-5
    check_step_against_oracle(dims, D, B, S, 'cuda', lr=lr, tf32=tf32, rtol=1e-5, rtol_gemm=rg, y_flat=(D == 1))


@pytest.mark.gpu
@pytest.mark.parametrize('lr', [False, True])
def test_gpu_fused_equals_unfused(lr):
    """The kernels' likelihood (bbb_nll_gauss_het) and the torch get_nll of fused=False, same eps, fp32."""
    dims, D, B, S = CFG1
    x, y = _data(B, dims[0], D)
    res = []
    for fused in (True, False):
        net = _make_net(dims, D, 'cuda', lr=lr, fused=fused)
        res.append(_net_step(net, x.cuda(), y.cuda(), S, 0.3, 4))
    (sa, ga), (sb, gb) = res
    np.testing.assert_allclose(sa, sb, rtol=1e-5)
    for la, lb in zip(ga, gb):
        for a, b in zip(la, lb):
            assert _maxnorm_err(a, b) <= 1e-5


@pytest.mark.gpu
def test_gpu_graphed_step_equals_eager_steps():
    """3 replays of the captured heteroscedastic step (FusedAdam) == 3 eager steps at the same Philox coordinates."""
    dims, D, B, S = CFG1
    x, y = _data(B, dims[0], D, seed=3)
    x, y = x.cuda(), y.cuda()
    seed, step0, warm = 77, 10, 2
    net_g = _make_net(dims, D, 'cuda').train()
    opt_g = bnn_b200.FusedAdam(net_g.parameters(), lr=1e-3)
    bnn_b200.manual_seed(seed, step0)
    before = [p.detach().clone() for p in net_g.parameters()]
    gs = bnn_b200.GraphedTrainStep(net_g, opt_g, x, y, S, beta=0.1, warmup=warm)
    for p, b in zip(net_g.parameters(), before):
        assert torch.equal(p, b)
    losses_g = [float(gs(x, y)[0].detach()) for _ in range(3)]
    net_e = _make_net(dims, D, 'cuda').train()
    opt_e = bnn_b200.FusedAdam(net_e.parameters(), lr=1e-3)
    bnn_b200.manual_seed(seed, step0 + warm)
    losses_e = []
    for _ in range(3):
        net_e.zero_grad()
        info = net_e.sample_elbo(x, y, 0.1, S)
        info[0].backward()
        opt_e.step()
        losses_e.append(float(info[0].detach()))
    np.testing.assert_allclose(losses_g, losses_e, rtol=1e-5)
    for p, q in zip(net_g.parameters(), net_e.parameters()):
        assert torch.allclose(p, q, rtol=1e-4, atol=2e-6), float((p - q).abs().max())
    assert losses_g[0] != losses_g[1]


@pytest.mark.gpu
def test_gpu_row_sharded_step_equals_full_batch():
    """The likelihood is per row: two row shards (parallel.sharded_elbo) back to back with the same Philox stream,
    gradients averaged, equal the full batch."""
    from bnn_b200 import parallel
    dims, D, B, S = CFG1
    x, y = _data(B, dims[0], D, seed=6)
    x, y = x.cuda(), y.cuda()
    net = _make_net(dims, D, 'cuda').train()
    bnn_b200.manual_seed(11, 3)
    net.zero_grad()
    full = net.sample_elbo(x, y, 0.2, S)
    full[0].backward()
    want = [p.grad.clone() for p in net.parameters()]
    acc, loss, nll = [torch.zeros_like(p) for p in net.parameters()], 0.0, 0.0
    for r in range(2):
        plan = parallel.ShardPlan(r, 2, S, B, row_shards=2)
        bnn_b200.manual_seed(11, 3)
        net.zero_grad()
        info = parallel.sharded_elbo(net, *plan.rows(x, y), 0.2, plan)
        info[0].backward()
        loss += float(info[0].detach()) / 2
        nll += float(info[3].detach())
        for a, p in zip(acc, net.parameters()):
            a += p.grad / 2
    assert abs(loss - float(full[0].detach())) <= 2e-5 * abs(float(full[0].detach()))
    assert nll == pytest.approx(float(full[3].detach()), rel=2e-5)
    for a, b in zip(acc, want):
        assert float((a - b).abs().max()) <= 2e-5 * float(b.abs().max())


@pytest.mark.gpu
@pytest.mark.parametrize('D', [1, 3, 40])
def test_gpu_predictive_matches_the_oracle(D):
    """Kind BBB_NLL_GAUSS_HET against the oracle on the very outputs of sample_predict: mean, both variances,
    log_pred, metrics(), and epistemic + aleatoric = the mixture's variance."""
    dims = (4, 32, 32)
    net = _make_net(dims, D, 'cuda', sigma_min=0.02).eval()
    with torch.no_grad():
        net.l3.bias_mu[D:] = torch.linspace(-2, 1, D)
        for l in net.layers():
            l.weight_rho.fill_(-2.0)
    x, y = _data(300, dims[0], D, seed=8)
    x, y = x.cuda(), y.cuda()
    S = 6
    bnn_b200.manual_seed(5, step=12)
    with torch.no_grad():
        outs = net.sample_predict(x, S).cpu()
    bnn_b200.manual_seed(5, step=12)
    res = net.predictive(x, S, target=y if D > 1 else y[:, 0])
    want = het_predictive(outs, y.cpu(), float(np.float32(0.02)))
    for k, v in (('mean', res.mean), ('variance', res.variance), ('aleatoric', res.aleatoric_variance),
                 ('log_pred', res.log_pred)):
        np.testing.assert_allclose(v.cpu().double().numpy(), want[k].numpy(), rtol=1e-5, atol=1e-6, err_msg=k)
    total = (res.variance + res.aleatoric_variance).cpu().double()
    np.testing.assert_allclose(total.numpy(), want['total'].numpy(), rtol=1e-5, atol=1e-6)
    assert float(res.variance.min()) > 0
    m, wm = res.metrics(), het_metrics(outs, y.cpu(), float(np.float32(0.02)))
    assert m['n'] == 300
    assert m['nll'] == pytest.approx(wm['nll'], rel=1e-5, abs=1e-6)
    assert m['rmse'] == pytest.approx(wm['rmse'], rel=1e-5)
    # no target: the per-row statistics alone
    bnn_b200.manual_seed(5, step=12)
    res2 = net.predictive(x, S)
    assert res2.log_pred is None
    np.testing.assert_allclose(res2.aleatoric_variance.cpu().numpy(), res.aleatoric_variance.cpu().numpy(), rtol=1e-6)


@pytest.mark.gpu
def test_gpu_predictive_ignores_chunking():
    """Weight sampling: chunks of every row, 64 rows and 7 rows share one eps plan and give the same result."""
    dims, D = (4, 32, 32), 2
    net = _make_net(dims, D, 'cuda').eval()
    x, y = _data(500, dims[0], D, seed=9)
    x, y = x.cuda(), y.cuda()
    runs = []
    for rows in (None, 64, 7):
        bnn_b200.manual_seed(2, step=3)
        res = net.predictive(x, 5, target=y, chunk_rows=rows)
        runs.append(res)
    for r in runs[1:]:
        for k in ('mean', 'variance', 'aleatoric_variance', 'log_pred'):
            assert _maxnorm_err(getattr(r, k), getattr(runs[0], k)) <= 1e-5, k
        m, m0 = r.metrics(), runs[0].metrics()
        assert m['nll'] == pytest.approx(m0['nll'], rel=1e-5) and m['rmse'] == pytest.approx(m0['rmse'], rel=1e-5)


def _fit(likelihood, steps=2000, seed=0):
    """y = sin(3x) + (0.05 + 0.4 (x + 1) / 2) eps, x ~ U[-1, 1], N = 1024; 1-64-64-(2 or 1), FusedAdam, captured
    steps over shuffled minibatches of 128.  Returns the held-out predictive of the trained net."""
    torch.manual_seed(seed)
    N, B, S = 1024, 128, 4
    x = 2 * torch.rand(N, 1) - 1
    noise = 0.05 + 0.4 * (x + 1) / 2
    y = torch.sin(3 * x) + noise * torch.randn(N, 1)
    mp = dict(input_shape=1, classes=1, batch_size=B, hidden_units=64, mode='regression', mu_init=[-0.2, 0.2],
              rho_init=[-5, -4], prior_init=[0.5, 0, -6], mixture_prior=True, likelihood=likelihood)
    net = bnn_b200.BayesianNetwork(mp).cuda().train()
    opt = bnn_b200.FusedAdam(net.parameters(), lr=3e-3)
    xg, yg = x.cuda(), y.cuda()
    sigma = 1.0 if likelihood == 'heteroscedastic' else 0.25
    bnn_b200.manual_seed(seed + 1)
    gs = bnn_b200.GraphedTrainStep(net, opt, xg[:B], yg[:B], S, sigma=sigma, beta=B / N, warmup=2)
    order = torch.randperm(N, generator=torch.Generator().manual_seed(seed)).cuda()
    for k in range(steps):
        j = (k * B) % N
        if j == 0:
            order = order[torch.randperm(N, generator=torch.Generator().manual_seed(seed + k)).cuda()]
        idx = order[j:j + B]
        gs(xg[idx], yg[idx])
    torch.cuda.synchronize()
    xt = torch.linspace(-1, 1, 401).view(-1, 1)
    g = torch.Generator().manual_seed(seed + 99)
    nt = 0.05 + 0.4 * (xt + 1) / 2
    yt = torch.sin(3 * xt) + nt * torch.randn(xt.shape, generator=g)
    bnn_b200.manual_seed(seed + 2)
    net.eval()
    if likelihood == 'heteroscedastic':
        res = net.predictive(xt.cuda(), 32, target=yt.cuda())
    else:
        res = net.predictive(xt.cuda(), 32, target=yt.cuda(), sigma=sigma)
    return res, nt


@pytest.mark.gpu
def test_gpu_learns_the_noise_level():
    """Trained on data whose noise std grows from 0.05 to 0.45 across the input range, the net's aleatoric std
    follows it (Pearson r > 0.8) and its held-out NLL beats the same net with the fixed sigma = 0.25; the run is
    deterministic."""
    res, nt = _fit('heteroscedastic')
    std = res.aleatoric_variance.sqrt().cpu().double().view(-1)
    corr = float(np.corrcoef(std.numpy(), nt.double().view(-1).numpy())[0, 1])
    assert corr > 0.8, corr
    nll_het = res.metrics()['nll']
    res_h, _ = _fit('gaussian')
    nll_hom = res_h.metrics()['nll']
    assert nll_het < nll_hom, (nll_het, nll_hom)
    again, _ = _fit('heteroscedastic')
    assert torch.equal(again.mean, res.mean) and torch.equal(again.aleatoric_variance, res.aleatoric_variance)
