"""GPU tests of the tcgen05 kind::tf32 path (BBB_F_TF32).

Stated bound for this mode (BASELINE.json north_star: "a stated looser bound in TF32"): TF32 keeps 10
mantissa bits of each GEMM operand, so everything downstream of a contraction (outputs, NLL, loss, gradients)
is held to 5e-3 relative (max-norm per tensor); the log prior / log posterior sums do not pass through a
GEMM and stay at the fp32 bound of 1e-5."""
import numpy as np
import pytest
import torch

import bnn_b200
from tests import parity_cases as PC
from tests.golden_util import Case, SMALL, BIG, SMALL_LR, BIG_LR, DEEP_SMALL, DEEP_BIG

pytestmark = pytest.mark.gpu
DEV = 'cuda'
RTOL_TF32 = 5e-3


@pytest.mark.parametrize('B,d_in,d_out', [(128, 64, 64), (128, 1200, 1200), (7, 32, 16), (128, 784, 1200),
                                          (128, 1200, 10), (64, 100, 100), (130, 68, 83), (1, 400, 1), (300, 256, 80)])
def test_tcgen05_plain_gemm(B, d_in, d_out):
    """sample=False turns the layer into y = x mu^T + b: isolates descriptors, swizzle, TMEM, split-K."""
    torch.manual_seed(B + d_in)
    layer = bnn_b200.BayesianLinear(d_in, d_out, [-0.2, 0.2], [-5, -4], [1.0], False).to(DEV).eval()
    layer.tf32 = True
    x = torch.randn(B, d_in, device=DEV)
    with torch.no_grad():
        y = layer(x)
    ref = (x.double() @ layer.weight_mu.double().t() + layer.bias_mu.double())
    err = (y.double() - ref).abs().max() / ref.abs().max()
    assert err < 2e-3, float(err)


@pytest.mark.parametrize('name', SMALL + BIG + SMALL_LR + BIG_LR + DEEP_SMALL + DEEP_BIG)
@pytest.mark.parametrize('fused', [True, False])
def test_tf32_train_step_matches_reference(name, fused):
    c = Case(name)
    # LR at the MNIST shape: 1.0e-2 on l1.weight_mu.  Not the variance contraction (delta agrees with the fp32 path to
    # 8e-5) and not the backward kernels (<= 1.4e-3 on an identical forward state, test below): the TF32 forward moves
    # pre-activations by ~4e-4 of their range, which flips the ReLU mask of ~1e-4 of the hidden units, and one flipped
    # unit changes a 256-term batch sum by a whole term (tools/debug_lr_tf32.py; the weight-sampling estimator shows
    # the same under an adversarial d_out).  Stated bound for this estimator: 2e-2.
    PC.check_train_step(c, DEV, fused=fused, rtol=1e-5, rtol_gemm=2e-2 if c.lr else RTOL_TF32, tf32=True)


def test_lr_tf32_backward_kernels_alone_within_bound():
    """The LR estimator's tcgen05 backward kernels against its exact fp32 kernels on the SAME stored forward state (same
    y, delta, eps, hence identical ReLU masks): every gradient within the TF32 bound of 5e-3."""
    from bnn_b200 import functional as F, rng as R
    torch.manual_seed(0)
    dims, B, S = (784, 1200, 1200, 10), 128, 2
    params = [(torch.empty(i, o, device=DEV).uniform_(-0.2, 0.2), torch.empty(i, o, device=DEV).uniform_(-5, -4),
               torch.empty(o, device=DEV).uniform_(-0.2, 0.2), torch.empty(o, device=DEV).uniform_(-5, -4))
              for i, o in zip(dims[:-1], dims[1:])]
    x = torch.rand(B, dims[0], device=DEV)
    d_out = torch.randn(S, B, dims[-1], device=DEV) / B
    R.manual_seed(7, 0)
    est = F._LocalReparam(1.0)
    eps = F.plan_eps(est.eps_shapes(params, B), S, x.device, True)
    kl = torch.zeros(1, dtype=torch.float64, device=DEV)
    ys, deltas = F._forward(est, x, params, S, eps, True, True, True, (kl,))
    got = {}
    for tf32 in (False, True):
        _, grads = F._backward(est, x, [t.clone() for t in ys], [t.clone() for t in deltas], d_out.clone(), params, S,
                               eps, True, tf32, est.elbo_grad_args(0.1, None, S), None, False)
        got[tf32] = [[g.clone() for g in lg] for lg in grads]
    for la, lb in zip(got[True], got[False]):
        for a, b in zip(la, lb):
            assert float((a - b).abs().max()) <= RTOL_TF32 * float(b.abs().max())


@pytest.mark.parametrize('S', [1, 2, 3, 5])
def test_tf32_matches_fp32_path_in_philox_mode(S):
    """Same Philox coordinates through both kernel families: sample groups, tails and eps regeneration agree."""
    c = Case('cfg4_bandit')
    x = c.x.to(DEV)
    y = torch.randn(c.B, 1, device=DEV)
    res = []
    for tf32 in (False, True):
        net = PC.build_net(c, DEV, tf32=tf32).train()
        bnn_b200.manual_seed(5, 9)
        info = net.sample_elbo(x, y, c.beta, S)
        info[0].backward()
        res.append(([float(v.detach()) for v in info], PC.net_grads(net)))
    (i0, g0), (i1, g1) = res
    np.testing.assert_allclose(i1[1:3], i0[1:3], rtol=1e-5)          # log prior / log posterior: no GEMM involved
    np.testing.assert_allclose([i1[0], i1[3]], [i0[0], i0[3]], rtol=RTOL_TF32)
    for a, b in zip(g0, g1):
        for ga, gb in zip(a, b):
            assert np.abs(ga - gb).max() <= RTOL_TF32 * np.abs(ga).max()


def test_tf32_large_batch_tiles():
    """B > 128 exercises multiple M tiles (weights regenerated per tile, log-probs counted once)."""
    torch.manual_seed(3)
    mp = dict(input_shape=64, classes=10, batch_size=300, hidden_units=96, mode='classification',
              mu_init=[-0.2, 0.2], rho_init=[-5, -4], prior_init=[0.5, 0, -6], mixture_prior=True)
    x = torch.randn(300, 64, device=DEV)
    y = torch.randint(0, 10, (300,), device=DEV)
    res = []
    for tf32 in (False, True):
        torch.manual_seed(0)
        net = bnn_b200.BayesianNetwork(dict(mp, tf32=tf32)).to(DEV).train()
        bnn_b200.manual_seed(1, 1)
        info = net.sample_elbo(x, y, 0.3, 3)
        info[0].backward()
        res.append(([float(v.detach()) for v in info], PC.net_grads(net)))
    (i0, g0), (i1, g1) = res
    np.testing.assert_allclose(i1[1:3], i0[1:3], rtol=1e-5)
    np.testing.assert_allclose([i1[0], i1[3]], [i0[0], i0[3]], rtol=RTOL_TF32)
    for a, b in zip(g0, g1):
        for ga, gb in zip(a, b):
            assert np.abs(ga - gb).max() <= RTOL_TF32 * np.abs(ga).max()


# ---------------------------------------------------------------------------------------------
# batch-resident kernels (csrc/bbb_linear_big.cu): batches of >= 384 rows
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize('B,d_in,d_out', [(384, 64, 64), (512, 256, 128), (700, 100, 72), (1030, 36, 200),
                                          (4096, 512, 256)])
def test_batch_resident_plain_gemm(B, d_in, d_out):
    """sample=False: y = x mu^T + b through the [128 weight rows x 512 batch] TMEM tile; ragged weight-row tiles,
    ragged batch tiles, a K tail (d_in % 32 != 0)."""
    torch.manual_seed(B + d_in)
    layer = bnn_b200.BayesianLinear(d_in, d_out, [-0.2, 0.2], [-5, -4], [1.0], False).to(DEV).eval()
    layer.tf32 = True
    x = torch.randn(B, d_in, device=DEV)
    with torch.no_grad():
        y = layer(x)
    ref = (x.double() @ layer.weight_mu.double().t() + layer.bias_mu.double())
    err = (y.double() - ref).abs().max() / ref.abs().max()
    assert err < 2e-3, float(err)


@pytest.fixture(params=[0, 1], ids=['auto', 'wgrad-split'])
def wgrad_split(request):
    """1: force the large-batch wgrad to split a tile's sample groups over two CTAs (partial gradients + combine kernel);
    the shapes of these tests are too small for the library to choose it by itself."""
    from bnn_b200 import _lib as L
    L.check(L.lib().bbb_debug_wgrad_split(request.param), 'bbb_debug_wgrad_split')
    yield request.param
    L.check(L.lib().bbb_debug_wgrad_split(0), 'bbb_debug_wgrad_split')


@pytest.mark.parametrize('name', DEEP_BIG)
def test_large_batch_fixture_with_wgrad_split(name, wgrad_split):
    # the reference-generated 5-layer fixture (batch 640, S = 3) through the large-batch kernels, both wgrad schedules
    PC.check_train_step(Case(name), DEV, fused=True, rtol=1e-5, rtol_gemm=RTOL_TF32, tf32=True)


@pytest.mark.parametrize('B,d_in,hidden,S', [(400, 64, 96, 3), (1024, 128, 160, 2), (600, 36, 200, 1), (512, 96, 288, 5)])
def test_batch_resident_train_step_matches_fp32_path(B, d_in, hidden, S, wgrad_split):
    """Forward (log-probs counted once per weight tile), dgrad (W^T sampled along i, (x > 0) mask in the drain) and
    the wgrad epilogue regenerate the same Philox eps: TF32 path == exact fp32 path within the TF32 bound."""
    mp = dict(input_shape=d_in, classes=10, batch_size=B, hidden_units=hidden, mode='classification',
              mu_init=[-0.2, 0.2], rho_init=[-5, -4], prior_init=[0.5, 0, -6], mixture_prior=True)
    torch.manual_seed(B)
    x = torch.randn(B, d_in, device=DEV)
    y = torch.randint(0, 10, (B,), device=DEV)
    res = []
    for tf32 in (False, True):
        torch.manual_seed(0)
        net = bnn_b200.BayesianNetwork(dict(mp, tf32=tf32)).to(DEV).train()
        bnn_b200.manual_seed(1, 1)
        info = net.sample_elbo(x, y, 0.3, S)
        info[0].backward()
        res.append(([float(v.detach()) for v in info], PC.net_grads(net)))
    (i0, g0), (i1, g1) = res
    np.testing.assert_allclose(i1[1:3], i0[1:3], rtol=1e-5)
    np.testing.assert_allclose([i1[0], i1[3]], [i0[0], i0[3]], rtol=RTOL_TF32)
    for a, b in zip(g0, g1):
        for ga, gb in zip(a, b):
            assert np.abs(ga - gb).max() <= RTOL_TF32 * np.abs(ga).max()
