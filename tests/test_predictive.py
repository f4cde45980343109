"""Posterior-predictive uncertainty and calibration (BayesianNetwork.predictive, functional.predictive[_stats],
bbb_predictive_stats) against the float64 restatement in oracle/predictive.py.

CPU: the host logic (eps planning across chunks, target handling, result assembly, metrics) on the CPU double of the C
ABI, extended here by a bbb_predictive_stats evaluated with the oracle; the argument checks of the real library, which
return before anything touches a device.  GPU: the same checks through the real kernels, plus Philox-mode chunking,
the decomposition's sanity, the absence of host synchronisation and the MNIST shape."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

import bnn_b200
from bnn_b200 import functional as F, rng as R
from oracle import bbb_oracle as O, predictive as OP
from tests import fake_bbb, parity_cases as PC
from tests.golden_util import Case, SMALL, SMALL_LR

EINVAL = -1
NAN = float('nan')


class PredictiveFake(fake_bbb.FakeLib):
    """The CPU double plus bbb_predictive_stats, evaluated with oracle/predictive.py (argument checks as bbb.h)."""

    def bbb_predictive_stats(self, out, target, S, B, Cc, kind, sigma, n_bins, mean, row_stats, pred, acc, st):
        if (kind not in (1, 2) or S < 1 or B < 0 or not 1 <= Cc <= 1024 or (kind == 1 and not 1 <= n_bins <= 1024)
                or (kind == 2 and not sigma > 0) or (target and not acc) or (B and not (out and mean and row_stats))):
            return EINVAL
        if B == 0:
            return 0
        self.calls.append('predictive_stats')
        Z = fake_bbb._f(out, S, B, Cc)
        M = fake_bbb._f(mean, B, Cc)
        if kind == 1:
            T = fake_bbb._arr(target, C.c_int64, B) if target else None
            valid = (T >= 0) & (T < Cc) if T is not None else np.zeros(B, dtype=bool)
            r = OP.classification(Z, np.where(valid, T, 0) if T is not None else None)
            RS = fake_bbb._f(row_stats, B, 5)
            M[...] = r['mean'].numpy()
            RS[:, 0], RS[:, 1], RS[:, 2], RS[:, 3] = (r[k].numpy() for k in
                                                      ('confidence', 'entropy', 'expected_entropy', 'mutual_info'))
            RS[:, 4] = np.where(valid, r['log_pred'].numpy(), NAN) if T is not None else NAN
            if pred:
                fake_bbb._arr(pred, C.c_int64, B)[...] = r['pred'].numpy()
            if T is not None:
                A = fake_bbb._d(acc, 5 + 3 * n_bins)
                conf, cor = r['confidence'].numpy()[valid], r['correct'].numpy()[valid]
                A[0] += valid.sum()
                A[1] += (~valid).sum()
                A[2] -= r['log_pred'].numpy()[valid].sum()
                A[3] += cor.sum()
                A[4] += r['brier'].numpy()[valid].sum()
                m = OP.bin_index(conf, n_bins)
                bins = A[5:].reshape(n_bins, 3)
                bins[:, 0] += np.bincount(m, minlength=n_bins)
                bins[:, 1] += np.bincount(m, weights=conf, minlength=n_bins)
                bins[:, 2] += np.bincount(m, weights=cor, minlength=n_bins)
        else:
            T = fake_bbb._f(target, B, Cc) if target else None
            r = OP.regression(Z, T, sigma)
            RS = fake_bbb._f(row_stats, B, Cc + 1)
            M[...] = r['mean'].numpy()
            RS[:, :Cc] = r['variance'].numpy()
            RS[:, Cc] = r['log_pred'].numpy() if T is not None else NAN
            if T is not None:
                A = fake_bbb._d(acc, 4)
                A[0] += B
                A[2] -= r['log_pred'].sum().item()
                A[3] += r['sq_err'].sum().item()
        return 0


@pytest.fixture
def fake(monkeypatch):
    lib = PredictiveFake()
    fake_bbb.FakeLib.calls = []
    monkeypatch.setattr(bnn_b200._lib, 'lib', lambda: lib)
    monkeypatch.setattr(bnn_b200._lib, 'require_cuda', lambda *a: None)
    monkeypatch.setattr(bnn_b200._lib, 'stream', lambda: None)
    return lib


# ---------------------------------------------------------------------------------------------------------------------
# shared checks (device 'cpu' runs on the double, 'cuda' on the real library)
# ---------------------------------------------------------------------------------------------------------------------
def _close(got, want, rtol=1e-5, atol=1e-6, what=''):
    g = got.detach().cpu().double().numpy() if torch.is_tensor(got) else np.asarray(got, dtype=np.float64)
    w = want.detach().cpu().double().numpy() if torch.is_tensor(want) else np.asarray(want, dtype=np.float64)
    np.testing.assert_allclose(g, w, rtol=rtol, atol=atol, err_msg=what)


def _check_against_oracle(res, outs, target, mode, sigma, n_bins, rtol=1e-5, atol=1e-6):
    """res (PredictiveResult) against the oracle applied to the sampled outputs `outs` [S,B,C]."""
    if mode == 'classification':
        want = OP.classification(outs, target)
        _close(res.mean, want['mean'], rtol, atol, 'mean')
        for k in ('confidence', 'entropy', 'expected_entropy', 'mutual_info', 'log_pred'):
            _close(getattr(res, k), want[k], rtol, atol, k)
        assert torch.equal(res.pred.cpu(), want['pred'])
        m = res.metrics()
        # binning of the kernel's own confidences and correct flags: a row on a bin edge may round either way
        conf = res.confidence.cpu().double().numpy()
        cor = (res.pred.cpu() == target.cpu()).double().numpy()
        ece, bins = OP.calibration(conf, cor, n_bins)
        assert m['n'] == len(conf)
        assert abs(m['ece'] - ece) <= 1e-6
        assert [b[0] for b in m['bins']] == [b[0] for b in bins]
        assert m['accuracy'] == pytest.approx(float(want['correct'].mean()), abs=1e-12)
        assert m['nll'] == pytest.approx(float(-want['log_pred'].mean()), rel=rtol, abs=atol)
        assert m['brier'] == pytest.approx(float(want['brier'].mean()), rel=rtol, abs=atol)
    else:
        want = OP.regression(outs, target, sigma)
        _close(res.mean, want['mean'], rtol, atol, 'mean')
        _close(res.variance, want['variance'], rtol, atol, 'variance')
        _close(res.log_pred, want['log_pred'], rtol, atol, 'log_pred')
        m = res.metrics()
        wm = OP.regression_metrics(outs, target, sigma)
        assert m['n'] == wm['n']
        assert m['nll'] == pytest.approx(wm['nll'], rel=rtol, abs=atol)
        assert m['rmse'] == pytest.approx(wm['rmse'], rel=rtol, abs=atol)


def _oracle_outputs(case, x, layers_eps):
    if case.lr:
        return torch.stack([O.mlp_forward_lr(x, case.layers, case.prior[1], e, case.mode, calc_kl=False)[0]
                            for e in layers_eps])
    return torch.stack([O.mlp_forward(x, case.layers, case.prior, e, case.mode, calc_log_probs=False)[0]
                        for e in layers_eps])


def check_against_oracle(case, device, S=4, n_bins=5, seed=11, rtol=1e-4, atol=1e-5):
    """net.predictive in the reference eps mode against the oracle's sampled forwards under the same draws
    (torch.manual_seed, then for s: for layer: weight eps, bias eps).  End to end, so the tolerance also covers the
    forward's fp32 round-off, which a likelihood with sigma = 0.1 amplifies a hundredfold in the log density."""
    net = PC.build_net(case, device).eval()
    with torch.random.fork_rng():
        torch.manual_seed(seed)
        eps = O.draw_eps(case.dims, S, batch=case.B, local_reparam=case.lr)
    outs = _oracle_outputs(case, case.x, eps)
    with bnn_b200.eps_mode('reference'):
        torch.manual_seed(seed)
        res = net.predictive(case.x.to(device), S, target=case.y.to(device), sigma=case.sigma, n_bins=n_bins)
    _check_against_oracle(res, outs, case.y, case.mode, case.sigma, n_bins, rtol, atol)


def _maxnorm_close(got, want, tol, what):
    """|got - want| <= tol * max|want| (the project's per-tensor max-norm relative bound)"""
    g, w = got.double(), want.double()
    scale = float(w[torch.isfinite(w)].abs().max()) if w.numel() else 0.0
    err = float((g - w).abs().max()) if w.numel() else 0.0
    assert err <= tol * max(scale, 1e-30), f'{what}: {err:.3e} > {tol:.1e} * {scale:.3e}'


def _stats(res):
    keys = ('mean', 'pred', 'confidence', 'entropy', 'expected_entropy', 'mutual_info', 'variance', 'log_pred')
    return {k: getattr(res, k).cpu() for k in keys if getattr(res, k) is not None}


def check_ws_chunking(case, device, S=3):
    """Weight sampling: chunk_rows B, 3 and 1 give the same per-row stats and aggregates; eps is planned once per
    call, so the injected eps queue of ONE call's draws suffices and is used up."""
    assert not case.lr
    net = PC.build_net(case, device).eval()
    x, y = case.x.to(device), case.y.to(device)
    with torch.random.fork_rng():
        torch.manual_seed(5)
        draws = [t for per_s in O.draw_eps(case.dims, S) for pair in per_s for t in pair]
    runs = []
    with bnn_b200.eps_mode('injected'):
        for rows in (case.B, 3, 1):
            R.set_injected_eps(draws)
            res = net.predictive(x, S, target=y, sigma=case.sigma, n_bins=4, chunk_rows=rows)
            assert R._st().queue == []
            runs.append((_stats(res), res.metrics()))
    for st, m in runs[1:]:
        for k, v in st.items():
            _maxnorm_close(v, runs[0][0][k], 1e-5, k)
        for k, v in m.items():
            if k == 'bins':
                assert [b[0] for b in v] == [b[0] for b in runs[0][1][k]]
            else:
                assert v == pytest.approx(runs[0][1][k], rel=1e-5, abs=1e-6), k


def check_lr_chunking(case, device, S=2, rows=3):
    """Local reparameterisation: chunk c equals the oracle on the rows of chunk c with the draws that chunk consumed,
    in order."""
    assert case.lr
    net = PC.build_net(case, device).eval()
    with torch.random.fork_rng():
        torch.manual_seed(7)
        outs = []
        for r0 in range(0, case.B, rows):
            xc = case.x[r0:r0 + rows]
            n = xc.shape[0]
            outs.append(_oracle_outputs(case, xc, O.draw_eps(case.dims, S, batch=n, local_reparam=True)))
    outs = torch.cat(outs, 1)
    with bnn_b200.eps_mode('reference'):
        torch.manual_seed(7)
        res = net.predictive(case.x.to(device), S, target=case.y.to(device), sigma=case.sigma, n_bins=4,
                             chunk_rows=rows)
    _check_against_oracle(res, outs, case.y, case.mode, case.sigma, 4, 1e-4, 1e-5)


def _logits(S, B, Cc, scale=3.0, seed=0):
    g = torch.Generator().manual_seed(seed)
    return (scale * torch.randn(S, B, Cc, generator=g)).float()


def check_edge_cases(device):
    # S = 1: the two entropies are formed differently; only round-off and the clamp separate them
    z = _logits(1, 64, 10)
    _, rs, _, _ = F.predictive_stats(z.to(device))
    assert float(rs[:, 3].max()) <= 1e-6
    # C = 1: one certain class
    y1 = torch.zeros(5, dtype=torch.int64)
    mean, rs, pred, acc = F.predictive_stats(_logits(3, 5, 1).to(device), y1.to(device), n_bins=3)
    _close(mean, np.ones((5, 1)), 0, 1e-7)
    _close(rs[:, :4], np.tile([1.0, 0.0, 0.0, 0.0], (5, 1)), 0, 1e-6)
    _close(rs[:, 4], np.zeros(5), 0, 1e-6)
    assert pred.cpu().tolist() == [0] * 5
    # C = 100: more than one pass of the warp's lanes over the classes
    z, y = _logits(5, 37, 100, seed=1), torch.randint(0, 100, (37,), generator=torch.Generator().manual_seed(2))
    for n_bins in (10, 1):
        mean, rs, pred, acc = F.predictive_stats(z.to(device), y.to(device), n_bins=n_bins)
        res = bnn_b200.PredictiveResult(mean, pred, *rs[:, :4].unbind(1), log_pred=rs[:, 4], acc=acc, n_bins=n_bins)
        _check_against_oracle(res, z, y, 'classification', 1.0, n_bins)
        if n_bins == 1:      # one bin: ECE = |accuracy - mean confidence|
            m = res.metrics()
            assert m['ece'] == pytest.approx(abs(m['accuracy'] - float(res.confidence.double().mean())), abs=1e-6)
    # regression with D > 32 outputs, and D = 1 with a [B] target
    for D, tshape in ((40, (9, 40)), (1, (9,))):
        f = _logits(4, 9, D, 1.0, seed=3)
        t = torch.randn(tshape, generator=torch.Generator().manual_seed(4))
        mean, rs, _, acc = F.predictive_stats(f.to(device), t.to(device), 'regression', 0.5)
        res = bnn_b200.PredictiveResult(mean, variance=rs[:, :-1], log_pred=rs[:, -1], acc=acc)
        _check_against_oracle(res, f, t, 'regression', 0.5, 0)
    # B = 0
    mean, rs, pred, acc = F.predictive_stats(torch.zeros(3, 0, 4, device=device), torch.zeros(0, dtype=torch.int64,
                                                                                               device=device))
    assert tuple(mean.shape) == (0, 4) and tuple(rs.shape) == (0, 5) and float(acc.abs().sum()) == 0.0
    # a label outside [0, C) is not read; metrics() refuses
    y = torch.tensor([0, 4, 1, -1], dtype=torch.int64)
    mean, rs, pred, acc = F.predictive_stats(_logits(2, 4, 4).to(device), y.to(device), n_bins=2)
    assert float(acc[1]) == 2.0 and float(acc[0]) == 2.0
    assert math.isnan(float(rs[1, 4])) and math.isnan(float(rs[3, 4])) and not math.isnan(float(rs[0, 4]))
    res = bnn_b200.PredictiveResult(mean, pred, *rs[:, :4].unbind(1), log_pred=rs[:, 4], acc=acc, n_bins=2)
    with pytest.raises(ValueError, match='outside'):
        res.metrics()


# ---------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('name', SMALL + SMALL_LR)
def test_predictive_matches_oracle(fake, name):
    check_against_oracle(Case(name), 'cpu')
    assert fake.calls.count('predictive_stats') == 1


@pytest.mark.parametrize('name', ['small_cls_mix', 'small_reg_mix'])
def test_weight_sampling_chunks_share_one_eps_plan(fake, name):
    check_ws_chunking(Case(name), 'cpu')


@pytest.mark.parametrize('name', SMALL_LR)
def test_local_reparam_chunks_draw_in_order(fake, name):
    check_lr_chunking(Case(name), 'cpu')


def test_predictive_edge_cases(fake):
    check_edge_cases('cpu')


def test_default_chunking_bounds_the_workspace(fake):
    """chunk_rows=None splits the rows into equal chunks whose activations fit the budget."""
    widths = [1200, 1200, 10]
    rows = F.predictive_chunk_rows(10, widths)
    assert 10 * rows * sum(widths) * 4 <= F.PREDICTIVE_BUDGET_BYTES < 10 * (rows + 1) * sum(widths) * 4
    case = Case('small_cls_mix')
    net = PC.build_net(case, 'cpu').eval()
    with bnn_b200.eps_mode('reference'):
        net.predictive(case.x, 2, target=case.y)
    assert fake.calls.count('predictive_stats') == 1


def test_target_shape_is_checked(fake):
    case = Case('small_reg_mix')
    net = PC.build_net(case, 'cpu').eval()
    with bnn_b200.eps_mode('reference'), pytest.raises(ValueError, match='regression target'):
        net.predictive(case.x, 2, target=case.y[:, 0])          # [B] against D = 3 outputs: no broadcast
    with bnn_b200.eps_mode('reference'):
        res = net.predictive(case.x, 2)
    assert res.log_pred is None
    with pytest.raises(ValueError, match='needs the target'):
        res.metrics()


def test_abi_rejects_bad_arguments():
    """The real library's argument checks (they return before any device work, so they run without a GPU)."""
    lib = bnn_b200._lib.lib()
    buf = C.c_void_p(16)            # never dereferenced: every call below is refused first
    ok = dict(out=buf, target=None, S=2, B=4, C=3, kind=1, sigma=1.0, n_bins=5, mean=buf, rs=buf, pred=None, acc=None)
    bad = [dict(kind=0), dict(kind=3), dict(S=0), dict(B=-1), dict(C=0), dict(C=1025), dict(n_bins=0),
           dict(n_bins=1025), dict(kind=2, sigma=0.0), dict(target=buf), dict(out=None), dict(mean=None),
           dict(rs=None)]
    for change in bad:
        a = dict(ok, **change)
        st = lib.bbb_predictive_stats(a['out'], a['target'], a['S'], a['B'], a['C'], a['kind'], a['sigma'],
                                      a['n_bins'], a['mean'], a['rs'], a['pred'], a['acc'], None)
        assert st == EINVAL, change
    # B == 0 is a no-op, null pointers included
    assert lib.bbb_predictive_stats(None, None, 2, 0, 3, 1, 1.0, 5, None, None, None, None, None) == 0


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
def _mnist_net(tf32, rho=None, dims=(784, 1200, 1200, 10), lr=False):
    mp = dict(input_shape=dims[0], classes=dims[-1], batch_size=128, hidden_units=list(dims[1:-1]),
              mode='classification', mu_init=[-0.2, 0.2], rho_init=[-5, -4], prior_init=[1.0] if lr else [0.5, 0, -8],
              mixture_prior=not lr, local_reparam=lr, tf32=tf32)
    torch.manual_seed(0)
    net = bnn_b200.BayesianNetwork(mp).cuda().eval()
    if rho is not None:
        with torch.no_grad():
            for l in net.layers():
                l.weight_rho.fill_(rho)
                l.bias_rho.fill_(rho)
    return net


def _mnist_data(N, seed=1):
    g = torch.Generator().manual_seed(seed)
    return torch.rand(N, 784, generator=g).cuda(), torch.randint(0, 10, (N,), generator=g).cuda()


@pytest.mark.gpu
@pytest.mark.parametrize('name', SMALL + SMALL_LR)
def test_gpu_predictive_matches_oracle(name):
    """Exact fp32 mode: the kernel's per-row stats against the float64 oracle applied to the very outputs the sampled
    forward produced (sample_predict under the same draws), and those outputs against the oracle's forward."""
    case = Case(name)
    net = PC.build_net(case, 'cuda').eval()
    x, y = case.x.cuda(), case.y.cuda()
    S, n_bins = 4, 5
    with bnn_b200.eps_mode('reference'):
        torch.manual_seed(11)
        outs = net.sample_predict(x, S)
        torch.manual_seed(11)
        res = net.predictive(x, S, target=y, sigma=case.sigma, n_bins=n_bins)
    _check_against_oracle(res, outs.cpu(), case.y, case.mode, case.sigma, n_bins)
    check_against_oracle(case, 'cuda')   # and against the oracle's own forward, end to end


@pytest.mark.gpu
@pytest.mark.parametrize('name', ['small_cls_mix', 'small_reg_mix'])
def test_gpu_weight_sampling_chunks_share_one_eps_plan(name):
    check_ws_chunking(Case(name), 'cuda')


@pytest.mark.gpu
@pytest.mark.parametrize('name', SMALL_LR)
def test_gpu_local_reparam_chunks_draw_in_order(name):
    check_lr_chunking(Case(name), 'cuda')


@pytest.mark.gpu
def test_gpu_predictive_edge_cases():
    check_edge_cases('cuda')


@pytest.mark.gpu
@pytest.mark.parametrize('tf32', [False, True])
def test_gpu_philox_predictive_equals_sample_predict_and_ignores_chunking(tf32):
    """Philox, weight sampling: the mean equals softmax_mean(sample_predict) at the same pinned step; chunks of 10 000,
    1 000 and 128 rows (in TF32 mode three different hidden-layer kernel families) agree; one step per call."""
    net = _mnist_net(tf32)
    x, y = _mnist_data(10000)
    S = 10
    bnn_b200.manual_seed(3, step=40)
    with torch.no_grad():
        want = F.softmax_mean(net.sample_predict(x[:512], S))
    bnn_b200.manual_seed(3, step=40)
    got = net.predictive(x[:512], S).mean
    _close(got, want, 0, 1e-6, 'mean vs softmax_mean(sample_predict)')
    runs = []
    for rows in (10000, 1000, 128):
        bnn_b200.manual_seed(3, step=40)
        res = net.predictive(x, S, target=y, chunk_rows=rows)
        assert R._st().step == 41
        runs.append((_stats(res), res.metrics()))
    tol = 5e-3 if tf32 else 1e-5
    base, mb = runs[0]
    top2 = base['mean'].double().topk(2, -1).values
    near_tie = (top2[:, 0] - top2[:, 1]) <= tol
    for st, m in runs[1:]:
        for k in ('mean', 'confidence', 'entropy', 'expected_entropy', 'mutual_info', 'log_pred'):
            _maxnorm_close(st[k], base[k], tol, k)
        differ = st['pred'] != base['pred']
        assert not bool((differ & ~near_tie).any())
        n_diff, n = int(differ.sum()), m['n']
        assert abs(m['accuracy'] - mb['accuracy']) * n <= n_diff
        assert abs(m['nll'] - mb['nll']) <= tol * float(base['log_pred'].abs().max())
        assert m['brier'] == pytest.approx(mb['brier'], rel=tol, abs=tol)
        # n ECE moves by |d confidence| for a row that stays in its bin, by <= 2 for one that changes bins, by <= 1
        # for one whose correctness flips
        d_conf = float((st['confidence'].double() - base['confidence'].double()).abs().sum())
        moved = int((OP.bin_index(st['confidence'], 15) != OP.bin_index(base['confidence'], 15)).sum())
        assert abs(m['ece'] - mb['ece']) * n <= d_conf + 2 * moved + n_diff + 1e-6 * n


@pytest.mark.gpu
def test_gpu_decomposition_sanity():
    """sigma ~ 0: every sample is the same network, no epistemic uncertainty; sigma = softplus(2): plenty."""
    x, _ = _mnist_data(2048)
    x = x[:, :64].contiguous()
    dims = (64, 128, 128, 10)
    for rho, check in ((-30.0, 'none'), (2.0, 'much')):
        net = _mnist_net(False, rho, dims)
        res = net.predictive(x, 8)
        mi, ent, ee = res.mutual_info.cpu(), res.entropy.cpu(), res.expected_entropy.cpu()
        if check == 'none':
            assert float(mi.max()) < 1e-6
        else:
            assert float((mi > 1e-3).double().mean()) >= 0.9
        assert float(ent.max()) <= math.log(10) + 1e-6
        assert bool((ee <= ent + 1e-6).all())


@pytest.mark.gpu
@pytest.mark.parametrize('lr', [False, True])
def test_gpu_predictive_does_not_synchronise(lr):
    net = _mnist_net(True, dims=(784, 256, 256, 10), lr=lr)
    x, y = _mnist_data(3000)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode('error')
    try:
        res = net.predictive(x, 4, target=y, chunk_rows=1024)
    finally:
        torch.cuda.set_sync_debug_mode('default')
    assert res.metrics()['n'] == 3000


@pytest.mark.gpu
def test_gpu_mnist_shape_tf32_aggregates():
    """784-1200-1200-10, N = 4096, S = 10, TF32: the aggregates against the oracle applied to sample_predict's outputs
    under the same pinned step (default chunking: two chunks of the same kernel family)."""
    net = _mnist_net(True)
    x, y = _mnist_data(4096, seed=2)
    S = 10
    bnn_b200.manual_seed(9, step=5)
    with torch.no_grad():
        outs = net.sample_predict(x, S).cpu()
    bnn_b200.manual_seed(9, step=5)
    m = net.predictive(x, S, target=y).metrics()
    want = OP.classification_metrics(outs, y.cpu(), 15)
    mean = OP.classification(outs)['mean']
    top2 = mean.topk(2, -1).values
    near = int(((top2[:, 0] - top2[:, 1]) <= 5e-3).sum())
    assert m['n'] == want['n'] == 4096
    assert abs(m['accuracy'] - want['accuracy']) * 4096 <= near
    assert m['nll'] == pytest.approx(want['nll'], rel=5e-3)
    assert m['brier'] == pytest.approx(want['brier'], rel=5e-3)
    assert abs(m['ece'] - want['ece']) <= 5e-3
