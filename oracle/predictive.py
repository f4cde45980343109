"""Float64 restatement of the posterior-predictive summaries (include/bbb.h: bbb_predictive_stats).  TEST
INFRASTRUCTURE ONLY: only tests/ imports it.

Every function takes the sampled outputs [S,B,C] as given (any float dtype; computed in float64) and states each
definition directly, without the kernel's streaming forms: the mean of the softmaxes, the entropies as -sum p log p,
the log predictive density as log of the mean probability / density (through logsumexp, so that it stays finite).
The binning takes the confidences and correct flags as given, so a test can apply it to the kernel's own values.
"""
import math

import numpy as np
import torch


def _entropy(p):
    """-sum_c p_c log p_c over the last axis, with 0 log 0 = 0."""
    return -torch.where(p > 0, p * torch.log(torch.where(p > 0, p, torch.ones_like(p))), torch.zeros_like(p)).sum(-1)


def classification(outs, target=None):
    """outs [S,B,C] logits -> dict of per-row float64 tensors: mean, pred, confidence, entropy, expected_entropy,
    mutual_info, and with target (int64 [B], every label in [0, C)) log_pred, correct, brier."""
    z = torch.as_tensor(outs).double()
    S = z.shape[0]
    p = torch.softmax(z, -1)
    mean = p.mean(0)
    conf, pred = mean.max(-1)                      # torch.max returns the lowest index among equal maxima
    ent = _entropy(mean)
    exp_ent = _entropy(p).mean(0)
    r = dict(mean=mean, pred=pred, confidence=conf, entropy=ent, expected_entropy=exp_ent,
             mutual_info=torch.clamp(ent - exp_ent, min=0.0))
    if target is not None:
        y = torch.as_tensor(target).long()
        logp = torch.log_softmax(z, -1).gather(-1, y.view(1, -1, 1).expand(S, -1, 1))[..., 0]   # [S,B]
        onehot = torch.nn.functional.one_hot(y, z.shape[-1]).double()
        r.update(log_pred=torch.logsumexp(logp, 0) - math.log(S), correct=(pred == y).double(),
                 brier=((mean - onehot) ** 2).sum(-1))
    return r


def regression(outs, target=None, sigma=1.0):
    """outs [S,B,D] -> dict: mean [B,D], variance [B,D] (epistemic, ddof 0), and with target ([B,D], or [B] when
    D = 1, row for row) log_pred [B] = log (1/S) sum_s prod_d N(y_d; f_s,d, sigma^2) and sq_err [B]."""
    f = torch.as_tensor(outs).double()
    S, B, D = f.shape
    r = dict(mean=f.mean(0), variance=f.var(0, unbiased=False))
    if target is not None:
        y = torch.as_tensor(target).double().reshape(B, D)
        ll = (-(y - f) ** 2 / (2 * sigma ** 2) - math.log(sigma) - 0.5 * math.log(2 * math.pi)).sum(-1)   # [S,B]
        r.update(log_pred=torch.logsumexp(ll, 0) - math.log(S), sq_err=((r['mean'] - y) ** 2).sum(-1))
    return r


def bin_index(confidence, n_bins):
    """Bin m holds the confidences in (m/M, (m+1)/M]: m = clamp(ceil(conf M) - 1, 0, M - 1)."""
    c = np.asarray(confidence, dtype=np.float64)
    return np.clip(np.ceil(c * n_bins) - 1, 0, n_bins - 1).astype(np.int64)


def calibration(confidence, correct, n_bins):
    """-> (ece, bins) with bins[m] = (count, mean confidence, accuracy) (NaN for an empty bin) and
    ece = (1/n) sum_m |sum correct_m - sum confidence_m|."""
    conf = np.asarray(confidence, dtype=np.float64)
    cor = np.asarray(correct, dtype=np.float64)
    m = bin_index(conf, n_bins)
    cnt = np.bincount(m, minlength=n_bins)
    s_conf = np.bincount(m, weights=conf, minlength=n_bins)
    s_cor = np.bincount(m, weights=cor, minlength=n_bins)
    n = len(conf)
    ece = float(np.abs(s_cor - s_conf).sum() / n) if n else math.nan
    bins = [(int(k), s_conf[i] / k if k else math.nan, s_cor[i] / k if k else math.nan) for i, k in enumerate(cnt)]
    return ece, bins


def classification_metrics(outs, target, n_bins):
    """The aggregates of a labelled set: dict(n, accuracy, nll, brier, ece, bins)."""
    r = classification(outs, target)
    ece, bins = calibration(r['confidence'].numpy(), r['correct'].numpy(), n_bins)
    n = len(r['correct'])
    return dict(n=n, accuracy=float(r['correct'].mean()), nll=float(-r['log_pred'].mean()),
                brier=float(r['brier'].mean()), ece=ece, bins=bins)


def regression_metrics(outs, target, sigma):
    """dict(n, nll, rmse), rmse over all n * D outputs."""
    r = regression(outs, target, sigma)
    n, D = r['mean'].shape
    return dict(n=n, nll=float(-r['log_pred'].mean()), rmse=math.sqrt(float(r['sq_err'].sum()) / (n * D)))
