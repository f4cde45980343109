"""BayesianNetwork (networks.py:140-225) on the CUDA kernels, plus the two stock baselines the
reference's callers import by name (MLP, MLP_Dropout: plain torch.nn, not part of the hot path)."""
import math
import os
from dataclasses import dataclass
from typing import Optional

import torch
from torch import nn

from . import functional as F
from .layers import PRIOR_BUFFERS, BayesianLinear, BayesianLinearLR, gauss_prior

_HALF_LOG_2PI = 0.5 * math.log(2 * math.pi)


@dataclass
class PredictiveResult:
    """What BayesianNetwork.predictive returns: per-row device tensors and the device aggregates behind metrics().

    classification: mean [B,C] (mean over the samples of softmax), pred [B] (argmax of mean, lowest index on ties),
    confidence [B] (mean[pred]), entropy [B] (of mean), expected_entropy [B] (mean over the samples of each softmax's
    entropy: aleatoric), mutual_info [B] (entropy - expected_entropy, clamped at 0: epistemic).
    regression: mean [B,D], variance [B,D] (epistemic, over the samples; total = variance + sigma**2).
    heteroscedastic regression: also aleatoric_variance [B,D] (the mean over the samples of sigma(x)**2; total =
    variance + aleatoric_variance).
    log_pred [B]: log predictive density of each row's target (None without a target)."""
    mean: torch.Tensor
    pred: Optional[torch.Tensor] = None
    confidence: Optional[torch.Tensor] = None
    entropy: Optional[torch.Tensor] = None
    expected_entropy: Optional[torch.Tensor] = None
    mutual_info: Optional[torch.Tensor] = None
    variance: Optional[torch.Tensor] = None
    log_pred: Optional[torch.Tensor] = None
    acc: Optional[torch.Tensor] = None       # fp64 aggregates of bbb_predictive_stats (include/bbb.h)
    n_bins: int = 0
    aleatoric_variance: Optional[torch.Tensor] = None

    def metrics(self):
        """The aggregates as python numbers; the one host read of a prediction.  Classification: dict(n, accuracy,
        nll, brier, ece, bins) with bins[m] = (count, mean confidence, accuracy) of the confidences in (m/M, (m+1)/M]
        (NaN for an empty bin) and ece = sum_m count_m |accuracy_m - confidence_m| / n.  Regression: dict(n, nll, rmse),
        rmse over all n * D outputs.  nll is the mean negative log predictive density.  Raises ValueError without a
        target, or when a label was outside [0, C)."""
        if self.acc is None:
            raise ValueError('metrics() needs the target: call predictive(x, samples, target=...)')
        a = self.acc.cpu().tolist()
        if a[1]:
            raise ValueError(f'{int(a[1])} target label(s) outside [0, {self.mean.shape[1]}): those rows were not scored')
        n = int(a[0])
        div = (lambda v: v / n) if n else (lambda v: math.nan)
        if self.pred is None:
            return dict(n=n, nll=div(a[2]), rmse=math.sqrt(div(a[3]) / self.mean.shape[1]))
        bins = []
        ece = 0.0
        for m in range(self.n_bins):
            cnt, conf, cor = a[5 + 3 * m:8 + 3 * m]
            bins.append((int(cnt), conf / cnt if cnt else math.nan, cor / cnt if cnt else math.nan))
            ece += abs(cor - conf)
        return dict(n=n, accuracy=div(a[3]), nll=div(a[2]), brier=div(a[4]), ece=div(ece), bins=bins)


class BayesianNetwork(nn.Module):
    """Same model_params dict, attributes (l1, l1_act, ...), methods and return tuples as the reference.

    Extensions (strict supersets): 'local_reparam' defaults to False when absent, which is what lets
    reinforcement_learning/bandits.py construct the net (SURVEY App. B-1); 'hidden_units' may be a list
    (or 'n_hidden' may be given) for nets deeper than the reference's fixed two hidden layers
    (BASELINE.json config 5); 'tf32' opts in to the tcgen05 kind::tf32 tensor path.

    'likelihood' (regression only): 'gaussian' (default), the reference's fixed noise sigma passed to sample_elbo; or
    'heteroscedastic', a learned per-input noise (Kendall & Gal 2017): the last layer has 2 * classes outputs [f | r],
    the mean f and a raw scale r, and sigma(x) = sigma_min + softplus(r) with 'sigma_min' (default 1e-3) > 0.  `classes`
    still counts the targets D; forward / sample_predict return the raw [.., 2D] outputs.

    Per-weight Gaussian priors (posterior_to_prior, set_prior, clear_prior): every weight and bias w_i can get its own
    prior N(m_i, sp_i^2), which replaces the model_params prior in the ELBO of both estimators (sample_elbo: Monte Carlo
    log p of the sampled weights; sample_elbo_lr: the closed-form KL) and in log_prior() / kl_cost() after a training
    forward.  posterior_to_prior() makes the current posterior the prior of the next task (variational continual
    learning, Nguyen et al. 2018).  The prior lives in non-persistent buffers of each layer (prior_weight_mu / _rho,
    prior_bias_mu / _rho, sp = softplus(rho)): it is NOT part of state_dict, which keeps the reference's keys.
    Prediction (sample_predict, predictive) and evaluation mode do not read it.  A captured GraphedTrainStep reads the
    buffers by pointer, so refreshing them in place (posterior_to_prior or set_prior on a net that already has a
    per-weight prior of the same shapes) is seen by later replays; switching between no per-weight prior and one
    changes the launch sequence and needs a new capture.
    """

    def __init__(self, model_params):
        super().__init__()
        self.input_shape = model_params['input_shape']
        self.classes = model_params['classes']
        self.batch_size = model_params['batch_size']
        self.hidden_units = model_params['hidden_units']
        self.mode = model_params['mode']
        self.mu_init = model_params['mu_init']
        self.rho_init = model_params['rho_init']
        self.prior_init = model_params['prior_init']
        self.mixture_prior = model_params['mixture_prior']
        self.local_reparam = model_params.get('local_reparam', False)
        # 'tf32' key, else the process-wide default BBB_TF32=1 (the switch for callers that build model_params themselves:
        # reg_task.py / class_task.py / bandits.py run unchanged and cannot pass the key)
        self.tf32 = bool(model_params.get('tf32', os.environ.get('BBB_TF32', '0') == '1'))
        self.fused = bool(model_params.get('fused', True))
        self.likelihood = model_params.get('likelihood', 'gaussian')
        self.sigma_min = float(model_params.get('sigma_min', 1e-3))
        if self.likelihood not in ('gaussian', 'heteroscedastic'):
            raise ValueError(f"likelihood must be 'gaussian' or 'heteroscedastic', got {self.likelihood!r}")
        if self.likelihood == 'heteroscedastic':
            if self.mode != 'regression':
                raise ValueError("the heteroscedastic likelihood is a regression likelihood: needs mode='regression'")
            if not self.sigma_min > 0:
                raise ValueError(f'sigma_min must be > 0, got {self.sigma_min}')
        self._het = self.likelihood == 'heteroscedastic'

        if isinstance(self.hidden_units, (list, tuple)):
            hidden = list(self.hidden_units)
        else:
            hidden = [self.hidden_units] * int(model_params.get('n_hidden', 2))
        dims = [self.input_shape] + hidden + [self.classes * (2 if self._het else 1)]
        layer = BayesianLinearLR if self.local_reparam else BayesianLinear
        self.n_layers = len(dims) - 1
        for i in range(self.n_layers):
            l = layer(dims[i], dims[i + 1], self.mu_init, self.rho_init, self.prior_init, self.mixture_prior)
            l.layer_id = i
            if not self.local_reparam:
                l.tf32 = self.tf32
            setattr(self, f'l{i + 1}', l)
            if i + 1 < self.n_layers:
                setattr(self, f'l{i + 1}_act', nn.ReLU())
        self._prior = None if self.local_reparam else F.make_prior(self.prior_init, self.mixture_prior)
        self._est = F._LocalReparam(self.prior_init[0]) if self.local_reparam else F._WeightSampling(self._prior)

    def layers(self):
        return [getattr(self, f'l{i + 1}') for i in range(self.n_layers)]

    # ---- per-weight Gaussian priors -------------------------------------------------------------------------------
    def _store_prior(self, layer, values):
        """Write a layer's four prior tensors: in place where the buffers exist with the same shape and device (a
        captured graph keeps reading them), else as new buffers."""
        for name, v in zip(PRIOR_BUFFERS, values):
            cur = getattr(layer, name)
            if cur is not None and cur.shape == v.shape and cur.device == v.device:
                cur.copy_(v)
            else:
                setattr(layer, name, v.detach().to(torch.float32).contiguous().clone())

    def posterior_to_prior(self):
        """Make the current posterior q(w) = N(mu, softplus(rho)^2) of every weight and bias its prior: a copy of
        (mu, rho) into the layer's prior buffers (in place when they exist)."""
        with torch.no_grad():
            for l in self.layers():
                self._store_prior(l, l.params())

    def set_prior(self, layers):
        """Set a per-weight Gaussian prior: `layers` holds one (weight_mean, weight_sigma, bias_mean, bias_sigma) per
        layer, each a tensor of the shape of that layer's weight_mu / bias_mu (its own layout: [out, in] for weight
        sampling, [in, out] for local reparameterisation) on the parameters' device, or a python number for all of
        them.  sigma is stored as rho = log(expm1(sigma)), formed in float64.  Raises ValueError for a wrong number of
        layers, a shape or device mismatch, or a sigma that is not finite and > 0; nothing is changed then."""
        ls = self.layers()
        layers = list(layers)
        if len(layers) != len(ls):
            raise ValueError(f'set_prior: expected one (weight_mean, weight_sigma, bias_mean, bias_sigma) per layer, '
                             f'{len(ls)} layers, got {len(layers)}')
        staged = []
        for i, (l, entry) in enumerate(zip(ls, layers)):
            entry = tuple(entry)
            if len(entry) != 4:
                raise ValueError(f'set_prior: layer {i + 1}: expected (weight_mean, weight_sigma, bias_mean, '
                                 f'bias_sigma), got {len(entry)} values')
            vals = []
            for k, (v, ref) in enumerate(zip(entry, (l.weight_mu, l.weight_mu, l.bias_mu, l.bias_mu))):
                what = f'set_prior: layer {i + 1} {("weight_mean", "weight_sigma", "bias_mean", "bias_sigma")[k]}'
                if torch.is_tensor(v):
                    if tuple(v.shape) != tuple(ref.shape):
                        raise ValueError(f'{what}: shape {tuple(v.shape)}, expected {tuple(ref.shape)}')
                    if v.device != ref.device:
                        raise ValueError(f'{what}: device {v.device}, expected {ref.device}')
                    v = v.detach().to(torch.float64)
                else:
                    v = torch.full(tuple(ref.shape), float(v), dtype=torch.float64, device=ref.device)
                if k % 2:
                    if not bool(torch.isfinite(v).all()) or not bool((v > 0).all()):
                        raise ValueError(f'{what}: every sigma must be finite and > 0')
                    v = v + torch.log(-torch.expm1(-v))      # log(expm1(sigma)), stable for large sigma
                vals.append(v.to(torch.float32).contiguous())
            staged.append(vals)
        with torch.no_grad():
            for l, vals in zip(ls, staged):
                self._store_prior(l, vals)

    def clear_prior(self):
        """Drop the per-weight priors: the model_params prior applies again."""
        for l in self.layers():
            for name in PRIOR_BUFFERS:
                setattr(l, name, None)

    def _gauss_priors(self):
        """Per layer (weight m, weight r, bias m, bias r) of the per-weight prior, or None when no layer has one."""
        ps = [gauss_prior(l) for l in self.layers()]
        if all(p is None for p in ps):
            return None
        if any(p is None for p in ps):
            raise ValueError('a per-weight prior must be set on every layer of the network or on none '
                             '(posterior_to_prior / set_prior set all of them)')
        return ps

    def forward(self, x, sample=False):
        if self.mode == 'classification':
            x = x.view(-1, self.input_shape)  # Flatten images
        for i, l in enumerate(self.layers()):
            x = l(x, sample)
            if i + 1 < self.n_layers:
                x = getattr(self, f'l{i + 1}_act')(x)
        return x

    # ---- prediction (SURVEY 8 f2): the reference's callers loop `net(x, sample=True)` test_samples times
    # (class_task.py:81-87, reg_task.py:76-83); these run all the sampled forwards in one launch per layer ----
    def sample_predict(self, x, samples):
        """`samples` sampled forward passes at once -> outputs [samples, B, classes].  Same values, in the
        reference eps mode the same draws in the same order, as `samples` calls of net(x, sample=True) in eval
        mode (no log-probs are evaluated)."""
        x2 = self._flat_input(x)
        params = [l.params() for l in self.layers()]
        with torch.no_grad():
            return F._network_forward(self._est, x2, params, samples, True, False, self.tf32)[0]

    def predict_proba(self, x, samples):
        """BNN_Classification.predict (class_task.py:81-87): softmax of every sampled forward, averaged."""
        return F.softmax_mean(self.sample_predict(x, samples))

    def predictive(self, x, samples, target=None, sigma=1.0, n_bins=15, chunk_rows=None):
        """Posterior predictive of `samples` sampled networks on the rows of x, with its uncertainty and, given the
        targets, its calibration -> PredictiveResult (device tensors; .metrics() reads the aggregates).  Eval
        semantics (sampled weights, no log-probs), no autograd, any depth, both estimators, fp32 or TF32 as the
        network is set.  Classification: the outputs are logits and target int64 [B]; regression: likelihood
        N(y; f, sigma^2) and target [B, D] ([B] when D = 1), matched row for row.  Heteroscedastic likelihood: the
        noise is the net's own sigma(x), `sigma` must stay at its default, and aleatoric_variance is filled.
        The rows are processed in chunks of chunk_rows (None: as many as keep the activations under a fixed budget,
        functional.predictive).  With weight sampling every chunk is scored by the same `samples` networks, so the
        result does not depend on chunk_rows beyond round-off, and the call consumes one Philox step, as
        sample_predict does; with local reparameterisation each chunk draws its own noise (one step per chunk)."""
        x2 = self._flat_input(x)
        params = [l.params() for l in self.layers()]
        mode = self.mode
        if self._het:
            self._check_no_sigma(sigma)
            mode, sigma = 'heteroscedastic', self.sigma_min
        F._check_predictive_mode(mode)
        with torch.no_grad():
            mean, rs, pred, acc = F._predictive(self._est, x2, params, samples, mode, target, sigma, n_bins, chunk_rows,
                                                self.tf32)
        log_pred = rs[:, -1] if target is not None else None
        if self._het:
            D = self.classes
            return PredictiveResult(mean, variance=rs[:, :D], aleatoric_variance=rs[:, D:2 * D], log_pred=log_pred,
                                    acc=acc)
        if self.mode == 'classification':
            return PredictiveResult(mean, pred, rs[:, 0], rs[:, 1], rs[:, 2], rs[:, 3], log_pred=log_pred, acc=acc,
                                    n_bins=n_bins)
        return PredictiveResult(mean, variance=rs[:, :-1], log_pred=log_pred, acc=acc)

    # ---- SNR pruning (SURVEY 8 f3; weight_pruning.py:81-115) on the (mu, rho) stream, one kernel pass per tensor ----
    def snr(self):
        """SNR in decibels of every weight and bias, flattened in the order weight_pruning.get_snr... walks the layers:
        per layer weights then biases.  Returns a 1-D device tensor."""
        parts = []
        for l in self.layers():
            parts.append(F.compute_snr(l.weight_mu.data, l.weight_rho.data).reshape(-1))
            parts.append(F.compute_snr(l.bias_mu.data, l.bias_rho.data).reshape(-1))
        return torch.cat(parts)

    def prune_weights(self, snrs, drop_percentage=0.5):
        """prune_weights(model, snrs, drop_percentage) of weight_pruning.py:85-115: the SNR threshold is the
        100 drop_percentage-th percentile of `snrs` (numpy semantics), then mu and rho of every weight and bias whose
        SNR is not above it are multiplied by zero, in place.  Returns the fraction of parameters kept."""
        import numpy as np
        snr_threshold = float(np.percentile(snrs.detach().cpu().numpy() if torch.is_tensor(snrs) else snrs,
                                            100 * drop_percentage))
        kept, total = 0, 0
        with torch.no_grad():
            for l in self.layers():
                for mu, rho in ((l.weight_mu, l.weight_rho), (l.bias_mu, l.bias_rho)):
                    kept = kept + F.snr_prune_(mu.data, rho.data, snr_threshold)
                    total += mu.numel()
        return float(kept) / max(total, 1)

    def log_prior(self):
        return sum(l.log_prior for l in self.layers())

    def log_variational_posterior(self):
        return sum(l.log_variational_posterior for l in self.layers())

    def kl_cost(self):
        return sum(l.kl_cost for l in self.layers())

    def get_nll(self, outputs, target, sigma=1.):
        if self._het:
            # outputs [.., 2D] = [f | r], sigma = sigma_min + softplus(r) (the stable form of bbb_nll_gauss_het)
            self._check_no_sigma(sigma)
            D = self.classes
            f, r = outputs[..., :D], outputs[..., D:]
            s = self.sigma_min + (torch.clamp(r, min=0) + torch.log1p(torch.exp(-r.abs())))
            y = self._het_target(target, f.shape[0])
            return (((y - f) / s) ** 2 / 2 + torch.log(s) + _HALF_LOG_2PI).sum()
        if self.mode == 'regression':
            # -Normal(outputs, sigma).log_prob(target).sum() (networks.py:185) written out -- same arithmetic and the same
            # broadcasting of target against outputs (SURVEY App. B-3) -- because the distribution object turns a python
            # sigma into a device tensor with a host-to-device copy, which a CUDA-graph capture does not allow
            if torch.is_tensor(sigma):
                nll = -torch.distributions.Normal(outputs, sigma).log_prob(target).sum()
            else:
                import math
                var = float(sigma) ** 2
                nll = -(-((target - outputs) ** 2) / (2 * var) - math.log(float(sigma)) - math.log(math.sqrt(2 * math.pi))).sum()
        elif self.mode == 'classification':
            nll = nn.CrossEntropyLoss(reduction='sum')(outputs, target)
        else:
            raise Exception("Training mode must be either 'regression' or 'classification'")
        return nll

    # ---- fused-path eligibility: the likelihood kernels cover the reference's two regular cases --------
    def _fusable(self, x2, target):
        if not self.fused:
            return False
        B = x2.shape[0]
        if self.mode == 'classification':
            return target.dtype == torch.int64 and target.dim() == 1 and target.shape[0] == B
        if self.mode == 'regression':      # [B, D] targets; the [B] vs [B,1] broadcast (SURVEY B-3) goes the general way
            return target.dim() == 2 and tuple(target.shape) == (B, self.classes) and target.is_floating_point()
        return False

    def _check_no_sigma(self, sigma):
        """The heteroscedastic net learns its noise: a fixed sigma would contradict it."""
        if torch.is_tensor(sigma) or sigma != 1.:
            raise ValueError('the heteroscedastic likelihood learns sigma(x): do not pass sigma (model_params '
                             "'sigma_min' bounds it from below)")

    def _het_target(self, target, B):
        """The heteroscedastic likelihood's target, [B, D] ([B] when D = 1), matched row for row (no broadcast)."""
        D = self.classes
        if not (tuple(target.shape) == (B, D) or (D == 1 and tuple(target.shape) == (B,))):
            raise ValueError(f'heteroscedastic target must have shape ({B}, {D})' + (f' or ({B},)' if D == 1 else '') +
                             f', got {tuple(target.shape)}')
        return target.reshape(B, D)

    def _flat_input(self, input):
        return input.view(-1, self.input_shape) if self.mode == 'classification' else input.reshape(-1, self.input_shape)

    def _sample_elbo(self, input, target, beta, samples, sigma):
        """The body both sample_elbo methods share -> (the fused path's result, None, None), or (None, the sampled
        forward's log-prob outputs, the NLL summed over the samples) for the caller to assemble."""
        x2 = self._flat_input(input)
        params = [l.params() for l in self.layers()]
        est = self._est.with_gauss(self._gauss_priors())
        if self._het:
            self._check_no_sigma(sigma)
            target = self._het_target(target, x2.shape[0])
            if self.fused:
                return F._elbo(est, x2, target, beta, samples, self.sigma_min, self.mode, params, self.tf32,
                               self.likelihood), None, None
        elif self._fusable(x2, target):
            return F._elbo(est, x2, target, beta, samples, sigma, self.mode, params, self.tf32, 'gaussian'), \
                None, None
        outs, *lp = F._network_forward(est, x2, params, samples, True, True, self.tf32)
        negative_log_likelihood = torch.zeros(1, device=outs.device)
        for i in range(samples):
            negative_log_likelihood = negative_log_likelihood + self.get_nll(outs[i], target, sigma)
        return None, lp, negative_log_likelihood

    def sample_elbo(self, input, target, beta, samples, sigma=1.):
        ''' Sample ELBO for BNN w/o Local Reparameterisation (networks.py:192-209) '''
        assert self.local_reparam == False, 'sample_elbo() method returns loss for BNNs without local reparameterisation, alternatively use sample_elbo_lr()'
        fused, lp, negative_log_likelihood = self._sample_elbo(input, target, beta, samples, sigma)
        if fused is not None:
            return fused
        lps, lqs = lp
        log_prior = beta * lps.mean()
        log_variational_posterior = beta * lqs.mean()
        negative_log_likelihood = negative_log_likelihood / samples
        loss = log_variational_posterior - log_prior + negative_log_likelihood
        return loss, lps.mean(), lqs.mean(), negative_log_likelihood

    def sample_elbo_lr(self, input, target, beta, samples, sigma=1.):
        ''' Sample ELBO for BNN w/ Local Reparameterisation (networks.py:211-225) '''
        assert self.local_reparam == True, 'sample_elbo_lr() method returns loss for BNNs with local reparameterisation, alternatively use sample_elbo()'
        fused, lp, negative_log_likelihood = self._sample_elbo(input, target, beta, samples, sigma)
        if fused is not None:
            return fused
        kl, = lp
        negative_log_likelihood = negative_log_likelihood / samples
        loss = beta * kl + negative_log_likelihood
        return loss, kl, negative_log_likelihood


class MLP(nn.Module):
    """Non-Bayesian baseline (networks.py:227-253): stock torch.nn, kept so `from networks import MLP` works."""

    def __init__(self, model_params):
        super().__init__()
        self.input_shape = model_params['input_shape']
        self.classes = model_params['classes']
        self.batch_size = model_params['batch_size']
        self.hidden_units = model_params['hidden_units']
        self.mode = model_params['mode']
        self.net = nn.Sequential(nn.Linear(self.input_shape, self.hidden_units), nn.ReLU(),
                                 nn.Linear(self.hidden_units, self.hidden_units), nn.ReLU(),
                                 nn.Linear(self.hidden_units, self.classes))

    def forward(self, x):
        assert self.mode in {'regression', 'classification'}, 'MLP Mode must be either regression or classification'
        if self.mode == 'classification':
            x = x.view(-1, self.input_shape)
        return self.net(x)


class MLP_Dropout(nn.Module):
    """MC-dropout baseline (networks.py:255-285): stock torch.nn."""

    def __init__(self, model_params):
        super().__init__()
        self.input_shape = model_params['input_shape']
        self.classes = model_params['classes']
        self.batch_size = model_params['batch_size']
        self.hidden_units = model_params['hidden_units']
        self.mode = model_params['mode']
        self.net = nn.Sequential(nn.Linear(self.input_shape, self.hidden_units), nn.ReLU(),
                                 nn.Dropout(0.5),      # fixed, as the reference (networks.py:268,271); the callers'
                                 nn.Linear(self.hidden_units, self.hidden_units), nn.ReLU(),
                                 nn.Dropout(0.5),      # 'dropout' key is a boolean routing flag, not a probability
                                 nn.Linear(self.hidden_units, self.classes))

    def forward(self, x):
        assert self.mode in {'regression', 'classification'}, 'MLP Mode must be either regression or classification'
        if self.mode == 'classification':
            x = x.view(-1, self.input_shape)
        return self.net(x)

    def enable_dropout(self):
        ''' Enable the dropout layers during test-time '''
        for m in self.modules():
            if m.__class__.__name__.startswith('Dropout'):
                m.train()
