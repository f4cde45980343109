"""nn.Module mirrors of the reference's L1/L2 classes (networks.py:14-138) on top of the CUDA kernels.

Same constructor signatures, Parameter names/shapes/initialisation, attributes and mode logic as the
reference, so state_dicts interchange and weight_pruning.py / logger_utils.py keep working.  The
arithmetic is in libbbb.so; these classes hold parameters and route calls.
"""
import math

import torch
from torch import nn

from . import functional as F
from . import _lib as L


class ScaleMixtureGaussian:
    """Scale-mixture prior (networks.py:14-27).  log_prob runs the single-pass reduction kernel."""

    def __init__(self, pi, sigma1, sigma2):
        self.pi, self.sigma1, self.sigma2 = pi, sigma1, sigma2
        self._prior = L.Prior(L.PRIOR_MIXTURE, float(pi), float(sigma1), float(sigma2))

    def log_prob(self, input):
        z = torch.full_like(input, -80.0)          # softplus(-80) * 0 = 0 => w = input
        lp, _, _ = F.logprob_reduce(input, z, self._prior, sample=False)
        return lp.to(torch.float32)


class GaussianNode:
    """Variational posterior node over a (mu, rho) pair (networks.py:29-46)."""

    def __init__(self, mu, rho):
        self.mu, self.rho = mu, rho

    @property
    def sigma(self):
        return torch.log1p(torch.exp(self.rho))

    def sample(self):
        """mu + sigma * eps with eps from the configured eps source (Philox, or the reference's
        CPU draw in 'reference' mode).  Not on the hot path: the layers fuse sampling into the GEMM."""
        from . import rng as R
        if R.get_eps_mode() == 'reference':
            eps = R.draw_reference_eps(self.rho.size(), self.rho.device)
        else:
            seed, step = R.next_step()
            eps = F.philox_normal(self.rho.numel(), self.rho.device, seed, step).view(self.rho.size())
        return self.mu + self.sigma * eps

    def log_prob(self, input):
        return (-math.log(math.sqrt(2 * math.pi)) - torch.log(self.sigma)
                - ((input - self.mu) ** 2) / (2 * self.sigma ** 2)).sum()


PRIOR_BUFFERS = ('prior_weight_mu', 'prior_weight_rho', 'prior_bias_mu', 'prior_bias_rho')


def _register_prior_buffers(layer):
    """The optional per-weight Gaussian prior N(prior_mu, softplus(prior_rho)^2) of a layer, in the posterior's own
    parametrisation and layout.  Not persistent: the state_dict keeps the reference's keys."""
    for name in PRIOR_BUFFERS:
        layer.register_buffer(name, None, persistent=False)


def gauss_prior(layer):
    """(weight m, weight r, bias m, bias r) of the layer's per-weight prior, or None."""
    bufs = tuple(getattr(layer, name) for name in PRIOR_BUFFERS)
    return None if bufs[0] is None else bufs


class BayesianLinear(nn.Module):
    """Weight-sampling Bayesian FC layer (networks.py:48-88)."""

    def __init__(self, in_features, out_features, mu_init, rho_init, prior_init, mixture_prior=True):
        super().__init__()
        self.weight_mu = nn.Parameter(torch.Tensor(out_features, in_features).uniform_(*mu_init))
        self.weight_rho = nn.Parameter(torch.Tensor(out_features, in_features).uniform_(*rho_init))
        self.weight = GaussianNode(self.weight_mu, self.weight_rho)
        self.bias_mu = nn.Parameter(torch.Tensor(out_features).uniform_(*mu_init))
        self.bias_rho = nn.Parameter(torch.Tensor(out_features).uniform_(*rho_init))
        self.bias = GaussianNode(self.bias_mu, self.bias_rho)
        self._prior = F.make_prior(prior_init, mixture_prior)      # asserts like networks.py:62,66
        if mixture_prior:
            self.weight_prior = ScaleMixtureGaussian(prior_init[0], math.exp(prior_init[1]), math.exp(prior_init[2]))
            self.bias_prior = ScaleMixtureGaussian(prior_init[0], math.exp(prior_init[1]), math.exp(prior_init[2]))
        else:
            self.weight_prior = torch.distributions.Normal(0, prior_init[0])
            self.bias_prior = torch.distributions.Normal(0, prior_init[0])
        self.log_prior = 0
        self.log_variational_posterior = 0
        self.layer_id = 0          # Philox tensor-id base; BayesianNetwork numbers its layers
        self.tf32 = False
        _register_prior_buffers(self)

    def params(self):
        return (self.weight_mu, self.weight_rho, self.bias_mu, self.bias_rho)

    def forward(self, input, sample=False, calculate_log_probs=False):
        do_sample = self.training or sample
        do_logp = self.training or calculate_log_probs
        y, lp, lq = F.bayes_linear(input, *self.params(), self._prior, do_sample, do_logp, self.layer_id, self.tf32,
                                   gauss_prior(self))
        if do_logp:
            self.log_prior, self.log_variational_posterior = lp, lq
        else:
            self.log_prior, self.log_variational_posterior = 0, 0
        return y


class BayesianLinearLR(nn.Module):
    """Local-reparameterisation Bayesian FC layer (networks.py:90-138); weights are [in, out]."""

    def __init__(self, in_features, out_features, mu_init, rho_init, prior_init, mixture_prior=False):
        super().__init__()
        self.weight_mu = nn.Parameter(torch.Tensor(in_features, out_features).uniform_(*mu_init))
        self.weight_rho = nn.Parameter(torch.Tensor(in_features, out_features).uniform_(*rho_init))
        self.bias_mu = nn.Parameter(torch.Tensor(out_features).uniform_(*mu_init))
        self.bias_rho = nn.Parameter(torch.Tensor(out_features).uniform_(*rho_init))
        assert len(prior_init) == 1, "Gaussian Prior requires one value in prior initialisation"
        self.weight_prior = [0, prior_init[0]]
        self.bias_prior = [0, prior_init[0]]
        self.weight_kl_cost = 0
        self.bias_kl_cost = 0
        self.kl_cost = 0
        self.layer_id = 0
        _register_prior_buffers(self)

    def params(self):
        return (self.weight_mu, self.weight_rho, self.bias_mu, self.bias_rho)

    def compute_kl_cost(self, p_params, q_params):
        """Closed-form KL between two Gaussians (networks.py:109-114); q_sigma given directly."""
        [p_mu, p_sigma] = p_params
        [q_mu, q_sigma] = q_params
        return 0.5 * (2 * torch.log(p_sigma / q_sigma) - 1 + (q_sigma / p_sigma).pow(2)
                      + ((p_mu - q_mu) / p_sigma).pow(2)).sum()

    def forward(self, input, sample=False, calculate_log_probs=False):
        # The reference's eval branch crashes (self.b_mu, networks.py:131) and its calculate_log_probs
        # without sampling reads an undefined w_sigma (networks.py:134); both are fixed here (SURVEY B-4).
        do_sample = self.training or sample
        do_kl = self.training or calculate_log_probs
        y, kl = F.lr_linear(input, *self.params(), self.weight_prior[1], do_sample, do_kl, self.layer_id,
                            gauss_prior(self))
        if do_kl:
            self.kl_cost = kl
        return y
