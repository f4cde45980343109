"""CPU oracle of the per-weight Gaussian prior p(w_i) = N(m_i, softplus(r_i)^2).  TEST INFRASTRUCTURE ONLY.

A float64 restatement of the two prior terms the ELBO takes from a per-weight prior, written so that torch autograd
gives their gradients:
  * weight sampling (networks.py:41-46, 81-83, 192-209 with the prior's log_prob per weight): the Monte Carlo
    log p(w_s) and log q(w_s) of w_s = mu + softplus(rho) eps_s, given eps;
  * local reparameterisation: the closed-form KL(q || p) of networks.py:109-114 (compute_kl_cost) with p_mu = m,
    which the reference always calls with p_mu = 0.
A layer's tensors are plain tensors; eps is [S, *mu.shape].
"""
import math

import torch

from .bbb_oracle import softplus

LOG_SQRT_2PI = math.log(math.sqrt(2 * math.pi))


def _normal_log_prob(x, mean, scale):
    return -LOG_SQRT_2PI - torch.log(scale) - ((x - mean) ** 2) / (2 * scale ** 2)


def logprob(mu, rho, prior_mu, prior_rho, eps):
    """Per sample s: (sum log N(w_s; m, sp^2), sum log N(w_s; mu, sigma^2)) with w_s = mu + softplus(rho) eps_s and
    sp = softplus(prior_rho); two [S] tensors."""
    sigma, sp = softplus(rho), softplus(prior_rho)
    w = mu + sigma * eps
    dims = tuple(range(1, eps.dim()))
    lp = _normal_log_prob(w, prior_mu, sp)
    lq = _normal_log_prob(w, mu, sigma)
    return (lp.sum(dims), lq.sum(dims)) if dims else (lp, lq)


def kl(mu, rho, prior_mu, prior_rho):
    """compute_kl_cost(p_params=(m, sp), q_params=(mu, sigma)) of networks.py:109-114:
    0.5 sum (2 log(sp / sigma) - 1 + (sigma / sp)^2 + ((m - mu) / sp)^2)."""
    p_sigma, q_sigma = softplus(prior_rho), softplus(rho)
    return 0.5 * (2 * torch.log(p_sigma / q_sigma) - 1 + (q_sigma / p_sigma).pow(2)
                  + ((prior_mu - mu) / p_sigma).pow(2)).sum()


def sigma_to_rho(sigma):
    """The inverse of softplus, log(expm1(sigma)), in float64."""
    s = torch.as_tensor(sigma, dtype=torch.float64)
    return s + torch.log(-torch.expm1(-s))
