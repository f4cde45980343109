"""bayesian-neural-network_b200: the Bayes-by-Backprop hot path of tennisonliu/bayesian-neural-network
as hand-written sm_100a CUDA kernels (csrc/, C ABI in include/bbb.h) behind the reference's own
networks.py API.  Import it as `bnn_b200` (bnn_b200.py at the repo root aliases this directory, whose
name is not a Python identifier) or through the drop-in top-level `networks` module."""
from . import _lib, rng, functional, parallel
from .rng import set_eps_mode, get_eps_mode, manual_seed, eps_mode, set_sample_base, use_device_step
from .layers import ScaleMixtureGaussian, GaussianNode, BayesianLinear, BayesianLinearLR
from .network import BayesianNetwork, PredictiveResult, MLP, MLP_Dropout
from .optim import FusedAdam, PeerShardedAdam
from .graphed import GraphedTrainStep
from .bandit import ReplayRing, GraphedBanditUpdate, reference_idx_pool, make_bandit_update

__all__ = ['ScaleMixtureGaussian', 'GaussianNode', 'BayesianLinear', 'BayesianLinearLR', 'BayesianNetwork',
           'PredictiveResult', 'MLP', 'MLP_Dropout', 'set_eps_mode', 'get_eps_mode', 'manual_seed', 'eps_mode',
           'set_sample_base', 'use_device_step', 'functional', 'rng', 'parallel', 'FusedAdam', 'PeerShardedAdam', 'GraphedTrainStep',
           'ReplayRing', 'GraphedBanditUpdate', 'reference_idx_pool', 'make_bandit_update']
