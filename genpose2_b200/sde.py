"""VE SDE of networks/gf_algorithms/sde.py (lines 15-34, 96-119).  Only `sde_mode == "ve"` is on the
hot path (configs/config.py:31, scripts/eval_*.sh); VP / sub-VP / EDM raise NotImplementedError.

These host-side callables exist so that code written against the reference keeps working
(`prior_fn`, `marginal_prob_fn`, `sde_fn` are handed around by PoseNet / GFObjectPose); the kernels
evaluate sigma(t) and g(t) on the device themselves.
"""
import functools

import numpy as np
import torch

SIGMA_MIN = 0.01
SIGMA_MAX = 50.0
SAMPLING_EPS = 1e-5


def ve_marginal_prob(x, t, sigma_min=0.01, sigma_max=90):
    std = sigma_min * (sigma_max / sigma_min) ** t
    return x, std


def ve_sde(t, sigma_min=0.01, sigma_max=90):
    sigma = sigma_min * (sigma_max / sigma_min) ** t
    drift_coeff = torch.tensor(0)
    diffusion_coeff = sigma * torch.sqrt(
        torch.tensor(2 * (np.log(sigma_max) - np.log(sigma_min)), device=t.device))
    return drift_coeff, diffusion_coeff


def ve_prior(shape, sigma_min=0.01, sigma_max=90, T=1.0):
    """CPU generator, exactly like the reference (sde.py:30-34): seeding `torch.manual_seed`
    reproduces the reference's initial noise."""
    _, sigma_max_prior = ve_marginal_prob(None, T, sigma_min=sigma_min, sigma_max=sigma_max)
    return torch.randn(*shape) * sigma_max_prior


def prior_std(T):
    """sigma(T) of the prior that init_sde's prior_fn draws from, as a Python float (ve_marginal_prob)."""
    return ve_marginal_prob(None, T, sigma_min=SIGMA_MIN, sigma_max=SIGMA_MAX)[1]


def init_sde(sde_mode):
    if sde_mode != "ve":
        raise NotImplementedError(
            f"sde_mode={sde_mode!r}: only the VE SDE is on the accelerated path (no fallback)")
    prior_fn = functools.partial(ve_prior, sigma_min=SIGMA_MIN, sigma_max=SIGMA_MAX)
    marginal_prob_fn = functools.partial(ve_marginal_prob, sigma_min=SIGMA_MIN, sigma_max=SIGMA_MAX)
    sde_fn = functools.partial(ve_sde, sigma_min=SIGMA_MIN, sigma_max=SIGMA_MAX)
    return prior_fn, marginal_prob_fn, sde_fn, SAMPLING_EPS, 1.0
