"""Unconditional DDPM ancestral sampler with the reference's surface
(Diffusion/Diffusion.py:50-102): GaussianDiffusionSampler(model, beta_1, beta_T, T)
with fp64 buffers betas / coeff1 / coeff2 / posterior_var, the public seam
p_mean_variance(x_t, t) -> (mean, var) (driven externally by the reference's own
Diffusion/Train.py:68-77), predict_xt_prev_mean_from_eps, and forward(x_T).
The training-side GaussianDiffusionTrainer (:19-47) is out of scope.
"""
from __future__ import annotations

import torch

from .._sampler_base import SamplerBase, extract  # noqa: F401  (extract is part of the module's surface)


class GaussianDiffusionSampler(SamplerBase):
    guided = False

    def __init__(self, model, beta_1, beta_T, T):
        super().__init__()
        self._init_schedule(model, beta_1, beta_T, T)

    def p_mean_variance(self, x_t, t):
        var = self._variance(x_t, t)
        eps = self.model(x_t, t)
        return self.predict_xt_prev_mean_from_eps(x_t, t, eps=eps), var

    def forward(self, x_T, *, noise=None, seed=None, cand_id0=0, t_start=None, clip=True, t_stop=0):
        """Algorithm 2 (Diffusion.py:84-102): T fused steps on the device, then
        clip to [-1, 1].  The steps replay the sampler's captured step graph,
        which `segment` shares; the candidate base is read from device memory,
        so a new `cand_id0` replays the same graph.  Extensions (keyword-only,
        defaults = reference behaviour): `noise` [T, *x_T.shape] injects the
        per-step Gaussians (entry t at time_step t, for parity runs); otherwise
        they come from the in-kernel Philox stream `seed` keyed by candidate id
        `cand_id0 + b`; `t_start` begins the loop at an intermediate step (search
        over paths) and `t_stop` ends it early (metrics tracking), returning the
        unclipped x_{t_stop-1}."""
        return self._run(x_T, None, t_start=t_start, t_stop=t_stop, seed=seed, cand_id0=cand_id0, noise=noise,
                         clip=clip, want_x0=False, check_nan=True)[0]
