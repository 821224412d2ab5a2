"""Classifier-free-guidance DDPM sampler with the reference's surface
(DiffusionFreeGuidence/DiffusionCondition.py:56-105): GaussianDiffusionSampler(
model, beta_1, beta_T, T, w=0.) with .w, p_mean_variance(x_t, t, labels),
forward(x_T, labels).  The conditional and unconditional evaluations of each step
run as ONE 2B-image UNet pass (no cross-sample op exists, so this is the same
arithmetic as the reference's two calls, :83-84); the guidance mix
(1+w)*eps - w*nonEps (:85) is fused into the DDPM step kernel.
"""
from __future__ import annotations

import torch

from .._sampler_base import SamplerBase, extract  # noqa: F401


class GaussianDiffusionSampler(SamplerBase):
    guided = True

    def __init__(self, model, beta_1, beta_T, T, w=0.):
        super().__init__()
        self.w = w
        self._init_schedule(model, beta_1, beta_T, T)

    def p_mean_variance(self, x_t, t, labels):
        var = self._variance(x_t, t)
        net = self._unet()
        B = x_t.shape[0]
        both = net(torch.cat([x_t, x_t]), torch.cat([t, t]), torch.cat([labels, torch.zeros_like(labels)]))
        eps, non_eps = both[:B], both[B:]
        eps = (1. + self.w) * eps - self.w * non_eps
        return self.predict_xt_prev_mean_from_eps(x_t, t, eps=eps), var

    def forward(self, x_T, labels, *, noise=None, seed=None, cand_id0=0, t_start=None, clip=True, t_stop=0):
        """Algorithm 2 with guidance (DiffusionCondition.py:89-105), replaying the
        sampler's captured step graph as the unconditional sampler does.
        Keyword-only extensions as in the unconditional sampler."""
        return self._run(x_T, labels, t_start=t_start, t_stop=t_stop, seed=seed, cand_id0=cand_id0, noise=noise,
                         clip=clip, want_x0=False, check_nan=True)[0]
