"""Search over the guidance weight restated in plain fp32 torch on the CPU: the specification RandomSearch and
FKSteering with per-candidate `guidance` are compared with in tests/test_guidance_search.py.  Candidate i runs the
pinned oracle's guided ancestral loop (oracle/ddpm_oracle.py) at its own weight; an FK particle takes its ancestor's
weight at every resampling (the resampling rule is tests/fk_steering_oracle.py's).  Test infrastructure only."""
from __future__ import annotations

import math
from typing import Callable, Optional, Sequence

import numpy as np
import torch

from its_b200.search.search_algorithm import fk_segments
from oracle import ddpm_oracle as O
from tests.fk_steering_oracle import resample

Tensor = torch.Tensor


def random_search(sd, sched, x_T: Tensor, step_noise_fn: Callable[[int], Tensor], guidance: Sequence[float],
                  verifier_fn, labels: Tensor, quant: Optional[str] = None):
    """Candidate i: x_T[i] denoised at weight guidance[i], scored on the clipped sample; the first maximum wins.
    Returns (best index, best score, scores)."""
    scores = []
    for i in range(x_T.shape[0]):
        img = O.sample(sd, sched, x_T[i], step_noise_fn, labels, float(guidance[i]), quant)
        scores.append(float(np.float32(verifier_fn(img))))
    ranked = [i for i, s in enumerate(scores) if not math.isnan(s) and s != -math.inf]
    best = max(ranked, key=lambda i: (scores[i], -i))
    return best, scores[best], scores


def fk_steering(sd, sched, x_T: Tensor, step_noise_fn: Callable[[int], Tensor], guidance: Sequence[float],
                start_step: int, interval: int, lam: float, seed: int, verifier_fn, labels: Tensor,
                quant: Optional[str] = None):
    """FK steering of one query (tests/fk_steering_oracle.fk_steering) with particle p at weight g[p]: after every
    resampling, g = g[ancestors].  Returns (best images, best score, history with 'segments', per-resampling
    'scores', 'ancestors', 'ess' and 'margin', 'lineage' and 'lineage_guidance')."""
    T = sched["betas"].shape[0]
    abar = sched["alphas_bar"]
    N = x_T.shape[0]
    parts = [x.clone() for x in x_T]
    g = [float(v) for v in guidance]
    carried = None
    segments = fk_segments(T, start_step, interval)
    history = {"segments": segments, "scores": [], "ancestors": [], "ess": [], "margin": [], "guidance": []}
    for r, (t_start, t_stop) in enumerate(segments):
        history["guidance"].append(list(g))
        scores = []
        for p in range(N):
            x_t = parts[p]
            for time_step in range(t_start, t_stop - 1, -1):
                t = torch.full((x_t.shape[0],), time_step, dtype=torch.long)
                x_in = x_t
                mean, var, eps = O.p_mean_variance(sd, sched, x_t, t, labels, g[p], quant)
                x_t = mean + torch.sqrt(var) * step_noise_fn(time_step) if time_step > 0 else mean
            if t_stop > 0:
                r1, r2 = torch.sqrt(1.0 / abar[t_stop]).float(), torch.sqrt(1.0 / abar[t_stop] - 1.0).float()
                judged = torch.clip(r1 * x_in - r2 * eps, -1, 1)
            else:
                x_t = torch.clip(x_t, -1, 1)
                judged = x_t
            parts[p] = x_t
            scores.append(float(np.float32(verifier_fn(judged))))
        if t_stop == 0:
            break
        anc, carried, ess, margin = resample(scores, carried, lam, 1, seed, r)
        history["scores"].append(scores)
        history["ancestors"].append(anc.tolist())
        history["ess"].append(float(ess[0]))
        history["margin"].append(margin)
        parts = [parts[i] for i in anc]
        g = [g[i] for i in anc]
    ranked = [p for p in range(N) if not math.isnan(scores[p]) and scores[p] != -math.inf]
    best = max(ranked, key=lambda p: (scores[p], -p))
    j, lineage = best, [best]
    for anc in reversed(history["ancestors"]):
        j = anc[j]
        lineage.append(j)
    history["lineage"] = lineage[::-1]
    history["lineage_guidance"] = [history["guidance"][r][j] for r, j in enumerate(history["lineage"])]
    history["final_scores"] = scores
    return parts[best], scores[best], history
