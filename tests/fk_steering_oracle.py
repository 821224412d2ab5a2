"""Feynman-Kac steering (Singhal et al. 2025) restated in numpy float64 and plain fp32 torch on the CPU: the
specification the GPU's its_resample_systematic and FKSteering are compared with in tests/test_fk_steering.py (the
reference has no such code).  Built on the pinned oracle's UNet and ancestral step (oracle/ddpm_oracle.py) and its
Philox restatement (oracle/philox.py); the segment schedule is the package's own `fk_segments`.  Test
infrastructure only."""
from __future__ import annotations

import math
from typing import Callable, Optional

import numpy as np
import torch

from its_b200.search.search_algorithm import fk_segments
from oracle import ddpm_oracle as O
from oracle import philox

Tensor = torch.Tensor
X_T_TAG = 0x40000000
TAG_RESAMPLE = X_T_TAG + 2


def uniform(seed: int, segment: int, round: int, tag: int = TAG_RESAMPLE) -> float:
    """The one uniform of (seed, segment, round): 53 bits of Philox4x32-10 at counter
    {segment, round lo, tag, round hi} under key {seed lo, seed hi}."""
    ctr = np.array([segment & 0xFFFFFFFF, round & 0xFFFFFFFF, tag & 0xFFFFFFFF, (round >> 32) & 0xFFFFFFFF],
                   dtype=np.uint32)
    key = np.array([seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF], dtype=np.uint32)
    c = philox.philox4x32_10(ctr, key)
    return ((int(c[0]) >> 5) * 2.0 ** 26 + (int(c[1]) >> 6)) * 2.0 ** -53


def weights(reward, carried, lam: float) -> np.ndarray:
    """w_i = exp(l_i - m) in float64, l_i = lam * (reward_i - carried_i) in float32; 0 where reward_i or l_i is
    not finite; all 0 when no l_i is finite."""
    r = np.asarray(reward, dtype=np.float32)
    c = np.zeros_like(r) if carried is None else np.asarray(carried, dtype=np.float32)
    with np.errstate(invalid="ignore", over="ignore"):
        l = np.float32(lam) * (r - c)
    ok = np.isfinite(r) & np.isfinite(l)
    w = np.zeros(r.shape, dtype=np.float64)
    if ok.any():
        w[ok] = np.exp(l[ok].astype(np.float64) - float(l[ok].max()))
    return w


def resample(reward, carried, lam: float, n_seg: int, seed: int, round: int, tag: int = TAG_RESAMPLE):
    """Systematic resampling per segment: child j takes the smallest i with C_i > (u + j) / seg_len * C_last.
    Returns (flat ancestors int64, carried rewards float32, ESS per segment, margin): `margin` is the smallest
    distance of a position from a cumulative sum, relative to C_last (inf where a segment has no weight), the
    room a reordered double sum has before it could choose another ancestor."""
    r = np.asarray(reward, dtype=np.float32)
    seg = r.size // n_seg
    anc = np.full(r.size, -1, dtype=np.int64)
    out = np.full(r.size, np.nan, dtype=np.float32)
    ess = np.zeros(n_seg)
    margin = math.inf
    for s in range(n_seg):
        sl = slice(s * seg, (s + 1) * seg)
        w = weights(r[sl], None if carried is None else np.asarray(carried, dtype=np.float32)[sl], lam)
        if not (w > 0).any():
            continue
        C = np.cumsum(w)
        pos = (uniform(seed, s, round, tag) + np.arange(seg)) / seg * C[-1]
        i = np.minimum(np.searchsorted(C, pos, side="right"), int(np.nonzero(w > 0)[0][-1]))
        anc[sl] = s * seg + i
        out[sl] = r[sl][i]
        ess[s] = w.sum() ** 2 / (w * w).sum()
        margin = min(margin, float(np.abs(pos[:, None] - C[None, :]).min() / C[-1]))
    return anc, out, ess, margin


def fk_steering(sd, sched, x_T: Tensor, step_noise_fn: Callable[[int], Tensor], N: int, start_step: int,
                interval: int, lam: float, seed: int, verifier_fn, labels: Optional[Tensor] = None, w: float = 0.0,
                quant: Optional[str] = None):
    """FK steering of one query: N particles x_T [N, *shape] denoised by the ancestral loop with the Gaussians
    step_noise_fn(t) of time step t; after every segment of `fk_segments` but the last, each particle is scored on
    x0 = clip(sqrt(1/abar_e) x_e - sqrt(1/abar_e - 1) eps_e, -1, 1) (eps_e the mixed eps of the segment's last UNet
    evaluation) and the population is resampled with lam * (reward - carried reward).  The last segment scores the
    clipped samples; the winner is the first maximum (NaN never wins).
    Returns (best images, best score, history with 'segments', per-resampling 'scores', 'ancestors', 'ess' and
    'margin', and 'lineage')."""
    T = sched["betas"].shape[0]
    abar = sched["alphas_bar"]
    segments = fk_segments(T, start_step, interval)
    parts = [x.clone() for x in x_T]
    carried = None
    history = {"segments": segments, "scores": [], "ancestors": [], "ess": [], "margin": []}
    for r, (t_start, t_stop) in enumerate(segments):
        scores = []
        for p in range(N):
            x_t = parts[p]
            for time_step in range(t_start, t_stop - 1, -1):
                t = torch.full((x_t.shape[0],), time_step, dtype=torch.long)
                x_in = x_t
                mean, var, eps = O.p_mean_variance(sd, sched, x_t, t, labels, w, quant)
                x_t = mean + torch.sqrt(var) * step_noise_fn(time_step) if time_step > 0 else mean
                assert torch.isnan(x_t).int().sum() == 0, "nan in tensor."
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
        if anc[0] < 0:
            raise ValueError(f"resampling round {r}: no particle has a finite score")
        history["scores"].append(scores)
        history["ancestors"].append(anc.tolist())
        history["ess"].append(float(ess[0]))
        history["margin"].append(margin)
        parts = [parts[i] for i in anc]
    ranked = [p for p in range(N) if not math.isnan(scores[p]) and scores[p] != -math.inf]
    if not ranked:
        raise ValueError("no finished sample has a score that can be ranked")
    best = max(ranked, key=lambda p: (scores[p], -p))
    j, lineage = best, [best]
    for anc in reversed(history["ancestors"]):
        j = anc[j]
        lineage.append(j)
    history["lineage"] = lineage[::-1]
    history["final_scores"] = scores
    return parts[best], scores[best], history
