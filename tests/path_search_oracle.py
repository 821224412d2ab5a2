"""Search over paths (Ma et al.) restated in plain fp32 torch on the CPU: the specification the GPU's
SearchOverPaths is compared with in tests/test_search_over_paths.py (the reference has no such code).  Built on
the pinned oracle's UNet and ancestral step (oracle/ddpm_oracle.py); the round schedule is the package's own
`path_rounds`.  Test infrastructure only."""
from __future__ import annotations

import math
from typing import Callable, Optional, Sequence

import torch

from its_b200.search.search_algorithm import path_rounds
from oracle import ddpm_oracle as O

Tensor = torch.Tensor


def search_over_paths(sd, sched, x_T: Tensor, step_noise_fn: Callable[[int], Tensor],
                      forward_noise: Sequence[Tensor], N: int, M: int, s0: int, delta_f: int, delta_b: int,
                      verifier_fn, labels: Optional[Tensor] = None, w: float = 0.0, quant: Optional[str] = None):
    """Search over paths of Ma et al. (a beam of N partial trajectories, each survivor re-noised M times per round
    and pruned by top-k on x0 predictions).  x_T [N, *shape] are the initial paths, step_noise_fn(t) the
    Gaussians of time step t, forward_noise[round] [N*M, *shape] the re-noising draws.  The round schedule is the
    package's `path_rounds`.  Scoring uses x0 = clip(sqrt(1/abar_e) x_e - sqrt(1/abar_e - 1) eps_e, -1, 1) with
    eps_e the mixed eps of the segment's last UNet evaluation; the last round scores the clipped samples.
    Selection: score descending, first index on ties, NaN never ranks.
    Returns (best images, best score, history with per-round 'rounds', 'scores', 'survivors', 'lineage')."""
    T = sched["betas"].shape[0]
    abar = sched["alphas_bar"]
    rounds = path_rounds(T, s0, delta_f, delta_b)
    states = [O.sample(sd, sched, x, step_noise_fn, labels, w, quant, t_stop=s0 + 1, clip=False) if s0 < T - 1
              else x.clone() for x in x_T]
    parents = list(range(N))
    history = {"rounds": [], "scores": [], "survivors": []}
    for r, (s, sp, e) in enumerate(rounds):
        ratio = abar[sp] / abar[s]
        a, b = torch.sqrt(ratio).float(), torch.sqrt(1.0 - ratio).float()
        kids, scores = [], []
        for c in range(N * M):
            x_t = a * states[parents[c // M]] + b * forward_noise[r][c]
            eps = None
            x_in = x_t
            for time_step in range(sp, e - 1, -1):
                t = torch.full((x_t.shape[0],), time_step, dtype=torch.long)
                x_in = x_t
                mean, var, eps = O.p_mean_variance(sd, sched, x_t, t, labels, w, quant)
                x_t = mean + torch.sqrt(var) * step_noise_fn(time_step) if time_step > 0 else mean
                assert torch.isnan(x_t).int().sum() == 0, "nan in tensor."
            if e > 0:
                r1, r2 = torch.sqrt(1.0 / abar[e]).float(), torch.sqrt(1.0 / abar[e] - 1.0).float()
                judged = torch.clip(r1 * x_in - r2 * eps, -1, 1)
            else:
                x_t = torch.clip(x_t, -1, 1)
                judged = x_t
            kids.append(x_t)
            scores.append(float(verifier_fn(judged)))
        ranked = [c for c in range(N * M) if not math.isnan(scores[c]) and scores[c] != float("-inf")]
        order = sorted(ranked, key=lambda c: -scores[c])
        history["rounds"].append((s, sp, e))
        history["scores"].append(scores)
        if e > 0:
            if len(order) < N:
                raise ValueError("fewer than N children have a score that can be ranked")
            survivors = order[:N]
            history["survivors"].append(survivors)
            states, parents = kids, survivors
        else:
            if not order:
                raise ValueError("no finished sample has a score that can be ranked")
            best = order[0]
            history["survivors"].append([best])
    child, lineage = best, [best]
    for ids in reversed(history["survivors"][:-1]):
        child = ids[child // M]
        lineage.append(child)
    lineage.reverse()
    history["lineage"] = {"path": lineage[0] // M, "children": lineage}
    return kids[best], scores[best], history
