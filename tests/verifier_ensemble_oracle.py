"""The rank-ensemble rule of its_rank_ensemble in numpy float64, stated by pairwise counting.

scores [n_seg * seg_len, V] (candidate-major, one column per member), weights [V] finite and > 0.  In each segment a
candidate is eligible when none of its V scores is NaN or -inf; over the eligible set E,
  r_v(i) = |{j in E : S[j][v] < S[i][v]}| + |{j in E, j != i : S[j][v] == S[i][v]}| / 2
  out_i  = (sum_v w_v r_v(i)) / ((sum_v w_v) (|E| - 1))   (float64, member order), rounded to fp32; 1 when |E| = 1
and NaN for an ineligible candidate."""
import numpy as np


def eligible(scores: np.ndarray) -> np.ndarray:
    s = np.asarray(scores, dtype=np.float32)
    return ~(np.isnan(s) | (s == -np.inf)).any(axis=1)


def average_ranks(x: np.ndarray) -> np.ndarray:
    """Average ranks from 0 of the values x (none NaN or -inf), by counting."""
    x = np.asarray(x, dtype=np.float32)
    less = (x[None, :] < x[:, None]).sum(axis=1)
    ties = (x[None, :] == x[:, None]).sum(axis=1) - 1
    return less.astype(np.float64) + 0.5 * ties.astype(np.float64)


def rank_ensemble(scores, weights, n_seg: int) -> np.ndarray:
    s = np.asarray(scores, dtype=np.float32)
    w = np.asarray(weights, dtype=np.float32).astype(np.float64)
    n, V = s.shape
    assert w.shape == (V,) and n % n_seg == 0
    seg_len = n // n_seg
    out = np.full(n, np.nan, dtype=np.float32)
    for q in range(n_seg):
        seg = s[q * seg_len:(q + 1) * seg_len]
        ok = eligible(seg)
        n_ok = int(ok.sum())
        if n_ok == 0:
            continue
        if n_ok == 1:
            out[q * seg_len + np.flatnonzero(ok)] = 1.0
            continue
        num = np.zeros(n_ok, dtype=np.float64)
        wsum = 0.0
        for v in range(V):
            num = num + w[v] * average_ranks(seg[ok, v])
            wsum = wsum + w[v]
        out[q * seg_len + np.flatnonzero(ok)] = (num / (wsum * float(n_ok - 1))).astype(np.float32)
    return out
