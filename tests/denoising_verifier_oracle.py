"""The denoising verifier restated in plain fp32 torch on the CPU: the specification the GPU's DenoisingVerifier is
compared with in tests/test_denoising_verifier.py (the reference has no such verifier).  Built on the pinned oracle's
UNet (oracle/ddpm_oracle.py) and Philox generator (oracle/philox.py).  Test infrastructure only."""
from __future__ import annotations

from typing import Optional

import torch

from oracle import ddpm_oracle as O
from oracle import philox

Tensor = torch.Tensor
X_T_TAG = 0x40000000
TAG_SCORE = X_T_TAG - 1


def levels(T: int, S: int):
    """t_s = ((2s + 1) T) // (2S): the midpoints of S equal strata of [0, T)."""
    if not 1 <= S <= T:
        raise ValueError(f"S={S} outside [1, T={T}]")
    return [((2 * s + 1) * T) // (2 * S) for s in range(S)]


def level_noise(seed: int, S: int, shape) -> Tensor:
    """eps_s [S, C, H, W]: Philox unit s under TAG_SCORE."""
    n_per = int(torch.Size(shape).numel())
    return torch.from_numpy(philox.normal(seed, 0, TAG_SCORE, S, n_per)).view(S, *shape)


def denoise_scores(sd, betas: Tensor, images: Tensor, per_cand: int, S: int, seed: int, kind: str = "likelihood",
                   labels: Optional[Tensor] = None, eps: Optional[Tensor] = None) -> Tensor:
    """[n_cand] fp32 scores of groups of `per_cand` consecutive images [n_img, C, H, W].
      likelihood: -D_c / count;  class: (D_u - D_c) / count,  count = per_cand * S * C * H * W,
    D = sum over the candidate's images b and levels s of (eps_hat(a_s x_b + b_s eps_s, t_s, y_b) - eps_s)^2, with
    y_b = `labels[b]` (conditional net), 0 for D_u, omitted for the unconditional net.  a_s = fp32(sqrt(abar_t)),
    b_s = fp32(sqrt(1 - abar_t)), abar = cumprod(1 - betas) in fp64.  Differences in fp32, squares and sums in
    double, rounded to fp32.  `eps` [S, C, H, W] replaces the Philox draws (same values up to the generator's
    last-bit differences between numpy and the device's fast math)."""
    T = betas.shape[0]
    ts = levels(T, S)
    abar = torch.cumprod(1. - betas.double(), dim=0)[ts]
    a, b = torch.sqrt(abar).float(), torch.sqrt(1. - abar).float()
    n_img = images.shape[0]
    if eps is None:
        eps = level_noise(seed, S, images.shape[1:])
    x = images.float()
    d_c = torch.zeros(n_img, dtype=torch.float64)
    d_u = torch.zeros(n_img, dtype=torch.float64)
    for s in range(S):
        x_s = a[s] * x + b[s] * eps[s]
        t = torch.full((n_img,), ts[s], dtype=torch.long)
        err = O.unet_forward(sd, x_s, t, labels) - eps[s]
        d_c += err.double().pow(2).flatten(1).sum(1)
        if kind == "class":
            err = O.unet_forward(sd, x_s, t, torch.zeros_like(labels)) - eps[s]
            d_u += err.double().pow(2).flatten(1).sum(1)
    d_c = d_c.view(-1, per_cand).sum(1)
    d_u = d_u.view(-1, per_cand).sum(1)
    count = per_cand * S * images[0].numel()
    score = (d_u - d_c) / count if kind == "class" else -d_c / count
    return score.float()
