"""Verifiers with the reference's surface (search/verifier.py): OracleVerifier
(:30-66), SelfSupervisedVerifier (:191-248), AestheticPredictor (:251-287), each
`.score(images, ...) -> float`.  Scores are computed by the warp-shuffle
reduction kernels of libits_b200 (its_image_stats / its_candidate_scores); the
extra `.score_candidates(images, per_cand)` returns one score per candidate as a
device tensor so a whole population is scored without a host round-trip.
EnsembleVerifier combines several of them by each candidate's rank within its
query's population (its_rank_ensemble).

SupervisedVerifier, CLIPScore and IntegratedVerifier (:69-188, :290-388) wrap
openai-CLIP, which is not installed and whose weights cannot be fetched: parity
unpinned, kept importable, raise at construction when `clip` is missing.
"""
from __future__ import annotations

from typing import Any, Dict, List, Optional

import numpy as np
import torch

from .. import _lib
from .._sampler_base import X_T_TAG

KIND_ORACLE, KIND_AESTHETIC, KIND_SELFSUP = 0, 1, 2


def _stats(images: torch.Tensor, want_feats: bool):
    _lib.require_cuda()
    if images.device.type != "cuda":
        raise RuntimeError("its_b200 verifiers run on CUDA only (no CPU fallback)")
    if images.dim() != 4:
        raise ValueError(f"expected images [B,C,H,W], got {tuple(images.shape)}")
    x = images.detach().to(torch.float32).contiguous()
    n, c, h, w = x.shape
    stats = torch.empty((n, 4), dtype=torch.float32, device=x.device)
    feats = torch.empty((n, c * 64), dtype=torch.float32, device=x.device) if want_feats else None
    L = _lib.lib()
    with torch.cuda.device(x.device):
        _lib.check(L.its_image_stats(stats.data_ptr(), feats.data_ptr() if want_feats else None, x.data_ptr(),
                                     n, c, h, w, _lib.stream_ptr(x.device)), "its_image_stats")
    return stats, feats


def candidate_scores(images: torch.Tensor, per_cand: int, kind: int) -> torch.Tensor:
    """One fp32 score per group of `per_cand` consecutive images (device tensor)."""
    n = images.shape[0]
    if per_cand <= 0 or n % per_cand:
        raise ValueError(f"{n} images do not split into candidates of {per_cand}")
    stats, feats = _stats(images, kind == KIND_SELFSUP)
    scores = torch.empty((n // per_cand,), dtype=torch.float32, device=images.device)
    L = _lib.lib()
    with torch.cuda.device(images.device):
        _lib.check(L.its_candidate_scores(scores.data_ptr(), stats.data_ptr(),
                                          feats.data_ptr() if feats is not None else None, n // per_cand,
                                          per_cand, images.shape[1] * 64, kind, _lib.stream_ptr(images.device)),
                   "its_candidate_scores")
    return scores


class _KernelVerifier:
    kind = KIND_ORACLE
    uses_labels = False     # True: the searches pass `labels=` (flat, one per image) to score_candidates

    def score_candidates(self, images: torch.Tensor, per_cand: int) -> torch.Tensor:
        return candidate_scores(images, per_cand, self.kind)


class OracleVerifier(_KernelVerifier):
    """Variance heuristic 1/(1+mean_b var(img_b)) when no dataset statistics are
    given (verifier.py:60-63); with statistics the reference's stub returns
    mean(images) (:65-66)."""
    kind = KIND_ORACLE

    def __init__(self, dataset_stats: Optional[Dict[str, np.ndarray]] = None):
        self.dataset_stats = dataset_stats

    def score(self, images: torch.Tensor, labels: Optional[torch.Tensor] = None) -> float:
        if self.dataset_stats is None:
            return float(self.score_candidates(images, images.shape[0]).item())
        stats, _ = _stats(images, False)
        return float(stats[:, 0].mean().item())   # equal-sized images: mean of means == global mean


class SelfSupervisedVerifier(_KernelVerifier):
    """Mean off-diagonal cosine similarity of L2-normalised 8x8 average-pooled
    images (verifier.py:207-248)."""
    kind = KIND_SELFSUP

    def __init__(self, denoising_features: Optional[torch.Tensor] = None):
        self.denoising_features = denoising_features

    def extract_features(self, images: torch.Tensor) -> torch.Tensor:
        """Un-normalised pooled features [B, C*64] (verifier.py:218-221)."""
        stats, feats = _stats(images, True)
        return feats * stats[:, 3:4]

    def score(self, images: torch.Tensor, reference_features: Optional[torch.Tensor] = None) -> float:
        if reference_features is None:
            return float(self.score_candidates(images, images.shape[0]).item())
        _, feats = _stats(images, True)                      # already normalised
        ref = torch.nn.functional.normalize(reference_features.to(feats), dim=-1)
        return torch.sum(feats * ref, dim=-1).item()         # raises for B > 1, like the reference


class AestheticPredictor(_KernelVerifier):
    """Contrast heuristic: 2 * mean_b std(img_b), on (x+1)/2 when the batch
    minimum is negative (verifier.py:277-287)."""
    kind = KIND_AESTHETIC

    def __init__(self, device: str = 'cuda'):
        self.device = device
        self.model = None

    def score(self, images: torch.Tensor) -> float:
        return float(self.score_candidates(images, images.shape[0]).item())


TAG_SCORE = X_T_TAG - 1     # noise of the denoising verifier: above every time step, below the search tags


def score_levels(T: int, n_levels: int) -> List[int]:
    """t_s = ((2s + 1) T) // (2S), s < S: the midpoints of S equal strata of [0, T)."""
    T, S = int(T), int(n_levels)
    if not 1 <= S <= T:
        raise ValueError(f"n_levels={n_levels} outside [1, T={T}]")
    return [((2 * s + 1) * T) // (2 * S) for s in range(S)]


class _ScoreGraph:
    """One plan's scoring graph {its_level_inputs, plan.run(), its_denoise_scores} and the buffers it points into."""

    def __init__(self, plan, tables, x: torch.Tensor, t_rows: torch.Tensor, scores: torch.Tensor):
        self.plan, self.tables = plan, tables    # holding them keeps the pointers the graph bakes in alive
        self.x, self.t_rows, self.scores = x, t_rows, scores
        self.graph: Optional[torch.cuda.CUDAGraph] = None


class DenoisingVerifier(_KernelVerifier):
    """The diffusion model as its own verifier (not in the reference).  Each image x is noised to S levels
    t_s (`score_levels`) with Gaussians eps_s common to every image (Philox unit s under TAG_SCORE and `seed`),
    x_s = sqrt(abar_t) x + sqrt(1 - abar_t) eps_s, and the UNet predicts eps_s back:
      kind="likelihood": score = -mean (eps_hat(x_s, t_s, y) - eps_s)^2  (the eps-prediction loss, Ho et al. 2020:
                         a Monte-Carlo estimate of the denoising ELBO; y omitted for the unconditional net);
      kind="class":      score = mean (eps_hat(x_s, t_s, 0) - eps_s)^2 - mean (eps_hat(x_s, t_s, y) - eps_s)^2,
                         guided net with label 0 as the null class: log p(y | x) - log p(y) up to a positive scale
                         (the diffusion classifier of Li et al. 2023 / Clark & Jaini 2023).
    The means run over a candidate's images, levels and elements.  A score is a deterministic function of
    (images, labels, seed): it does not depend on chunking, population, rank or batch position.  The UNet passes
    use the net's plan in per-image-time-step mode with the net's `precision` and `residual_fp16`; candidates go
    through whole-candidate chunks of at most `max_images` UNet images, one captured graph per plan."""
    uses_labels = True

    def __init__(self, sampler, kind: str = "likelihood", n_levels: int = 8, seed: int = 0, max_images: int = 256):
        if kind not in ("likelihood", "class"):
            raise ValueError(f"kind {kind!r}: 'likelihood' or 'class'")
        self.sampler = sampler
        self.kind = kind
        self.conditional = bool(getattr(sampler._unet(), "is_conditional", False))
        if kind == "class" and not self.conditional:
            raise ValueError("kind='class' needs the guided net (ModelCondition.UNet, label 0 = null class)")
        self.levels = score_levels(sampler.T, n_levels)
        self.n_levels = len(self.levels)
        self.seed = int(seed)
        self.max_images = int(max_images)
        self.graph_captures = 0
        self._graphs: Dict = {}
        self._tables: Dict = {}

    def _tables_for(self, dev, n_per: int):
        """(eps_tab [S, n_per], coef [S, 2]) on `dev`: the common noise and {sqrt(abar_t), sqrt(1 - abar_t)}."""
        key = (str(dev), n_per, self.sampler.betas.data_ptr())
        tab = self._tables.get(key)
        if tab is None:
            abar = torch.cumprod(1. - self.sampler.betas.detach().double().cpu(), dim=0)[self.levels]
            coef = torch.stack([torch.sqrt(abar), torch.sqrt(1. - abar)], dim=1).float().to(dev).contiguous()
            eps = torch.empty((self.n_levels, n_per), dtype=torch.float32, device=dev)
            _lib.check(_lib.lib().its_philox_normal(eps.data_ptr(), None, 0, 1.0, self.n_levels, n_per, self.seed, 0,
                                                    TAG_SCORE, _lib.stream_ptr(dev)), "its_philox_normal")
            tab = self._tables[key] = (eps, coef)
        return tab

    def score_candidates(self, images: torch.Tensor, per_cand: int,
                         labels: Optional[torch.Tensor] = None) -> torch.Tensor:
        """[n_cand] fp32 device scores of groups of `per_cand` consecutive images; `labels` [n_img] int64, one per
        image (required for the conditional net)."""
        _lib.require_cuda()
        if images.device.type != "cuda":
            raise RuntimeError("its_b200 verifiers run on CUDA only (no CPU fallback)")
        if images.dim() != 4:
            raise ValueError(f"expected images [B,C,H,W], got {tuple(images.shape)}")
        n_img, C, H, W = images.shape
        B = int(per_cand)
        if B <= 0 or n_img % B:
            raise ValueError(f"{n_img} images do not split into candidates of {per_cand}")
        net = self.sampler._unet()
        if net.head.weight.device != images.device:
            raise RuntimeError(f"images live on {images.device} but the UNet on {net.head.weight.device}")
        if self.conditional:
            if labels is None:
                raise ValueError("the conditional net's denoising verifier needs labels (one per image)")
            labels = labels.reshape(-1).to(device=images.device, dtype=torch.int64)
            if labels.numel() != n_img:
                raise ValueError(f"labels must hold one label per image ({n_img}), got {labels.numel()}")
            net.check_indices(None, labels)
        x = images.detach().to(torch.float32).contiguous()
        n_cand, S, n_per = n_img // B, self.n_levels, C * H * W
        halves = 2 if self.kind == "class" else 1
        per_chunk = max(1, self.max_images // (halves * B * S))
        out = torch.empty(n_cand, dtype=torch.float32, device=x.device)
        L = _lib.lib()
        with torch.cuda.device(x.device), torch.no_grad():
            eps_tab, coef = self._tables_for(x.device, n_per)
            for c0 in range(0, n_cand, per_chunk):
                n = min(per_chunk, n_cand - c0)
                rows = n * B * S
                plan = net.plan(halves * rows, H, W, n_img_in=rows, uniform_t=False, impl=getattr(net, "impl", None))
                g = self._graph_for(net, plan, (eps_tab, coef), n, B, x.device)
                g.x.copy_(x[c0 * B:(c0 + n) * B])
                plan.t_idx.copy_(g.t_rows)       # the plan is shared with UNet.forward of the same batch: restate
                if self.conditional:
                    lab = labels[c0 * B:(c0 + n) * B].repeat_interleave(S)
                    plan.labels.copy_(torch.cat([lab, torch.zeros_like(lab)]) if halves == 2 else lab)
                    plan.run_label_ops()
                eps_u = plan.eps[rows:].data_ptr() if halves == 2 else None

                def run():
                    s = _lib.stream_ptr()
                    _lib.check(L.its_level_inputs(plan.x_in.data_ptr(), g.x.data_ptr(), eps_tab.data_ptr(),
                                                  coef.data_ptr(), n * B, S, n_per, s), "its_level_inputs")
                    plan.run()
                    _lib.check(L.its_denoise_scores(g.scores.data_ptr(), plan.eps.data_ptr(), eps_u,
                                                    eps_tab.data_ptr(), n, B, S, n_per, s), "its_denoise_scores")

                if g.graph is None:
                    # one eager pass first: it scores this chunk and performs the lazy one-time kernel attribute
                    # setup outside of stream capture
                    run()
                    g.graph = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g.graph):
                        run()
                    self.graph_captures += 1
                else:
                    g.graph.replay()
                out[c0:c0 + n] = g.scores
        return out

    def _graph_for(self, net, plan, tables, n: int, B: int, dev) -> _ScoreGraph:
        key = (plan, n, B, tables[0].data_ptr())
        g = self._graphs.get(key)
        if g is None:
            live = list(net._plans.values())     # drop the graphs of plans the net has since rebuilt
            self._graphs = {k: v for k, v in self._graphs.items() if any(k[0] is p for p in live)}
            t = torch.tensor(self.levels, dtype=torch.int64, device=dev).repeat(plan.n_img // self.n_levels)
            g = self._graphs[key] = _ScoreGraph(plan, tables, torch.empty((n * B,) + tuple(plan.x_in.shape[1:]),
                                                                  dtype=torch.float32, device=dev),
                                                t, torch.empty(n, dtype=torch.float32, device=dev))
        return g

    def score(self, images: torch.Tensor, labels: Optional[torch.Tensor] = None) -> float:
        """The whole batch as one candidate (the reference's verifier protocol)."""
        return float(self.score_candidates(images, images.shape[0], labels).item())


MAX_ENSEMBLE = 8     # its_rank_ensemble's member limit


def rank_ensemble(scores: torch.Tensor, weights: torch.Tensor, n_seg: int = 1) -> torch.Tensor:
    """[n] fp32 device tensor: the rank ensemble (its_rank_ensemble) of the member scores [n, V] over `n_seg`
    equal segments, with device fp32 `weights` [V].  Eligible candidates score in [0, 1], higher is better; a
    candidate with a NaN or -inf member score gets NaN."""
    _lib.require_cuda()
    s = scores.detach().to(torch.float32).contiguous()
    if s.dim() != 2 or not 1 <= s.shape[1] <= MAX_ENSEMBLE:
        raise ValueError(f"member scores must be [n, V] with 1 <= V <= {MAX_ENSEMBLE}, got {tuple(s.shape)}")
    n, V = s.shape
    if n_seg < 1 or n % n_seg:
        raise ValueError(f"{n} candidates do not split into {n_seg} equal segments")
    w = weights.to(device=s.device, dtype=torch.float32).contiguous()
    if w.numel() != V:
        raise ValueError(f"{w.numel()} weights for {V} members")
    out = torch.empty(n, dtype=torch.float32, device=s.device)
    with torch.cuda.device(s.device):
        _lib.check(_lib.lib().its_rank_ensemble(out.data_ptr(), s.data_ptr(), w.data_ptr(), V, int(n_seg), n // n_seg,
                                                _lib.stream_ptr(s.device)), "its_rank_ensemble")
    return out


class EnsembleVerifier(_KernelVerifier):
    """Several kernel verifiers combined by rank (the verifier ensemble of Ma et al., a guard against one verifier
    being exploited by a large search; not in the reference).  Each member scores the same candidates; within each
    query's population a candidate's score is the weighted mean of its average ranks under the members, scaled to
    [0, 1] (`rank_ensemble`).  Ranks do not depend on the members' scales, so a likelihood of ~-0.1, a class gap of
    ~1e-4 and a pixel statistic weigh as the weights say.

    A rank exists only within a population, so the searches use an ensemble in population mode: they gather the
    member scores [n, V] (`score_candidates`) and turn them into one score per candidate with `combine` before
    selecting.  `score` (one batch as one candidate) raises.  Zero-order search and FK steering compare scores of
    different populations and refuse an ensemble (`ranks_population`)."""
    ranks_population = True

    def __init__(self, members, weights=None):
        members = list(members)
        if not 1 <= len(members) <= MAX_ENSEMBLE:
            raise ValueError(f"an ensemble takes 1 to {MAX_ENSEMBLE} members, got {len(members)}")
        for m in members:
            if isinstance(m, EnsembleVerifier):
                raise ValueError("an ensemble cannot be a member of another ensemble")
            if not isinstance(m, _KernelVerifier):
                raise ValueError(f"ensemble member {type(m).__name__} is not a kernel verifier")
            if isinstance(m, OracleVerifier) and m.dataset_stats is not None:
                raise ValueError("an OracleVerifier with dataset_stats scores a batch, not candidates: it cannot be "
                                 "an ensemble member")
        w = [1.0] * len(members) if weights is None else [float(x) for x in weights]
        if len(w) != len(members):
            raise ValueError(f"{len(w)} ensemble weights for {len(members)} members")
        if not all(np.isfinite(x) and x > 0.0 for x in w):
            raise ValueError(f"ensemble weights must be finite and > 0, got {w}")
        self.members = members
        self.weights = w
        self.uses_labels = any(getattr(m, "uses_labels", False) for m in members)
        self._w: Dict[str, torch.Tensor] = {}

    def score_candidates(self, images: torch.Tensor, per_cand: int,
                         labels: Optional[torch.Tensor] = None) -> torch.Tensor:
        """[n_cand, V] fp32 device scores: column v is member v's scores of the same candidates; `labels` go to the
        members that use them."""
        cols = [m.score_candidates(images, per_cand, labels=labels) if getattr(m, "uses_labels", False)
                else m.score_candidates(images, per_cand) for m in self.members]
        return torch.stack(cols, dim=1)

    def combine(self, scores: torch.Tensor, n_seg: int) -> torch.Tensor:
        """[n] ensemble scores of the gathered member scores [n, V], ranked within each of `n_seg` equal segments."""
        key = str(scores.device)
        w = self._w.get(key)
        if w is None:
            w = self._w[key] = torch.tensor(self.weights, dtype=torch.float32, device=scores.device)
        return rank_ensemble(scores, w, n_seg)

    def score(self, images: torch.Tensor, labels: Optional[torch.Tensor] = None) -> float:
        raise ValueError("a rank ensemble scores a population: one image batch has no rank.  Pass the ensemble's "
                         ".score to a search with a SamplerDenoiser, or use score_candidates + combine")


def _need_clip():
    try:
        import clip  # noqa: F401
    except ImportError as e:
        raise RuntimeError("this verifier wraps openai-CLIP, which is not installed here and has no "
                           "pinned weights (parity unpinned; outside the kernel scope)") from e


class SupervisedVerifier:
    def __init__(self, model_name: str = 'ViT-B/32', device: str = 'cuda', **kwargs: Any):
        _need_clip()
        raise NotImplementedError("CLIP-backed SupervisedVerifier is outside the accelerated path")


class CLIPScore:
    def __init__(self, device: str = 'cuda', **kwargs: Any):
        _need_clip()
        raise NotImplementedError("CLIP-backed CLIPScore is outside the accelerated path")


class IntegratedVerifier:
    def __init__(self, device: str = 'cuda', weights: Dict[str, float] = None):
        _need_clip()
        raise NotImplementedError("CLIP-backed IntegratedVerifier is outside the accelerated path")
