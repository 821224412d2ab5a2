"""Search over noise candidates with the reference's surface
(search/search_algorithm.py): RandomSearch (:18-87), ZeroOrderSearch (:90-235),
PathSearch (:238-340); same constructors, `.search(...)` signatures, return
values, `.nfes` / `.reset_nfes()`.

Two execution modes
  * population mode — taken when `denoise_fn` is an its_b200 `SamplerDenoiser`
    (see `make_denoise_fn`) and `verifier_fn` is the bound `.score` of an
    its_b200 verifier: the whole candidate population of a round is denoised as
    device batches (candidates are the batch dimension), scored on the device,
    and selected with the first-index argmax kernel.  With torch.distributed
    initialised the candidates are block-sharded over the ranks; the only
    collective is one all_gather of the per-candidate fp32 scores per round (and
    nothing inside the T-step loop); every rank then holds the same selection.
  * callable mode — any other `denoise_fn` / `verifier_fn`: the reference's
    serial loop, candidate by candidate, with its exact update rule.

Selection semantics in both modes are the reference's: strict `>` (first maximum
wins, NaN never wins), ZeroOrder moves the pivot only when the round's best beats
the global best (:193-196), PathSearch is the reference's placeholder (perturb
x_T, denoise fully, :307-316) unless `restart=True` is passed (opt-in extension:
true mid-trajectory restart at `injection_step`).

SearchOverPaths is not in the reference: it is the search over paths of Ma et al. (a beam of partial
trajectories, re-noised and pruned by top-k on x0 predictions), in population mode only.

Batched searches (not in the reference): `RandomSearch.search_batch`, `SearchOverPaths.search_batch` and
`FKSteering.search_batch` run K
independent queries, each with its own labels, as one candidate population and select every query's winner
(or survivors) on the device with one segmented top-k.  `search` is the K = 1 case of the same code.

FKSteering is not in the reference either: Feynman-Kac steering of Singhal et al. (a population of particles
resampled by verifier potentials on their x0 predictions), in population mode only.

GradientBasedSearch (:343-438) needs autograd through the whole trajectory: it is kept
for arbitrary differentiable callables (callable mode only, the reference's loop); the
kernel sampler is not differentiable and is refused with a clear error.
"""
from __future__ import annotations

import math
from typing import Any, Callable, Dict, List, Optional, Sequence, Tuple

import torch

from .. import _lib
from .._sampler_base import X_T_TAG
from . import verifier as _ver

TAG_X_T = X_T_TAG            # candidate x_T draws
TAG_NEIGHBOR = X_T_TAG + 16  # + iteration
TAG_PATH = X_T_TAG + 8
TAG_FORWARD = X_T_TAG + 4    # SearchOverPaths re-noising draws, keyed by round and child
TAG_RESAMPLE = X_T_TAG + 2   # FKSteering: the one uniform of each systematic resampling, keyed by query and round
# SearchOverPaths: image b of child c in round r (1-based; the initial paths are round 0) draws its step noise from
# Philox candidate id r * ROUND_STRIDE + c * B + b
ROUND_STRIDE = 1 << 40


# ------------------------------------------------------------------ adapter --
class SamplerDenoiser:
    """`denoise_fn` adapter around an its_b200 sampler: the reference's samplers
    do not accept `show_progress`, and its search classes pass the same **kwargs
    to the denoiser and the verifier (search_algorithm.py:71,75)."""

    def __init__(self, sampler, labels: Optional[torch.Tensor] = None, *, max_images: int = 256,
                 seed: Optional[int] = None, step_noise: Optional[torch.Tensor] = None):
        self.sampler = sampler
        self.labels = labels
        self.max_images = int(max_images)
        self.seed = seed
        self.step_noise = step_noise     # [T, B, C, H, W] shared by every candidate (parity runs)
        self._calls = 0                  # callable mode: the i-th call of a search is global candidate i
        self._fallback_seed: Optional[int] = None

    def reset_calls(self) -> None:
        """Callable mode numbers its candidates by call order; a search starts counting at zero."""
        self._calls = 0

    def step_seed(self, shared: Optional[int] = None) -> int:
        """Seed of the per-step Philox noise: the denoiser's own, else the search's shared (broadcast) seed, else
        one draw that then stays fixed for this denoiser (never a fresh one per call: a candidate's trajectory
        must not depend on which call, rank or search round evaluates it)."""
        if self.seed is not None:
            return int(self.seed)
        if shared is not None:
            return int(shared)
        if self._fallback_seed is None:
            self._fallback_seed = int(torch.randint(0, 2 ** 62, (1,)).item())
        return self._fallback_seed

    def image_labels(self, n_cand: int, labels=None, cand_labels: Optional[torch.Tensor] = None
                     ) -> Optional[torch.Tensor]:
        """Flat per-image labels [n_cand * B] the guided sampler is fed for `n_cand` candidates: `cand_labels`
        [n_cand, B] (one row per candidate) when given, else `labels` (or the denoiser's own) [B] for every
        candidate; None for an unguided sampler.  The verifiers that read labels score with the same vector."""
        if not getattr(self.sampler, "guided", False):
            return None
        if cand_labels is not None:
            return cand_labels.reshape(-1)
        lab = labels if labels is not None else self.labels
        if lab is None:
            return None
        return lab.reshape(-1).repeat(n_cand)

    def __call__(self, noise: torch.Tensor, show_progress: bool = False, **kwargs) -> torch.Tensor:
        # the reference draws fresh step noise for every candidate (Diffusion.py:96): candidate i of a serial
        # search uses Philox stream i, exactly the stream population mode gives global candidate i
        i = self._calls
        self._calls += 1
        return self.denoise_candidates(noise.unsqueeze(0), i, labels=kwargs.get("labels"))[0]

    def denoise_candidates(self, cands: torch.Tensor, first_cand: int, *, labels=None,
                           t_start: Optional[int] = None, seed: Optional[int] = None, t_stop: int = 0,
                           cand_labels: Optional[torch.Tensor] = None) -> torch.Tensor:
        """cands [n, B, C, H, W] -> images [n, B, C, H, W]; candidate i is global
        candidate first_cand + i (its Philox streams are keyed by that id).  `t_start` (default T-1) and `t_stop`
        bound the loop as the sampler's own arguments do (a `t_stop` > 0 returns the states step t_stop - 1
        starts from)."""
        t_start = self.sampler.T - 1 if t_start is None else t_start
        return self.denoise_segment(cands, first_cand, t_start=t_start, t_stop=t_stop, labels=labels, seed=seed,
                                    x0=False, cand_labels=cand_labels)[0]

    def denoise_segment(self, states: torch.Tensor, first_cand: int, *, t_start: int, t_stop: int,
                        cand_offset: int = 0, labels=None, seed: Optional[int] = None,
                        x0: bool = True, cand_labels: Optional[torch.Tensor] = None
                        ) -> Tuple[torch.Tensor, Optional[torch.Tensor]]:
        """states [n, B, C, H, W] at step t_start -> (states after step t_stop, x0 predictions of step t_stop or
        None), in chunks of `max_images`.  Candidate i's per-step Philox streams are keyed by
        cand_offset + (first_cand + i) * B + image; every chunk replays the sampler's one step graph.  The guided
        sampler's labels are `cand_labels` [n, B] (int64, one row per candidate) when given, else `labels` (or the
        denoiser's own) [B] for every candidate."""
        n, B = states.shape[:2]
        if cand_labels is not None and tuple(cand_labels.shape) != (n, B):
            raise ValueError(f"cand_labels must be [{n}, {B}] (one label row per candidate), got "
                             f"{tuple(cand_labels.shape)}")
        per_call = max(1, self.max_images // B)
        out = torch.empty_like(states)
        out_x0 = torch.empty_like(states) if x0 else None
        seed = self.step_seed(seed)
        for i0 in range(0, n, per_call):
            i1 = min(n, i0 + per_call)
            x = states[i0:i1].reshape((i1 - i0) * B, *states.shape[2:])
            kw: Dict[str, Any] = dict(t_start=t_start, t_stop=t_stop, seed=seed,
                                      cand_id0=cand_offset + (first_cand + i0) * B, x0=x0)
            if self.step_noise is not None:
                kw["noise"] = self.step_noise.repeat(1, i1 - i0, 1, 1, 1)
            lab = self.image_labels(i1 - i0, labels, None if cand_labels is None else cand_labels[i0:i1])
            y, p = self.sampler.segment(x, lab, **kw)
            out[i0:i1] = y.view(i1 - i0, B, *states.shape[2:])
            if x0:
                out_x0[i0:i1] = p.view(i1 - i0, B, *states.shape[2:])
        return out, out_x0


def make_denoise_fn(sampler, labels: Optional[torch.Tensor] = None, **kw) -> SamplerDenoiser:
    """The glue the reference leaves to the user: wrap a sampler as `denoise_fn`."""
    return SamplerDenoiser(sampler, labels, **kw)


def _population_mode(denoise_fn, verifier_fn) -> Optional[Any]:
    if not isinstance(denoise_fn, SamplerDenoiser):
        return None
    owner = getattr(verifier_fn, "__self__", None)
    if isinstance(owner, _ver._KernelVerifier) and getattr(verifier_fn, "__name__", "") == "score":
        if isinstance(owner, _ver.OracleVerifier) and owner.dataset_stats is not None:
            return None
        return owner
    return None


# ---------------------------------------------------------------- utilities --
def _dist():
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        return dist, dist.get_rank(), dist.get_world_size()
    return None, 0, 1


def _shard(n: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous block of candidates owned by `rank` (ids stay global, so the
    result does not depend on the number of ranks)."""
    per = -(-n // world)
    lo = min(n, rank * per)
    return lo, min(n, lo + per)


def _gather_states(local: torch.Tensor, n: int) -> torch.Tensor:
    """All n rows of a population block-sharded by `_shard` ([n_local, ...] fp32 per rank), in global order on
    every rank: one all_gather of equal-sized, padded blocks."""
    dist, rank, world = _dist()
    if dist is None:
        return local
    per = -(-n // world)
    buf = torch.full((per, *local.shape[1:]), float("nan"), dtype=torch.float32, device=local.device)
    buf[: local.shape[0]] = local
    parts = [torch.empty_like(buf) for _ in range(world)]
    dist.all_gather(parts, buf)
    sizes = [_shard(n, r, world)[1] - _shard(n, r, world)[0] for r in range(world)]
    return torch.cat([p[:k] for p, k in zip(parts, sizes)])


def _gather_scores(local: torch.Tensor, n: int) -> torch.Tensor:
    return _gather_states(local, n)                   # the only collective of RandomSearch / ZeroOrder / PathSearch


def _shared_seed(seed: Optional[int], device) -> int:
    dist, rank, world = _dist()
    if seed is None:
        seed = int(torch.randint(0, 2 ** 62, (1,)).item())
    if dist is not None:
        t = torch.tensor([seed], dtype=torch.int64, device=device)
        dist.broadcast(t, src=0)
        seed = int(t.item())
    return seed


def philox_normal(shape: Sequence[int], seed: int, cand_id0: int, tag: int, device, *, base=None,
                  scale: float = 1.0) -> torch.Tensor:
    """[n_units, ...] N(0,1)*scale (+ base broadcast over units) from the library's
    counter-based generator; unit i (a whole candidate tensor) uses stream
    (seed, cand_id0 + i, tag), so a candidate can be regenerated from its id."""
    _lib.require_cuda()
    out = torch.empty(tuple(shape), dtype=torch.float32, device=device)
    n_img = shape[0]
    n_per = out.numel() // n_img
    b = None if base is None else base.to(device=device, dtype=torch.float32).contiguous()
    with torch.cuda.device(out.device):
        _lib.check(_lib.lib().its_philox_normal(out.data_ptr(), None if b is None else b.data_ptr(), 1, float(scale),
                                                n_img, n_per, seed, cand_id0, tag, _lib.stream_ptr(out.device)),
                   "its_philox_normal")
    return out


def argmax_first(scores: torch.Tensor) -> Tuple[int, float]:
    """(index, value) of the first maximum; (-1, -inf) when nothing beats -inf."""
    _lib.require_cuda()
    s = scores.detach().to(torch.float32).contiguous()
    idx = torch.empty(1, dtype=torch.int32, device=s.device)
    val = torch.empty(1, dtype=torch.float32, device=s.device)
    with torch.cuda.device(s.device):
        _lib.check(_lib.lib().its_argmax_first(idx.data_ptr(), val.data_ptr(), s.data_ptr(), s.numel(),
                                               _lib.stream_ptr(s.device)), "its_argmax_first")
    return int(idx.item()), float(val.item())


def _topk_device(scores: torch.Tensor, k: int, n_seg: int = 1) -> Tuple[torch.Tensor, torch.Tensor]:
    """topk_first of each of `n_seg` equal segments of `scores`, with the (int32 indices, fp32 values) left on the
    device: [n_seg * k], segment s's ranks at s*k ... s*k + k - 1, indices flat into `scores`."""
    _lib.require_cuda()
    s = scores.detach().to(torch.float32).contiguous()
    if n_seg < 1 or s.numel() % n_seg:
        raise ValueError(f"{s.numel()} scores do not split into {n_seg} equal segments")
    idx = torch.empty(n_seg * k, dtype=torch.int32, device=s.device)
    val = torch.empty(n_seg * k, dtype=torch.float32, device=s.device)
    with torch.cuda.device(s.device):
        _lib.check(_lib.lib().its_topk_first_segmented(idx.data_ptr(), val.data_ptr(), s.data_ptr(), int(n_seg),
                                                       s.numel() // n_seg, int(k), _lib.stream_ptr(s.device)),
                   "its_topk_first_segmented")
    return idx, val


def resample_systematic(reward: torch.Tensor, carried: Optional[torch.Tensor], lam: float, n_seg: int, seed: int,
                        round: int, tag: int = TAG_RESAMPLE) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """Systematic resampling of `n_seg` equal segments of particles by the potentials exp(lam * (reward - carried))
    (its_resample_systematic; `carried` None = 0), left on the device: (ancestors int32 [n], flat into `reward`
    like `_topk_device`'s indices, the ancestors' rewards fp32 [n] for the next call's `carried`, ESS fp32
    [n_seg]).  A segment without a finite weight gets ancestors -1, NaN rewards and ESS 0.  One uniform per
    (seed, segment, round), so every rank draws the same ancestors from the same gathered rewards."""
    _lib.require_cuda()
    r = reward.detach().to(torch.float32).contiguous()
    if n_seg < 1 or r.numel() % n_seg:
        raise ValueError(f"{r.numel()} rewards do not split into {n_seg} equal segments")
    c = None if carried is None else carried.detach().to(device=r.device, dtype=torch.float32).contiguous()
    if c is not None and c.numel() != r.numel():
        raise ValueError(f"carried holds {c.numel()} values, reward {r.numel()}")
    anc = torch.empty(r.numel(), dtype=torch.int32, device=r.device)
    out = torch.empty(r.numel(), dtype=torch.float32, device=r.device)
    ess = torch.empty(n_seg, dtype=torch.float32, device=r.device)
    with torch.cuda.device(r.device):
        _lib.check(_lib.lib().its_resample_systematic(anc.data_ptr(), out.data_ptr(), ess.data_ptr(), r.data_ptr(),
                                                      None if c is None else c.data_ptr(), float(lam), int(n_seg),
                                                      r.numel() // n_seg, int(seed), int(round), int(tag),
                                                      _lib.stream_ptr(r.device)), "its_resample_systematic")
    return anc, out, ess


def topk_first(scores: torch.Tensor, k: int) -> Tuple[List[int], List[float]]:
    """The k best (indices, values) under argmax_first's rule (strict '>', first index on ties, NaN never ranks);
    indices are -1 past the number of eligible scores."""
    idx, val = _topk_device(scores, k)
    return idx.tolist(), val.tolist()


def path_expand(x: torch.Tensor, parent: torch.Tensor, m: int, child0: int, n_child: int, a: float, b: float, *,
                z: Optional[torch.Tensor] = None, seed: int = 0, cand_id0: int = 0,
                tag: int = TAG_FORWARD) -> torch.Tensor:
    """[n_child, *x.shape[1:]]: child i = a * x[parent[(child0 + i) // m]] + b * z_i (fp32, separately rounded),
    z_i = z[i] or the Philox unit cand_id0 + child0 + i of `philox_normal` under `tag`.  `parent` is a device int32
    tensor (survivor indices into x, e.g. straight from the top-k kernel)."""
    _lib.require_cuda()
    xs = x.detach().to(torch.float32).contiguous()
    par = parent.to(device=xs.device, dtype=torch.int32).contiguous()
    out = torch.empty((n_child, *xs.shape[1:]), dtype=torch.float32, device=xs.device)
    zz = None if z is None else z.to(device=xs.device, dtype=torch.float32).contiguous()
    if zz is not None and zz.numel() != out.numel():
        raise ValueError(f"z must hold {tuple(out.shape)} values, got {tuple(zz.shape)}")
    with torch.cuda.device(xs.device):
        _lib.check(_lib.lib().its_path_expand(out.data_ptr(), xs.data_ptr(), par.data_ptr(), par.numel(), int(m),
                                              int(child0), int(n_child), xs.shape[0], out[0].numel(), float(a),
                                              float(b), None if zz is None else zz.data_ptr(), int(seed),
                                              int(cand_id0), int(tag), _lib.stream_ptr(xs.device)),
                   "its_path_expand")
    return out


def _score_candidates(ver, images: torch.Tensor, B: int, denoise: SamplerDenoiser, labels=None,
                      cand_labels: Optional[torch.Tensor] = None) -> torch.Tensor:
    """ver.score_candidates over candidates of B images; a verifier with `uses_labels` also gets the flat labels
    the denoiser fed the sampler for them."""
    if not getattr(ver, "uses_labels", False):
        return ver.score_candidates(images, B)
    return ver.score_candidates(images, B, labels=denoise.image_labels(images.shape[0] // B, labels, cand_labels))


def _score_population(cands_local: torch.Tensor, lo: int, n_total: int, denoise: SamplerDenoiser, ver,
                      kwargs, t_start=None, seed=None, cand_labels=None) -> torch.Tensor:
    """Denoise + score this rank's block of candidates, return ALL n_total scores.  `seed`: the search's
    shared seed, used for the step noise when the denoiser has none of its own (same on every rank).
    `cand_labels`: label rows of this rank's candidates ([n_local, B]), else kwargs' `labels` for all."""
    B = cands_local.shape[1] if cands_local.numel() else 1
    if cands_local.shape[0] > 0:
        imgs = denoise.denoise_candidates(cands_local, lo, labels=kwargs.get("labels"), t_start=t_start, seed=seed,
                                          cand_labels=cand_labels)
        local = _score_candidates(ver, imgs.reshape(-1, *imgs.shape[2:]), B, denoise, kwargs.get("labels"),
                                  cand_labels)
    else:
        local = torch.empty(0, dtype=torch.float32, device=cands_local.device)
    return _gather_scores(local, n_total)


def _check_queries(n_queries: int, noise_shape: Sequence[int], labels: Optional[torch.Tensor]) -> int:
    """K of a batched search; its `labels` must be [K] (one label per query) or [K, B] (one row per query)."""
    K = int(n_queries)
    if K < 1:
        raise ValueError(f"n_queries={n_queries} must be >= 1")
    B = int(noise_shape[0])
    if labels is not None and tuple(labels.shape) not in ((K,), (K, B)):
        raise ValueError(f"labels must be [{K}] or [{K}, {B}] (one label or one label row per query), got "
                         f"{list(labels.shape)}")
    return K


def _check_shape(name: str, t: Optional[torch.Tensor], want: Sequence[int]) -> None:
    if t is not None and tuple(t.shape) != tuple(want):
        raise ValueError(f"{name} must be {list(want)}, got {list(t.shape)}")


def _label_rows(labels: Optional[torch.Tensor], K: int, per_query: int, B: int, device) -> Optional[torch.Tensor]:
    """Query labels ([K] or [K, B]) as one int64 row per population member, query-major: [K * per_query, B]."""
    if labels is None:
        return None
    lab = labels.to(device=device, dtype=torch.int64).reshape(K, 1, -1).expand(K, per_query, B)
    return lab.reshape(K * per_query, B)


def _rows(rows: Optional[torch.Tensor], lo: int, hi: int) -> Optional[torch.Tensor]:
    return None if rows is None else rows[lo:hi]


def _query(K: int, q: int) -> str:
    """Prefix naming the query in the errors of a batched search (a single search keeps its messages)."""
    return f"query {q}, " if K > 1 else ""


# ------------------------------------------------------------ RandomSearch --
class RandomSearch:
    """N random x_T candidates; keep the best verifier score (:18-87).  `search_batch` runs K such searches at once."""

    def __init__(self, n_candidates: int = 4):
        self.n_candidates = n_candidates
        self.nfes = 0

    def search(self, noise_shape: Tuple[int, ...], denoise_fn: Callable, verifier_fn: Callable,
               device: str = 'cuda', verbose: bool = True, **kwargs) -> Tuple[torch.Tensor, float]:
        cand_noise = kwargs.pop("candidate_noise", None)   # [n, *noise_shape]: injected candidates
        seed = kwargs.pop("seed", None)
        ver = _population_mode(denoise_fn, verifier_fn)
        n = self.n_candidates
        if isinstance(denoise_fn, SamplerDenoiser):
            denoise_fn.reset_calls()
        if ver is None:
            best_noise, best_score = None, float('-inf')
            for i in range(n):
                noise = cand_noise[i].to(device) if cand_noise is not None else torch.randn(noise_shape, device=device)
                with torch.no_grad():
                    denoised = denoise_fn(noise, show_progress=(i == 0), **kwargs)
                    self.nfes += 1
                score = verifier_fn(denoised, **kwargs)
                if score > best_score:
                    best_score, best_noise = score, noise.clone()
            return best_noise, best_score
        best, vals, ids = self._population(noise_shape, denoise_fn, ver, 1, cand_noise=cand_noise, cand_labels=None,
                                           seed=seed, device=device, kwargs=kwargs)
        self.last_scores = self.last_scores[0]
        if ids[0] < 0:
            return None, float('-inf')
        self.last_index = ids[0]
        return best[0], vals[0]

    def search_batch(self, noise_shape: Tuple[int, ...], denoise_fn: Callable, verifier_fn: Callable,
                     n_queries: int, *, labels: Optional[torch.Tensor] = None,
                     candidate_noise: Optional[torch.Tensor] = None, seed: Optional[int] = None,
                     device: str = 'cuda') -> Tuple[torch.Tensor, List[float]]:
        """K = `n_queries` independent random searches of `n_candidates` (N) each, evaluated as one population of
        K*N candidates, with one winner per query selected on the device.  Population mode only.

        `labels` [K] or [K, B]: query q's labels (guided sampler; default: the denoiser's own for every query).
        `candidate_noise` [K, N, *noise_shape]: injected candidates.  Query q's candidate i is global candidate
        q*N + i (its x_T draw under TAG_X_T and its step noise are keyed by that id), so an unguided batch of K
        searches draws and scores exactly the population of RandomSearch(K*N).search with the same seed.
        Returns (best_noise [K, *noise_shape], best_scores); sets `last_scores` [K, N] (device), `last_index`
        (within-query indices) and `last_seed`.  A query with no rankable score gets a NaN row, -inf and -1."""
        K = _check_queries(n_queries, noise_shape, labels)
        ver = _population_mode(denoise_fn, verifier_fn)
        if ver is None:
            raise ValueError("search_batch needs an its_b200 SamplerDenoiser and a kernel verifier's .score "
                             "(population mode)")
        N = self.n_candidates
        _check_shape("candidate_noise", candidate_noise, (K, N, *noise_shape))
        denoise_fn.reset_calls()
        cand = None if candidate_noise is None else candidate_noise.reshape(K * N, *noise_shape)
        best, vals, ids = self._population(noise_shape, denoise_fn, ver, K, cand_noise=cand,
                                           cand_labels=_label_rows(labels, K, N, noise_shape[0], device),
                                           seed=seed, device=device, kwargs={})
        self.last_index = ids
        return best, vals

    def _population(self, noise_shape, denoise_fn: SamplerDenoiser, ver, K: int, *, cand_noise, cand_labels, seed,
                    device, kwargs) -> Tuple[torch.Tensor, List[float], List[int]]:
        """K queries of N candidates as one population sharded over the ranks; query q's candidate i is global
        candidate q*N + i.  One segmented top-k (k = 1 per query) selects every winner.  Sets `last_seed` and
        `last_scores` [K, N]; returns (winners [K, *noise_shape], scores, within-query indices), a NaN row, -inf
        and -1 for a query with no rankable score."""
        dist, rank, world = _dist()
        dev = torch.device(device)
        seed = _shared_seed(seed, dev)
        self.last_seed = seed
        N = self.n_candidates
        n = K * N
        lo, hi = _shard(n, rank, world)
        if cand_noise is not None:
            local = cand_noise[lo:hi].to(dev, torch.float32)
        else:
            local = philox_normal((hi - lo,) + tuple(noise_shape), seed, lo, TAG_X_T, dev) \
                if hi > lo else torch.empty((0, *noise_shape), device=dev)
        with torch.no_grad():
            scores = _score_population(local, lo, n, denoise_fn, ver, kwargs, seed=seed,
                                       cand_labels=_rows(cand_labels, lo, hi))
        self.nfes += n
        self.last_scores = scores.view(K, N)
        idx, val = _topk_device(scores, 1, n_seg=K)
        ids, vals = idx.tolist(), val.tolist()
        best = torch.full((K, *noise_shape), float('nan'), dtype=torch.float32, device=dev)
        for q, i in enumerate(ids):
            if i < 0:
                continue
            if cand_noise is not None:
                best[q] = cand_noise[i].to(dev, torch.float32)
            else:  # every rank regenerates the winner from its key: no broadcast needed
                best[q] = philox_normal((1,) + tuple(noise_shape), seed, i, TAG_X_T, dev)[0]
        return best, vals, [i - q * N if i >= 0 else -1 for q, i in enumerate(ids)]

    def reset_nfes(self):
        self.nfes = 0


# --------------------------------------------------------- ZeroOrderSearch --
class ZeroOrderSearch:
    """Iterative neighbourhood search around a pivot (:90-235)."""

    def __init__(self, n_neighbors: int = 4, lambda_radius: float = 0.95, n_iterations: int = 10,
                 verbose: bool = False):
        self.n_neighbors = n_neighbors
        self.lambda_radius = lambda_radius
        self.n_iterations = n_iterations
        self.verbose = verbose
        self.nfes = 0

    def _sample_neighbors(self, pivot: torch.Tensor, device: str) -> list:
        """pivot + randn_like(pivot) * (1 - lambda_radius), n_neighbors times (:210-231)."""
        return [pivot + torch.randn_like(pivot) * (1 - self.lambda_radius) for _ in range(self.n_neighbors)]

    def search(self, initial_noise: torch.Tensor, denoise_fn: Callable, verifier_fn: Callable,
               device: str = 'cuda', verbose: Optional[bool] = None,
               **kwargs) -> Tuple[torch.Tensor, float, Dict[str, Any]]:
        perts = kwargs.pop("perturbations", None)    # [iters][K, *shape] injected N(0,1) draws
        seed = kwargs.pop("seed", None)
        ver = _population_mode(denoise_fn, verifier_fn)
        current = initial_noise.clone()
        best_noise, best_score = initial_noise.clone(), float('-inf')
        history: Dict[str, Any] = {'scores': [], 'candidates_per_iter': []}
        K = self.n_neighbors
        radius = 1 - self.lambda_radius
        self.last_index = -1                # global candidate id (round * K + neighbour) of the returned noise
        if isinstance(denoise_fn, SamplerDenoiser):
            denoise_fn.reset_calls()
        if ver is not None:
            dist, rank, world = _dist()
            seed = _shared_seed(seed, initial_noise.device)
            self.last_seed = seed
        for it in range(self.n_iterations):
            if ver is None:
                if perts is not None:
                    neighbors = [current + perts[it][k].to(current) * radius for k in range(K)]
                else:
                    neighbors = self._sample_neighbors(current, device)
                it_scores, it_best, it_best_noise = [], float('-inf'), None
                for k, nb in enumerate(neighbors):
                    with torch.no_grad():
                        denoised = denoise_fn(nb, show_progress=(k == 0), **kwargs)
                        self.nfes += 1
                    score = verifier_fn(denoised, **kwargs)
                    it_scores.append(score)
                    if score > it_best:
                        it_best, it_best_noise, idx = score, nb.clone(), k
            else:
                lo, hi = _shard(K, rank, world)
                B = current.shape[0]
                if perts is not None:
                    local = current.unsqueeze(0) + perts[it][lo:hi].to(current) * radius
                elif hi > lo:
                    local = philox_normal((hi - lo,) + tuple(current.shape), seed, lo, TAG_NEIGHBOR + it,
                                          current.device, base=current.reshape(-1), scale=radius)
                else:
                    local = current.new_empty((0, *current.shape))
                with torch.no_grad():
                    scores = _score_population(local, lo + it * K, K, denoise_fn, ver, kwargs, seed=seed)
                self.nfes += K
                it_scores = [float(s) for s in scores.tolist()]
                idx, it_best = argmax_first(scores)
                it_best_noise = None
                if idx >= 0:
                    if perts is not None:
                        it_best_noise = current + perts[it][idx].to(current) * radius
                    else:
                        it_best_noise = philox_normal((1,) + tuple(current.shape), seed, idx, TAG_NEIGHBOR + it,
                                                      current.device, base=current.reshape(-1),
                                                      scale=radius)[0]
            history['scores'].append(it_scores)
            history['candidates_per_iter'].append(K)
            if it_best > best_score:
                best_score = it_best
                best_noise = it_best_noise.clone()
                current = it_best_noise.clone()
                self.last_index = it * K + idx
        return best_noise, best_score, history

    def reset_nfes(self):
        self.nfes = 0


# -------------------------------------------------------------- PathSearch --
class PathSearch:
    """Search over denoising paths (:238-340).  Default = the reference's
    placeholder: perturb x_T by noise_scale*N(0,1), denoise from T.  With
    `restart=True` (extension) the pivot trajectory is run once down to
    `injection_step`, the perturbation is applied to x_t there and only the
    remaining steps are denoised for every path."""

    def __init__(self, n_paths: int = 4, injection_step: int = 400, noise_scale: float = 0.1,
                 verbose: bool = False):
        self.n_paths = n_paths
        self.injection_step = injection_step
        self.noise_scale = noise_scale
        self.verbose = verbose
        self.nfes = 0

    def search(self, initial_noise: torch.Tensor, denoise_fn: Callable, verifier_fn: Callable,
               timesteps: int = 1000, device: str = 'cuda', verbose: Optional[bool] = None,
               **kwargs) -> Tuple[torch.Tensor, float, Dict[str, Any]]:
        variations = kwargs.pop("variations", None)   # [n_paths, *shape] injected N(0,1) draws
        seed = kwargs.pop("seed", None)
        restart = bool(kwargs.pop("restart", False))
        ver = _population_mode(denoise_fn, verifier_fn)
        best_noise, best_score = initial_noise.clone(), float('-inf')
        history: Dict[str, Any] = {'scores': [], 'injection_points': []}
        P = self.n_paths
        self.last_index = -1                # path index of the returned noise
        if isinstance(denoise_fn, SamplerDenoiser):
            denoise_fn.reset_calls()
        if ver is None:
            if restart:
                raise ValueError("restart=True needs an its_b200 SamplerDenoiser (population mode)")
            for p in range(P):
                var = variations[p].to(initial_noise) if variations is not None else torch.randn_like(initial_noise)
                perturbed = initial_noise + var * self.noise_scale
                with torch.no_grad():
                    denoised = denoise_fn(perturbed, show_progress=(p == 0), **kwargs)
                    self.nfes += 1
                score = verifier_fn(denoised, **kwargs)
                history['scores'].append(score)
                history['injection_points'].append(self.injection_step)
                if score > best_score:
                    best_score, best_noise, self.last_index = score, perturbed.clone(), p
            return best_noise, best_score, history
        dist, rank, world = _dist()
        seed = _shared_seed(seed, initial_noise.device)
        self.last_seed = seed
        lo, hi = _shard(P, rank, world)
        B = initial_noise.shape[0]
        base = initial_noise
        t_start = None
        if restart:
            # pivot trajectory T-1 .. injection_step (exclusive) on every rank, unclipped
            smp = denoise_fn.sampler
            T = smp.T
            if not (0 < self.injection_step < T):
                raise ValueError("injection_step must lie in (0, T)")
            base = denoise_fn.denoise_candidates(initial_noise.unsqueeze(0), 0, labels=kwargs.get("labels"), seed=seed,
                                                 t_stop=self.injection_step)[0]
            t_start = self.injection_step - 1

        def perturbed(i0, i1):
            if variations is not None:
                return base.unsqueeze(0) + variations[i0:i1].to(base) * self.noise_scale
            if i1 <= i0:
                return base.new_empty((0, *base.shape))
            return philox_normal((i1 - i0,) + tuple(base.shape), seed, i0, TAG_PATH, base.device,
                                 base=base.reshape(-1), scale=self.noise_scale)

        with torch.no_grad():
            scores = _score_population(perturbed(lo, hi), lo, P, denoise_fn, ver, kwargs, t_start=t_start, seed=seed)
        self.nfes += P
        history['scores'] = [float(s) for s in scores.tolist()]
        history['injection_points'] = [self.injection_step] * P
        idx, val = argmax_first(scores)
        if idx >= 0:
            best_score, best_noise, self.last_index = val, perturbed(idx, idx + 1)[0].clone(), idx
        return best_noise, best_score, history

    def reset_nfes(self):
        self.nfes = 0


# --------------------------------------------------------- SearchOverPaths --
def path_rounds(T: int, start_step: int, delta_f: int, delta_b: int) -> List[Tuple[int, int, int]]:
    """Round schedule of search over paths: (s, s', e) per round.  A round starts from states at step s, re-noises
    them to step s' = min(s + delta_f, T - 1) and denoises steps s' ... e = max(s' - delta_b + 1, 0); the next
    round starts at e - 1.  The last round ends with step 0.  Raises ValueError for parameters outside
    0 <= start_step <= T - 1, 0 <= delta_f < delta_b."""
    T, s, delta_f, delta_b = int(T), int(start_step), int(delta_f), int(delta_b)
    if T < 1:
        raise ValueError(f"T={T} must be >= 1")
    if not 0 <= s <= T - 1:
        raise ValueError(f"start_step={s} outside [0, T-1={T - 1}]")
    if delta_f < 0:
        raise ValueError(f"delta_f={delta_f} must be >= 0")
    if delta_b <= delta_f:
        raise ValueError(f"delta_b={delta_b} must exceed delta_f={delta_f} (each round must make progress)")
    rounds = []
    while True:
        sp = min(s + delta_f, T - 1)
        e = max(sp - delta_b + 1, 0)
        rounds.append((s, sp, e))
        if e == 0:
            return rounds
        s = e - 1


class SearchOverPaths:
    """Search over paths (Ma et al., "Inference-Time Scaling for Diffusion Models beyond Scaling Denoising
    Steps"): a beam of `n_beams` (N) partial trajectories.  Stage 0 denoises N initial x_T (Philox TAG_X_T keyed
    by path id, as RandomSearch draws candidates, or `candidate_noise` [N, *noise_shape]) down to the state at
    `start_step`.  Each round (`path_rounds`) re-noises every survivor `n_children` (M) times with q(x_s' | x_s)
    (`delta_f` forward steps), denoises all N*M children `delta_b` steps, scores each on the x0 prediction of its
    segment's last UNet evaluation (no extra evaluation) and keeps the N best (`topk_first`); the last round
    ends at step 0 and returns the best finished sample (k = 1, `argmax_first`'s rule).

    Population mode only: an its_b200 `SamplerDenoiser` and a kernel verifier's `.score`.  Paths and children
    are sharded over the ranks by global id; per round one score all_gather and one all_gather of the fp32
    states.  Random streams depend on (seed, inputs) only: step noise of a child by (seed, round, child id),
    re-noising by TAG_FORWARD, so results do not depend on rank count, `max_images` or batch.

    `search(noise_shape, denoise_fn, verifier_fn, ...)` returns (best_images [B,C,H,W], best_score, history);
    keyword extensions: `seed`, `labels`, `candidate_noise`, `forward_noise` ([rounds][N*M, *noise_shape]
    injected re-noising draws).  `last_index` is the winner's initial path id, `last_seed` the search seed.
    `nfes` counts UNet steps x candidates (the reference's classes count denoise_fn calls).  `search_batch` runs
    K such searches, with their own labels, as one population."""

    def __init__(self, n_beams: int = 4, n_children: int = 4, start_step: int = 800, delta_f: int = 50,
                 delta_b: int = 100, verbose: bool = False):
        self.n_beams = n_beams
        self.n_children = n_children
        self.start_step = start_step
        self.delta_f = delta_f
        self.delta_b = delta_b
        self.verbose = verbose
        self.nfes = 0

    def search(self, noise_shape: Tuple[int, ...], denoise_fn: Callable, verifier_fn: Callable,
               device: str = 'cuda', verbose: Optional[bool] = None,
               **kwargs) -> Tuple[torch.Tensor, float, Dict[str, Any]]:
        cand_noise = kwargs.pop("candidate_noise", None)
        fwd_noise = kwargs.pop("forward_noise", None)
        seed = kwargs.pop("seed", None)
        ver, rounds = self._schedule(denoise_fn, verifier_fn)
        if fwd_noise is not None and len(fwd_noise) < len(rounds):
            raise ValueError(f"forward_noise has {len(fwd_noise)} rounds, the schedule {len(rounds)}")
        images, best, h = self._population(tuple(noise_shape), denoise_fn, ver, rounds, 1, labels=kwargs.get("labels"),
                                           query_labels=None, cand_noise=cand_noise, fwd_noise=fwd_noise, seed=seed,
                                           device=device)
        history = {'rounds': h['rounds'], 'scores': h['scores'][0], 'survivors': h['survivors'][0],
                   'lineage': h['lineage'][0], 'unet_image_steps': h['unet_image_steps']}
        self.last_index = history['lineage']['path']
        return images[0], best[0], history

    def search_batch(self, noise_shape: Tuple[int, ...], denoise_fn: Callable, verifier_fn: Callable,
                     n_queries: int, *, labels: Optional[torch.Tensor] = None,
                     candidate_noise: Optional[torch.Tensor] = None, forward_noise=None, seed: Optional[int] = None,
                     device: str = 'cuda') -> Tuple[torch.Tensor, List[float], Dict[str, Any]]:
        """K = `n_queries` independent searches over paths evaluated as one population: K*N paths in stage 0 and
        K*N*M children per round, with the N survivors (and at the end the winner) of every query selected on the
        device by one segmented top-k.  Population mode only.

        `labels` [K] or [K, B]: query q's labels (guided sampler; default: the denoiser's own for every query).
        `candidate_noise` [K, N, *noise_shape] and `forward_noise` [rounds][K, N*M, *noise_shape]: injected draws.
        Query q's path i is global path q*N + i and its child c global child q*N*M + c; x_T, step noise and
        re-noising draws are keyed by those ids, so K = 1 is `search` and a query's result does not depend on
        the other queries, the rank count or `max_images`.
        Returns (best_images [K, *noise_shape], best_scores, history): history 'rounds' as in `search`; 'scores',
        'survivors' and 'lineage' are lists over the queries, with within-query ids; 'unet_image_steps' is the
        whole batch's.  `last_index` is the list of the winners' initial path ids.  A query whose children cannot
        be ranked raises ValueError naming the query and the round."""
        K = _check_queries(n_queries, noise_shape, labels)
        ver, rounds = self._schedule(denoise_fn, verifier_fn)
        shape = tuple(noise_shape)
        N, NM = int(self.n_beams), int(self.n_beams) * int(self.n_children)
        _check_shape("candidate_noise", candidate_noise, (K, N) + shape)
        fwd = None
        if forward_noise is not None:
            if len(forward_noise) < len(rounds):
                raise ValueError(f"forward_noise has {len(forward_noise)} rounds, the schedule {len(rounds)}")
            for r in range(len(rounds)):
                _check_shape(f"forward_noise[{r}]", forward_noise[r], (K, NM) + shape)
            fwd = [forward_noise[r].reshape((K * NM,) + shape) for r in range(len(rounds))]
        images, best, history = self._population(
            shape, denoise_fn, ver, rounds, K, labels=None, query_labels=labels,
            cand_noise=None if candidate_noise is None else candidate_noise.reshape((K * N,) + shape),
            fwd_noise=fwd, seed=seed, device=device)
        self.last_index = [lin['path'] for lin in history['lineage']]
        return images, best, history

    def _schedule(self, denoise_fn, verifier_fn) -> Tuple[Any, List[Tuple[int, int, int]]]:
        """(kernel verifier, round schedule) after checking the mode and the parameters against sampler.T."""
        ver = _population_mode(denoise_fn, verifier_fn)
        if ver is None:
            raise ValueError("SearchOverPaths needs an its_b200 SamplerDenoiser and a kernel verifier's .score "
                             "(population mode)")
        N, M = int(self.n_beams), int(self.n_children)
        if N < 1 or M < 1:
            raise ValueError(f"n_beams={N} and n_children={M} must be >= 1")
        return ver, path_rounds(denoise_fn.sampler.T, self.start_step, self.delta_f, self.delta_b)

    def _population(self, shape: Tuple[int, ...], denoise_fn: SamplerDenoiser, ver, rounds, K: int, *, labels,
                    query_labels, cand_noise, fwd_noise, seed, device):
        """K queries as one population sharded over the ranks (query q's path i is global path q*N + i, its child c
        global child q*N*M + c).  `labels`: shared labels of every member; `query_labels` ([K] or [K, B]): one
        label row per query.  Returns (best images [K, *shape], best scores, history with per-query 'scores',
        'survivors' and 'lineage' in within-query ids)."""
        N, M = int(self.n_beams), int(self.n_children)
        NM = N * M
        smp = denoise_fn.sampler
        T = smp.T
        dist, rank, world = _dist()
        dev = torch.device(device)
        seed = _shared_seed(seed, dev)
        self.last_seed = seed
        B = shape[0]
        abar = torch.cumprod(1. - smp.betas.detach().double().cpu(), dim=0)
        denoise_fn.reset_calls()
        path_labels, child_labels = _label_rows(query_labels, K, N, B, dev), _label_rows(query_labels, K, NM, B, dev)
        history: Dict[str, Any] = {'rounds': [], 'scores': [[] for _ in range(K)],
                                   'survivors': [[] for _ in range(K)]}
        steps = 0                                     # UNet steps x candidates
        with torch.no_grad():
            # stage 0: K*N paths from x_T down to the states at step start_step
            n_p = K * N
            lo, hi = _shard(n_p, rank, world)
            if cand_noise is not None:
                local = cand_noise[lo:hi].to(dev, torch.float32)
            elif hi > lo:
                local = philox_normal((hi - lo,) + shape, seed, lo, TAG_X_T, dev)
            else:
                local = torch.empty((0,) + shape, device=dev)
            s0 = rounds[0][0]
            if s0 < T - 1 and hi > lo:
                local = denoise_fn.denoise_candidates(local, lo, labels=labels, seed=seed, t_stop=s0 + 1,
                                                      cand_labels=_rows(path_labels, lo, hi))
            steps += n_p * (T - 1 - s0)
            parents = _gather_states(local.contiguous(), n_p)
            parent_idx = torch.arange(n_p, dtype=torch.int32, device=dev)
            n_c = K * NM
            lo, hi = _shard(n_c, rank, world)
            for r, (s, sp, e) in enumerate(rounds):
                ratio = float(abar[sp] / abar[s])
                a, b = math.sqrt(ratio), math.sqrt(1. - ratio)
                if hi > lo:
                    z = None if fwd_noise is None else fwd_noise[r][lo:hi]
                    kids = path_expand(parents.reshape(parents.shape[0], -1), parent_idx, M, lo, hi - lo, a, b,
                                       z=None if z is None else z.reshape(hi - lo, -1), seed=seed,
                                       cand_id0=(r + 1) * ROUND_STRIDE, tag=TAG_FORWARD).view((hi - lo,) + shape)
                    states, x0 = denoise_fn.denoise_segment(kids, lo, t_start=sp, t_stop=e, labels=labels, seed=seed,
                                                            cand_offset=(r + 1) * ROUND_STRIDE, x0=True,
                                                            cand_labels=_rows(child_labels, lo, hi))
                    judged = x0 if e > 0 else states   # the last round scores the finished, clipped samples
                    local_scores = _score_candidates(ver, judged.reshape(-1, *shape[1:]), B, denoise_fn, labels,
                                                     _rows(child_labels, lo, hi))
                else:
                    states = torch.empty((0,) + shape, device=dev)
                    local_scores = torch.empty(0, dtype=torch.float32, device=dev)
                steps += n_c * (sp - e + 1)
                scores = _gather_scores(local_scores, n_c)
                history['rounds'].append((s, sp, e))
                for q, row in enumerate(scores.view(K, NM).tolist()):
                    history['scores'][q].append(row)
                parents = _gather_states(states.contiguous(), n_c)
                # survivors (k = N per query) or the winner (k = 1): flat child ids, passed on as parents as they are
                parent_idx, best = _topk_device(scores, N if e > 0 else 1, n_seg=K)
                ids = parent_idx.tolist()
                k = len(ids) // K
                for q in range(K):
                    own = [i - q * NM if i >= 0 else -1 for i in ids[q * k:(q + 1) * k]]
                    if min(own) >= 0:
                        history['survivors'][q].append(own)
                    elif e > 0:
                        raise ValueError(f"{_query(K, q)}round {r}: only {sum(i >= 0 for i in own)} of {NM} children "
                                         f"have a score that can be ranked; {N} survivors are needed")
                    else:
                        raise ValueError(f"{_query(K, q)}last round: none of the {NM} finished samples has a score "
                                         "that can be ranked")
        # lineage of each winner: child id in every round, back to its initial path
        history['lineage'] = []
        for surv in history['survivors']:
            child = surv[-1][0]
            lineage = [child]
            for ids in reversed(surv[:-1]):
                child = ids[child // M]
                lineage.append(child)
            lineage.reverse()
            history['lineage'].append({'path': lineage[0] // M, 'children': lineage})
        history['unet_image_steps'] = steps * B * (2 if getattr(smp, "guided", False) else 1)
        self.nfes += steps
        return parents[parent_idx.long()].clone(), best.tolist(), history

    def reset_nfes(self):
        self.nfes = 0


# -------------------------------------------------------------- FKSteering --
def fk_segments(T: int, start_step: int, interval: int) -> List[Tuple[int, int]]:
    """Segment schedule of Feynman-Kac steering: (t_start, t_stop) per segment, steps t_start ... t_stop inclusive.
    The first segment is (T-1, start_step); each following one starts one step below the previous stop and runs
    `interval` steps, (stop - 1, max(stop - interval, 0)); the last one ends with step 0.  The population is
    resampled after every segment but the last.  Raises ValueError unless 0 <= start_step <= T-1, interval >= 1."""
    T, s, interval = int(T), int(start_step), int(interval)
    if T < 1:
        raise ValueError(f"T={T} must be >= 1")
    if not 0 <= s <= T - 1:
        raise ValueError(f"start_step={s} outside [0, T-1={T - 1}]")
    if interval < 1:
        raise ValueError(f"resample_interval={interval} must be >= 1")
    segments = [(T - 1, s)]
    while segments[-1][1] > 0:
        stop = segments[-1][1]
        segments.append((stop - 1, max(stop - interval, 0)))
    return segments


class FKSteering:
    """Feynman-Kac steering (Singhal et al., "A General Framework for Inference-time Scaling and Steering of
    Diffusion Models", 2025): `n_particles` (N) trajectories denoised together from x_T (Philox TAG_X_T keyed by
    particle id, as RandomSearch draws candidates, or `candidate_noise` [N, *noise_shape]).  After each segment of
    `fk_segments(T, start_step, resample_interval)` but the last, every particle's x0 prediction (the segment's last
    UNet evaluation, no extra one) is scored and the population is resampled systematically with the potentials
    exp(lam * (reward - reward at the previous resampling)) (`resample_systematic`).  Nothing is re-noised and no
    step runs twice: the UNet budget is RandomSearch(N)'s.  The last segment ends at step 0; the best finished
    sample wins under `argmax_first`'s rule.

    Population mode only: an its_b200 `SamplerDenoiser` and a kernel verifier's `.score`.  Particle j of segment r
    draws its step noise from Philox candidate id r * ROUND_STRIDE + j * B + image, so segment 0 continues
    RandomSearch's streams and the copies a resampling makes of one particle go on with streams of their own.
    Particles are sharded over the ranks; per resampling one score all_gather and one all_gather of the fp32
    states, and every rank draws the same ancestors.

    `search(noise_shape, denoise_fn, verifier_fn, ...)` returns (best_images [B,C,H,W], best_score, history);
    keyword extensions: `seed`, `labels`, `candidate_noise`.  history: 'segments'; per resampling 'scores' (N),
    'ancestors' (N particle ids) and 'ess'; 'lineage', the winner's particle id in every segment (lineage[0] is its
    x_T id); 'unet_image_steps'.  `last_index` is the winner's x_T id, `last_seed` the search seed; `nfes` counts
    UNet steps x particles (N * T per search).  `search_batch` runs K such searches, with their own labels, as one
    population."""

    def __init__(self, n_particles: int = 4, start_step: int = 800, resample_interval: int = 100, lam: float = 10.0):
        self.n_particles = n_particles
        self.start_step = start_step
        self.resample_interval = resample_interval
        self.lam = lam
        self.nfes = 0

    def search(self, noise_shape: Tuple[int, ...], denoise_fn: Callable, verifier_fn: Callable,
               device: str = 'cuda', verbose: Optional[bool] = None,
               **kwargs) -> Tuple[torch.Tensor, float, Dict[str, Any]]:
        cand_noise = kwargs.pop("candidate_noise", None)
        seed = kwargs.pop("seed", None)
        shape = tuple(noise_shape)
        ver, segments = self._schedule(denoise_fn, verifier_fn)
        _check_shape("candidate_noise", cand_noise, (int(self.n_particles),) + shape)
        images, best, h = self._population(shape, denoise_fn, ver, segments, 1, labels=kwargs.get("labels"),
                                           query_labels=None, cand_noise=cand_noise, seed=seed, device=device)
        history = {'segments': h['segments'], 'scores': h['scores'][0], 'ancestors': h['ancestors'][0],
                   'ess': h['ess'][0], 'lineage': h['lineage'][0], 'unet_image_steps': h['unet_image_steps']}
        self.last_index = history['lineage'][0]
        return images[0], best[0], history

    def search_batch(self, noise_shape: Tuple[int, ...], denoise_fn: Callable, verifier_fn: Callable,
                     n_queries: int, *, labels: Optional[torch.Tensor] = None,
                     candidate_noise: Optional[torch.Tensor] = None, seed: Optional[int] = None,
                     device: str = 'cuda') -> Tuple[torch.Tensor, List[float], Dict[str, Any]]:
        """K = `n_queries` independent FK-steering searches evaluated as one population of K*N particles, resampled
        per query by one segmented kernel launch, with every query's winner selected on the device by one segmented
        top-k.  Population mode only.

        `labels` [K] or [K, B]: query q's labels (guided sampler; default: the denoiser's own for every query).
        `candidate_noise` [K, N, *noise_shape]: injected x_T.  Query q's particle j is global particle q*N + j
        (its x_T draw and step noise are keyed by that id, its resampling uniform by q, ancestors never cross
        queries), so K = 1 is `search`, query 0 is the single search with query 0's inputs, and a query's result
        does not depend on the other queries' inputs, the rank count or `max_images`.
        Returns (best_images [K, *noise_shape], best_scores, history): 'segments' as in `search`; 'scores',
        'ancestors', 'ess' and 'lineage' are lists over the queries, with within-query ids; 'unet_image_steps' is
        the whole batch's.  `last_index` is the list of the winners' x_T ids.  A query none of whose particles can
        be weighted raises ValueError naming the query and the resampling round."""
        K = _check_queries(n_queries, noise_shape, labels)
        shape = tuple(noise_shape)
        ver, segments = self._schedule(denoise_fn, verifier_fn)
        N = int(self.n_particles)
        _check_shape("candidate_noise", candidate_noise, (K, N) + shape)
        images, best, history = self._population(
            shape, denoise_fn, ver, segments, K, labels=None, query_labels=labels,
            cand_noise=None if candidate_noise is None else candidate_noise.reshape((K * N,) + shape),
            seed=seed, device=device)
        self.last_index = [lin[0] for lin in history['lineage']]
        return images, best, history

    def _schedule(self, denoise_fn, verifier_fn) -> Tuple[Any, List[Tuple[int, int]]]:
        """(kernel verifier, segment schedule) after checking the mode and the parameters against sampler.T."""
        ver = _population_mode(denoise_fn, verifier_fn)
        if ver is None:
            raise ValueError("FKSteering needs an its_b200 SamplerDenoiser and a kernel verifier's .score "
                             "(population mode)")
        if int(self.n_particles) < 1:
            raise ValueError(f"n_particles={self.n_particles} must be >= 1")
        if not (math.isfinite(float(self.lam)) and float(self.lam) >= 0.0):
            raise ValueError(f"lam={self.lam} must be finite and >= 0")
        return ver, fk_segments(denoise_fn.sampler.T, self.start_step, self.resample_interval)

    def _population(self, shape: Tuple[int, ...], denoise_fn: SamplerDenoiser, ver, segments, K: int, *, labels,
                    query_labels, cand_noise, seed, device):
        """K queries of N particles as one population sharded over the ranks (query q's particle j is global
        particle q*N + j).  `labels`: shared labels of every particle; `query_labels` ([K] or [K, B]): one label row
        per query.  Returns (best images [K, *shape], best scores, history with per-query 'scores', 'ancestors',
        'ess' and 'lineage' in within-query ids)."""
        N = int(self.n_particles)
        n = K * N
        smp = denoise_fn.sampler
        dist, rank, world = _dist()
        dev = torch.device(device)
        seed = _shared_seed(seed, dev)
        self.last_seed = seed
        B = shape[0]
        denoise_fn.reset_calls()
        rows = _label_rows(query_labels, K, N, B, dev)
        lo, hi = _shard(n, rank, world)
        history: Dict[str, Any] = {'segments': list(segments), 'scores': [[] for _ in range(K)],
                                   'ancestors': [[] for _ in range(K)], 'ess': [[] for _ in range(K)]}
        steps = 0                                     # UNet steps x particles
        carried = None
        with torch.no_grad():
            if cand_noise is not None:
                local = cand_noise[lo:hi].to(dev, torch.float32)
            elif hi > lo:
                local = philox_normal((hi - lo,) + shape, seed, lo, TAG_X_T, dev)
            else:
                local = torch.empty((0,) + shape, device=dev)
            for r, (t_start, t_stop) in enumerate(segments):
                last = t_stop == 0
                if hi > lo:
                    local, x0 = denoise_fn.denoise_segment(local, lo, t_start=t_start, t_stop=t_stop, labels=labels,
                                                           seed=seed, cand_offset=r * ROUND_STRIDE, x0=True,
                                                           cand_labels=_rows(rows, lo, hi))
                    judged = local if last else x0    # the last segment scores the finished, clipped samples
                    local_scores = _score_candidates(ver, judged.reshape(-1, *shape[1:]), B, denoise_fn, labels,
                                                     _rows(rows, lo, hi))
                else:
                    local_scores = torch.empty(0, dtype=torch.float32, device=dev)
                steps += n * (t_start - t_stop + 1)
                scores = _gather_scores(local_scores, n)
                states = _gather_states(local.contiguous(), n)
                if last:
                    break
                anc, carried, ess = resample_systematic(scores, carried, self.lam, K, seed, r)
                ids, vals, ess_q = anc.tolist(), scores.view(K, N).tolist(), ess.tolist()
                for q in range(K):
                    own = [i - q * N if i >= 0 else -1 for i in ids[q * N:(q + 1) * N]]
                    if own[0] < 0:
                        raise ValueError(f"{_query(K, q)}resampling round {r}: none of the {N} particles has a "
                                         "finite score to weight")
                    history['scores'][q].append(vals[q])
                    history['ancestors'][q].append(own)
                    history['ess'][q].append(ess_q[q])
                local = states.index_select(0, anc[lo:hi].long())
            idx, best = _topk_device(scores, 1, n_seg=K)
            winners = idx.tolist()
        history['lineage'] = []
        for q, i in enumerate(winners):
            if i < 0:
                raise ValueError(f"{_query(K, q)}last segment: none of the {N} finished samples has a score that can "
                                 "be ranked")
            j = i - q * N
            lineage = [j]
            for own in reversed(history['ancestors'][q]):
                j = own[j]
                lineage.append(j)
            lineage.reverse()
            history['lineage'].append(lineage)
        history['unet_image_steps'] = steps * B * (2 if getattr(smp, "guided", False) else 1)
        self.nfes += steps
        return states.index_select(0, idx.long()), best.tolist(), history

    def reset_nfes(self):
        self.nfes = 0


# ----------------------------------------------------- GradientBasedSearch --
class GradientBasedSearch:
    """Adam ascent on the verifier score through a DIFFERENTIABLE denoise_fn / verifier_fn pair
    (:343-438).  Host-side torch only: the its_b200 kernel sampler has no backward pass, so a
    `SamplerDenoiser` is refused; any autograd-capable callables work as in the reference."""

    def __init__(self, n_iterations: int = 20, lr: float = 0.01, verbose: bool = False):
        self.n_iterations = n_iterations
        self.lr = lr
        self.verbose = verbose
        self.nfes = 0

    def search(self, initial_noise: torch.Tensor, denoise_fn: Callable, verifier_fn: Callable,
               device: str = 'cuda', **kwargs) -> Tuple[torch.Tensor, float, Dict[str, Any]]:
        if isinstance(denoise_fn, SamplerDenoiser):
            raise TypeError("GradientBasedSearch differentiates through denoise_fn; the its_b200 kernel sampler "
                            "is inference-only (use RandomSearch / ZeroOrderSearch / PathSearch with it)")
        noise = initial_noise.clone().requires_grad_(True)
        opt = torch.optim.Adam([noise], lr=self.lr)
        history: Dict[str, Any] = {'scores': [], 'grad_norms': []}
        best_noise, best_score = noise.clone(), float('-inf')
        for it in range(self.n_iterations):
            opt.zero_grad()
            score = verifier_fn(denoise_fn(noise, **kwargs), **kwargs)
            self.nfes += 1
            (-score).backward()                               # maximise the score
            history['grad_norms'].append(noise.grad.norm().item())
            opt.step()                                        # the score recorded below belongs to the pre-step noise,
            value = score.item() if isinstance(score, torch.Tensor) else score
            history['scores'].append(value)
            if value > best_score:                            # ... but, as in the reference, the stored noise is post-step
                best_score, best_noise = value, noise.clone().detach()
            if self.verbose:
                print(f"Gradient-Based Search Iteration {it + 1}/{self.n_iterations}: score {value:.4f}")
        return best_noise, best_score, history

    def reset_nfes(self):
        self.nfes = 0
