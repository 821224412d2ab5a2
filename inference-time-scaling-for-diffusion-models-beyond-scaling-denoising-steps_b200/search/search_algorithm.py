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
(or survivors) on the device with one segmented top-k.  In population mode these classes have one path: `search`
runs it with one query (its inputs gain a query axis of length 1) and `_unwrap` hands back query 0's results.  Every
population search draws its initial x_T with `_x_T` and evaluates its members with `_evaluate` (denoise a segment,
score, gather).

FKSteering is not in the reference either: Feynman-Kac steering of Singhal et al. (a population of particles
resampled by verifier potentials on their x0 predictions), in population mode only.

Search over the guidance weight (guided sampler, population mode): RandomSearch, SearchOverPaths and FKSteering take
`guidance` ([N], or [K, N] in `search_batch`), one classifier-free-guidance weight per candidate, path or particle,
which the sampler's step mixes per image (its_ddpm_step_x0_w).  A child of search over paths inherits its parent's
weight and an FK particle its ancestor's, so selection and resampling choose the weight together with the noise.
Every search then sets `last_guidance`, the winner's weight (a list over the queries in `search_batch`).

A rank ensemble (`verifier.EnsembleVerifier`) scores relative to a population: RandomSearch, PathSearch and
SearchOverPaths gather its [n, V] member scores and combine them per query right after the gather, on every rank,
with the segments the selection uses.  ZeroOrderSearch and FKSteering compare scores across populations and refuse
it.

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

    def _check_cand_guidance(self, cand_guidance, n: int):
        if cand_guidance is None:
            return None
        if not getattr(self.sampler, "guided", False):
            raise ValueError("cand_guidance needs the guided sampler: an unguided one has no weight to vary")
        if tuple(cand_guidance.shape) != (n,):
            raise ValueError(f"cand_guidance must be [{n}] (one weight per candidate), got "
                             f"{list(cand_guidance.shape)}")
        return cand_guidance

    def __call__(self, noise: torch.Tensor, show_progress: bool = False, **kwargs) -> torch.Tensor:
        # the reference draws fresh step noise for every candidate (Diffusion.py:96): candidate i of a serial
        # search uses Philox stream i, exactly the stream population mode gives global candidate i
        i = self._calls
        self._calls += 1
        return self.denoise_candidates(noise.unsqueeze(0), i, labels=kwargs.get("labels"))[0]

    def denoise_candidates(self, cands: torch.Tensor, first_cand: int, *, labels=None,
                           t_start: Optional[int] = None, seed: Optional[int] = None, t_stop: int = 0,
                           cand_labels: Optional[torch.Tensor] = None,
                           cand_guidance: Optional[torch.Tensor] = None) -> torch.Tensor:
        """cands [n, B, C, H, W] -> images [n, B, C, H, W]; candidate i is global
        candidate first_cand + i (its Philox streams are keyed by that id).  `t_start` (default T-1) and `t_stop`
        bound the loop as the sampler's own arguments do (a `t_stop` > 0 returns the states step t_stop - 1
        starts from)."""
        t_start = self.sampler.T - 1 if t_start is None else t_start
        return self.denoise_segment(cands, first_cand, t_start=t_start, t_stop=t_stop, labels=labels, seed=seed,
                                    x0=False, cand_labels=cand_labels, cand_guidance=cand_guidance)[0]

    def denoise_segment(self, states: torch.Tensor, first_cand: int, *, t_start: int, t_stop: int,
                        cand_offset: int = 0, labels=None, seed: Optional[int] = None,
                        x0: bool = True, cand_labels: Optional[torch.Tensor] = None,
                        cand_guidance: Optional[torch.Tensor] = None
                        ) -> Tuple[torch.Tensor, Optional[torch.Tensor]]:
        """states [n, B, C, H, W] at step t_start -> (states after step t_stop, x0 predictions of step t_stop or
        None), in chunks of `max_images`.  Candidate i's per-step Philox streams are keyed by
        cand_offset + (first_cand + i) * B + image; every chunk replays the sampler's one step graph.  The guided
        sampler's labels are `cand_labels` [n, B] (int64, one row per candidate) when given, else `labels` (or the
        denoiser's own) [B] for every candidate.  `cand_guidance` [n] (guided sampler): candidate i's guidance weight
        for all its B images, instead of the sampler's `w`."""
        n, B = states.shape[:2]
        if cand_labels is not None and tuple(cand_labels.shape) != (n, B):
            raise ValueError(f"cand_labels must be [{n}, {B}] (one label row per candidate), got "
                             f"{tuple(cand_labels.shape)}")
        cand_guidance = self._check_cand_guidance(cand_guidance, n)
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
            if cand_guidance is not None:
                kw["guidance"] = cand_guidance[i0:i1].repeat_interleave(B)
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


def _require_population(denoise_fn, verifier_fn, search: str) -> Any:
    """`_population_mode`'s kernel verifier, for the searches (and options) that have no callable mode."""
    ver = _population_mode(denoise_fn, verifier_fn)
    if ver is None:
        raise ValueError(f"{search} needs an its_b200 SamplerDenoiser and a kernel verifier's .score "
                         "(population mode)")
    return ver


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


def _no_scores(ver, device) -> torch.Tensor:
    """The score block of a rank that owns no candidates: [0] fp32, or [0, V] for a rank ensemble of V members (its
    gathered scores are the [n, V] member matrix)."""
    shape = (0, len(ver.members)) if getattr(ver, "ranks_population", False) else (0,)
    return torch.empty(shape, dtype=torch.float32, device=device)


def _combine(ver, scores: torch.Tensor, n_seg: int) -> torch.Tensor:
    """One score per candidate from the gathered scores: a rank ensemble ranks its member matrix within each of
    `n_seg` equal segments (one query's population each); any other verifier's scores are returned as they are
    (no copy, no launch)."""
    if not getattr(ver, "ranks_population", False):
        return scores
    return ver.combine(scores, n_seg)


def _refuse_ranks(verifier_fn, search: str, why: str) -> None:
    """Searches that compare scores of different populations cannot use a population-relative verifier."""
    if getattr(getattr(verifier_fn, "__self__", None), "ranks_population", False):
        raise ValueError(f"{search} cannot use a rank ensemble: {why}, and ranks from different populations "
                         "cannot be compared")


def _evaluate(states: torch.Tensor, lo: int, n_total: int, denoise: SamplerDenoiser, ver, *, t_start: int,
              t_stop: int = 0, cand_offset: int = 0, x0: bool = False, seed: int, labels=None,
              cand_labels: Optional[torch.Tensor] = None, cand_guidance: Optional[torch.Tensor] = None,
              n_seg: int = 1) -> Tuple[torch.Tensor, torch.Tensor]:
    """The evaluate step of every population search: denoise this rank's block of members (`states`
    [n_local, B, ...] at step t_start, global ids lo, lo + 1, ...; step noise keyed as in `denoise_segment`) through
    step t_stop, score it and gather the scores.  A segment ending at step 0 scores the finished, clipped samples,
    any other the x0 predictions of step t_stop, which `x0` must then ask for (SearchOverPaths and FKSteering ask
    in their last segment too, so that it replays the step graph of their other segments).  `seed`: the search's
    shared seed, used for the step noise when the denoiser has none of its own (same on every rank).  `labels`:
    shared labels of every member; `cand_labels`: label rows of this rank's members ([n_local, B]);
    `cand_guidance`: their guidance weights ([n_local]), else the sampler's `w`.  A verifier with `uses_labels`
    gets the flat labels the sampler was fed.  Returns (this rank's states after step t_stop, ALL n_total scores);
    a rank ensemble's member scores are combined over `n_seg` equal segments of the population."""
    if states.shape[0] > 0:
        B = states.shape[1]
        out, pred = denoise.denoise_segment(states, lo, t_start=t_start, t_stop=t_stop, cand_offset=cand_offset,
                                            labels=labels, seed=seed, x0=x0, cand_labels=cand_labels,
                                            cand_guidance=cand_guidance)
        judged = (out if t_stop == 0 else pred).reshape(-1, *states.shape[2:])
        if getattr(ver, "uses_labels", False):
            local = ver.score_candidates(judged, B, labels=denoise.image_labels(states.shape[0], labels, cand_labels))
        else:
            local = ver.score_candidates(judged, B)
    else:
        out, local = states, _no_scores(ver, states.device)
    return out, _combine(ver, _gather_scores(local, n_total), n_seg)


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


def _guidance(guidance, K: int, N: int, denoise_fn, search: str, device, batch: bool) -> Optional[torch.Tensor]:
    """Per-member guidance weights, query-major float64 [K * N] on `device`, from `guidance` [N] (every query) or,
    in `search_batch`, [K, N]; None stays None.  Checked on the host before any device work (and after
    `_require_population`): the guided sampler, the shape and finite values."""
    if guidance is None:
        return None
    if not getattr(denoise_fn.sampler, "guided", False):
        raise ValueError(f"{search}: guidance weights need the guided sampler (DiffusionFreeGuidence)")
    g = torch.as_tensor(guidance, dtype=torch.float64).detach().cpu()
    shapes = [(N,), (K, N)] if batch else [(N,)]
    if tuple(g.shape) not in shapes:
        raise ValueError(f"{search}: guidance must be " + " or ".join(str(list(x)) for x in shapes) +
                         f" (one weight per member), got {list(g.shape)}")
    if not bool(torch.isfinite(g).all()):
        raise ValueError(f"{search}: guidance weights must be finite")
    return g.reshape(-1, N).expand(K, N).reshape(K * N).to(device)


def _refuse_guidance(kwargs, search: str) -> None:
    if kwargs.pop("guidance", None) is not None:
        raise ValueError(f"{search} does not search over the guidance weight; use RandomSearch, SearchOverPaths or "
                         "FKSteering")


def _winner_guidance(g: Optional[torch.Tensor], ids: List[int]) -> Optional[List[Optional[float]]]:
    """Weights of the winners (flat population ids, -1 for none) as host floats; None without guidance."""
    if g is None:
        return None
    host = g.tolist()
    return [host[i] if i >= 0 else None for i in ids]


def _rows(rows: Optional[torch.Tensor], lo: int, hi: int) -> Optional[torch.Tensor]:
    return None if rows is None else rows[lo:hi]


def _query(K: int, q: int) -> str:
    """Prefix naming the query in the errors of a batched search (a single search keeps its messages)."""
    return f"query {q}, " if K > 1 else ""


def _one(t: Optional[torch.Tensor]) -> Optional[torch.Tensor]:
    """A single search's input with the query axis of a one-query `search_batch` in front."""
    return None if t is None else t.unsqueeze(0)


def _unwrap(search, history: Optional[Dict[str, Any]] = None) -> Optional[Dict[str, Any]]:
    """The results of a single search from those of a one-query population: query 0's `last_index`,
    `last_guidance` and `last_scores`, and query 0's entry of every history list over the queries."""
    for name in ("last_index", "last_guidance", "last_scores"):
        value = getattr(search, name, None)
        if value is not None:
            setattr(search, name, value[0])
    if history is None:
        return None
    whole = ("rounds", "segments", "unet_image_steps")      # entries of the whole population
    return {k: v if k in whole else v[0] for k, v in history.items()}


def _x_T(cand_noise: Optional[torch.Tensor], seed: int, lo: int, hi: int, shape: Sequence[int], dev) -> torch.Tensor:
    """Initial x_T of members lo ... hi-1 ([hi - lo, *shape] fp32 on `dev`): rows of the injected `cand_noise`
    ([n, *shape]), else Philox draws under TAG_X_T keyed by member id, so any member can be regenerated."""
    if cand_noise is not None:
        return cand_noise[lo:hi].to(dev, torch.float32)
    if hi > lo:
        return philox_normal((hi - lo,) + tuple(shape), seed, lo, TAG_X_T, dev)
    return torch.empty((0,) + tuple(shape), device=dev)


def _per_query(ids: List[int], K: int, size: int) -> List[List[int]]:
    """Flat population ids ([K * k], query q's k at q*k ..., -1 for none) as K lists of ids within their query,
    whose members are q*size ... q*size + size - 1."""
    k = len(ids) // K
    return [[i - q * size if i >= 0 else -1 for i in ids[q * k:(q + 1) * k]] for q in range(K)]


def _lineage(last: int, parents: List[List[int]], m: int = 1) -> List[int]:
    """A member's id in every round, the first to the last, from `last`, its id in the last round: member c of
    round r + 1 descends from member parents[r][c // m] of round r."""
    line = [last]
    for ids in reversed(parents):
        line.append(ids[line[-1] // m])
    return line[::-1]


def _finish(search, history: Dict[str, Any], lineages: List[List[int]], g_rounds: Optional[List[List[float]]],
           size: int, steps: int, B: int, sampler) -> None:
    """The per-query ends of SearchOverPaths and FKSteering.  With guidance (`g_rounds`: the weights of the
    population's members in every round, host lists; None without), history 'lineage_guidance', each winner's
    weight along its lineage (ids within queries of `size` members), and `last_guidance`; then
    'unet_image_steps' and `nfes` from `steps` (UNet steps x members of B images)."""
    search.last_guidance = None
    if g_rounds is not None:
        history['lineage_guidance'] = [[g_rounds[r][q * size + c] for r, c in enumerate(line)]
                                       for q, line in enumerate(lineages)]
        search.last_guidance = [lg[-1] for lg in history['lineage_guidance']]
    history['unet_image_steps'] = steps * B * (2 if getattr(sampler, "guided", False) else 1)
    search.nfes += steps


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
        guidance = kwargs.pop("guidance", None)            # [n] per-candidate guidance weights
        if guidance is not None or _population_mode(denoise_fn, verifier_fn) is not None:
            best, vals = self._search(noise_shape, denoise_fn, verifier_fn, 1, labels=kwargs.get("labels"),
                                      candidate_noise=_one(cand_noise), seed=seed, device=device, guidance=guidance,
                                      batch=False)
            _unwrap(self)
            return (best[0], vals[0]) if self.last_index >= 0 else (None, float('-inf'))
        self.last_guidance = None
        if isinstance(denoise_fn, SamplerDenoiser):
            denoise_fn.reset_calls()
        best_noise, best_score = None, float('-inf')
        for i in range(self.n_candidates):
            noise = cand_noise[i].to(device) if cand_noise is not None else torch.randn(noise_shape, device=device)
            with torch.no_grad():
                denoised = denoise_fn(noise, show_progress=(i == 0), **kwargs)
                self.nfes += 1
            score = verifier_fn(denoised, **kwargs)
            if score > best_score:
                best_score, best_noise = score, noise.clone()
        return best_noise, best_score

    def search_batch(self, noise_shape: Tuple[int, ...], denoise_fn: Callable, verifier_fn: Callable,
                     n_queries: int, *, labels: Optional[torch.Tensor] = None,
                     candidate_noise: Optional[torch.Tensor] = None, seed: Optional[int] = None,
                     device: str = 'cuda', guidance=None) -> Tuple[torch.Tensor, List[float]]:
        """K = `n_queries` independent random searches of `n_candidates` (N) each, evaluated as one population of
        K*N candidates, with one winner per query selected on the device.  Population mode only.

        `labels` [K] or [K, B]: query q's labels (guided sampler; default: the denoiser's own for every query).
        `candidate_noise` [K, N, *noise_shape]: injected candidates.  Query q's candidate i is global candidate
        q*N + i (its x_T draw under TAG_X_T and its step noise are keyed by that id), so an unguided batch of K
        searches draws and scores exactly the population of RandomSearch(K*N).search with the same seed.
        `guidance` [N] or [K, N] (guided sampler): candidate i of query q runs at weight guidance[q, i] (or [i]).
        Returns (best_noise [K, *noise_shape], best_scores); sets `last_scores` [K, N] (device), `last_index`
        (within-query indices), `last_guidance` (the winners' weights, None without `guidance`) and `last_seed`.
        A query with no rankable score gets a NaN row, -inf and -1 (and weight None)."""
        return self._search(noise_shape, denoise_fn, verifier_fn, n_queries, query_labels=labels,
                            candidate_noise=candidate_noise, seed=seed, device=device, guidance=guidance)

    def _search(self, noise_shape, denoise_fn, verifier_fn, K: int, *, labels=None, query_labels=None,
                candidate_noise=None, seed=None, device='cuda', guidance=None,
                batch: bool = True) -> Tuple[torch.Tensor, List[float]]:
        """`search_batch`, and `search` in population mode: K queries of N candidates as one population sharded over
        the ranks, every winner selected by one segmented top-k (k = 1 per query).  `labels`: shared labels of every
        candidate (a single search's); `query_labels`: one label row per query (`search_batch`'s `labels`); `batch`:
        `guidance` may be [K, N].  Every argument is checked before any device work."""
        K = _check_queries(K, noise_shape, query_labels)
        ver = _require_population(denoise_fn, verifier_fn, "RandomSearch")
        N, shape = self.n_candidates, tuple(noise_shape)
        _check_shape("candidate_noise", candidate_noise, (K, N) + shape)
        guidance = _guidance(guidance, K, N, denoise_fn, "RandomSearch", device, batch)
        denoise_fn.reset_calls()
        dist, rank, world = _dist()
        dev = torch.device(device)
        seed = _shared_seed(seed, dev)
        self.last_seed = seed
        n = K * N
        cand = None if candidate_noise is None else candidate_noise.reshape((n,) + shape)
        rows = _label_rows(query_labels, K, N, shape[0], dev)
        lo, hi = _shard(n, rank, world)
        with torch.no_grad():
            _, scores = _evaluate(_x_T(cand, seed, lo, hi, shape, dev), lo, n, denoise_fn, ver,
                                  t_start=denoise_fn.sampler.T - 1, seed=seed, labels=labels,
                                  cand_labels=_rows(rows, lo, hi), cand_guidance=_rows(guidance, lo, hi), n_seg=K)
        self.nfes += n
        self.last_scores = scores.view(K, N)
        idx, val = _topk_device(scores, 1, n_seg=K)
        ids, vals = idx.tolist(), val.tolist()
        self.last_guidance = _winner_guidance(guidance, ids)
        self.last_index = [own[0] for own in _per_query(ids, K, N)]
        best = torch.full((K,) + shape, float('nan'), dtype=torch.float32, device=dev)
        for q, i in enumerate(ids):
            if i >= 0:   # every rank regenerates the winner from its key (or its row): no broadcast needed
                best[q] = _x_T(cand, seed, i, i + 1, shape, dev)[0]
        return best, vals

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
        _refuse_ranks(verifier_fn, "ZeroOrderSearch", "it compares each round's best with the best of earlier "
                      "rounds")
        _refuse_guidance(kwargs, "ZeroOrderSearch")
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
                    _, scores = _evaluate(local, lo + it * K, K, denoise_fn, ver, t_start=denoise_fn.sampler.T - 1,
                                          seed=seed, labels=kwargs.get("labels"))
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
        _refuse_guidance(kwargs, "PathSearch")
        variations = kwargs.pop("variations", None)   # [n_paths, *shape] injected N(0,1) draws
        seed = kwargs.pop("seed", None)
        restart = bool(kwargs.pop("restart", False))
        ver = _require_population(denoise_fn, verifier_fn, "PathSearch with restart=True") if restart else \
            _population_mode(denoise_fn, verifier_fn)
        best_noise, best_score = initial_noise.clone(), float('-inf')
        history: Dict[str, Any] = {'scores': [], 'injection_points': []}
        P = self.n_paths
        self.last_index = -1                # path index of the returned noise
        if isinstance(denoise_fn, SamplerDenoiser):
            denoise_fn.reset_calls()
        if ver is None:
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
        T = denoise_fn.sampler.T
        t_start = T - 1
        if restart:
            # pivot trajectory T-1 .. injection_step (exclusive) on every rank, unclipped
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
            _, scores = _evaluate(perturbed(lo, hi), lo, P, denoise_fn, ver, t_start=t_start, seed=seed,
                                  labels=kwargs.get("labels"))
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
    injected re-noising draws), `guidance` ([N] guidance weights of the initial paths, guided sampler: a child
    runs at its parent's weight; history 'lineage_guidance' holds the winner's weight in every round and
    `last_guidance` the winner's weight).  `last_index` is the winner's initial path id, `last_seed` the search
    seed.
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
        fwd_noise = kwargs.pop("forward_noise", None)
        images, best, history = self._search(
            noise_shape, denoise_fn, verifier_fn, 1, labels=kwargs.get("labels"),
            candidate_noise=_one(kwargs.pop("candidate_noise", None)),
            forward_noise=None if fwd_noise is None else [_one(f) for f in fwd_noise], seed=kwargs.pop("seed", None),
            device=device, guidance=kwargs.pop("guidance", None), batch=False)
        return images[0], best[0], _unwrap(self, history)

    def search_batch(self, noise_shape: Tuple[int, ...], denoise_fn: Callable, verifier_fn: Callable,
                     n_queries: int, *, labels: Optional[torch.Tensor] = None,
                     candidate_noise: Optional[torch.Tensor] = None, forward_noise=None, seed: Optional[int] = None,
                     device: str = 'cuda', guidance=None) -> Tuple[torch.Tensor, List[float], Dict[str, Any]]:
        """K = `n_queries` independent searches over paths evaluated as one population: K*N paths in stage 0 and
        K*N*M children per round, with the N survivors (and at the end the winner) of every query selected on the
        device by one segmented top-k.  Population mode only.

        `labels` [K] or [K, B]: query q's labels (guided sampler; default: the denoiser's own for every query).
        `candidate_noise` [K, N, *noise_shape] and `forward_noise` [rounds][K, N*M, *noise_shape]: injected draws.
        Query q's path i is global path q*N + i and its child c global child q*N*M + c; x_T, step noise and
        re-noising draws are keyed by those ids, so K = 1 is `search` and a query's result does not depend on
        the other queries, the rank count or `max_images`.
        `guidance` [N] or [K, N] (guided sampler): path i of query q starts at weight guidance[q, i] (or [i]); its
        children, and theirs, keep it.
        Returns (best_images [K, *noise_shape], best_scores, history): history 'rounds' as in `search`; 'scores',
        'survivors' and 'lineage' (and with `guidance` 'lineage_guidance') are lists over the queries, with
        within-query ids; 'unet_image_steps' is the whole batch's.  `last_index` is the list of the winners' initial
        path ids, `last_guidance` of their weights.  A query whose children cannot be ranked raises ValueError naming
        the query and the round."""
        return self._search(noise_shape, denoise_fn, verifier_fn, n_queries, query_labels=labels,
                            candidate_noise=candidate_noise, forward_noise=forward_noise, seed=seed, device=device,
                            guidance=guidance)

    def _search(self, noise_shape, denoise_fn, verifier_fn, K: int, *, labels=None, query_labels=None,
                candidate_noise=None, forward_noise=None, seed=None, device='cuda', guidance=None,
                batch: bool = True) -> Tuple[torch.Tensor, List[float], Dict[str, Any]]:
        """`search_batch`, and `search` with one query: K queries as one population sharded over the ranks.
        `labels`: shared labels of every member (a single search's); `query_labels`: one label row per query
        (`search_batch`'s `labels`); `guidance` ([N], or with `batch` [K, N]): the initial paths' weights, which
        every child inherits from its parent (re-indexed by the same device survivor ids the expansion reads).
        Every argument, and the parameters against sampler.T, is checked before any device work."""
        K = _check_queries(K, noise_shape, query_labels)
        ver = _require_population(denoise_fn, verifier_fn, "SearchOverPaths")
        N, M = int(self.n_beams), int(self.n_children)
        if N < 1 or M < 1:
            raise ValueError(f"n_beams={N} and n_children={M} must be >= 1")
        smp = denoise_fn.sampler
        T = smp.T
        rounds = path_rounds(T, self.start_step, self.delta_f, self.delta_b)
        NM, shape = N * M, tuple(noise_shape)
        _check_shape("candidate_noise", candidate_noise, (K, N) + shape)
        guidance = _guidance(guidance, K, N, denoise_fn, "SearchOverPaths", device, batch)
        if forward_noise is not None:
            if len(forward_noise) < len(rounds):
                raise ValueError(f"forward_noise has {len(forward_noise)} rounds, the schedule {len(rounds)}")
            for r in range(len(rounds)):
                _check_shape(f"forward_noise[{r}]", forward_noise[r], (K, NM) + shape)
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
        g_rows = guidance                             # weight of each row of `parents`
        g_rounds = None if guidance is None else []   # children's weights per round
        steps = 0                                     # UNet steps x candidates
        with torch.no_grad():
            # stage 0: K*N paths from x_T down to the states at step start_step
            n_p = K * N
            lo, hi = _shard(n_p, rank, world)
            cand = None if candidate_noise is None else candidate_noise.reshape((n_p,) + shape)
            local = _x_T(cand, seed, lo, hi, shape, dev)
            s0 = rounds[0][0]
            if s0 < T - 1 and hi > lo:
                local = denoise_fn.denoise_candidates(local, lo, labels=labels, seed=seed, t_stop=s0 + 1,
                                                      cand_labels=_rows(path_labels, lo, hi),
                                                      cand_guidance=_rows(g_rows, lo, hi))
            steps += n_p * (T - 1 - s0)
            parents = _gather_states(local.contiguous(), n_p)
            parent_idx = torch.arange(n_p, dtype=torch.int32, device=dev)
            n_c = K * NM
            lo, hi = _shard(n_c, rank, world)
            for r, (s, sp, e) in enumerate(rounds):
                ratio = float(abar[sp] / abar[s])
                a, b = math.sqrt(ratio), math.sqrt(1. - ratio)
                if g_rows is not None:                # child c runs at the weight of its parent parent_idx[c // M]
                    g_rows = g_rows.index_select(0, parent_idx.long()).repeat_interleave(M)
                    g_rounds.append(g_rows.tolist())
                if hi > lo:
                    z = None if forward_noise is None else forward_noise[r].reshape((n_c,) + shape)[lo:hi]
                    kids = path_expand(parents.reshape(parents.shape[0], -1), parent_idx, M, lo, hi - lo, a, b,
                                       z=None if z is None else z.reshape(hi - lo, -1), seed=seed,
                                       cand_id0=(r + 1) * ROUND_STRIDE, tag=TAG_FORWARD).view((hi - lo,) + shape)
                else:
                    kids = torch.empty((0,) + shape, device=dev)
                states, scores = _evaluate(kids, lo, n_c, denoise_fn, ver, t_start=sp, t_stop=e,
                                           cand_offset=(r + 1) * ROUND_STRIDE, x0=True, seed=seed, labels=labels,
                                           cand_labels=_rows(child_labels, lo, hi),
                                           cand_guidance=_rows(g_rows, lo, hi), n_seg=K)
                steps += n_c * (sp - e + 1)
                history['rounds'].append((s, sp, e))
                for q, row in enumerate(scores.view(K, NM).tolist()):
                    history['scores'][q].append(row)
                parents = _gather_states(states.contiguous(), n_c)
                # survivors (k = N per query) or the winner (k = 1): flat child ids, passed on as parents as they are
                parent_idx, best = _topk_device(scores, N if e > 0 else 1, n_seg=K)
                for q, own in enumerate(_per_query(parent_idx.tolist(), K, NM)):
                    if min(own) >= 0:
                        history['survivors'][q].append(own)
                    elif e > 0:
                        raise ValueError(f"{_query(K, q)}round {r}: only {sum(i >= 0 for i in own)} of {NM} children "
                                         f"have a score that can be ranked; {N} survivors are needed")
                    else:
                        raise ValueError(f"{_query(K, q)}last round: none of the {NM} finished samples has a score "
                                         "that can be ranked")
        # lineage of each winner: child id in every round, back to its initial path
        lineages = [_lineage(surv[-1][0], surv[:-1], M) for surv in history['survivors']]
        history['lineage'] = [{'path': line[0] // M, 'children': line} for line in lineages]
        self.last_index = [lin['path'] for lin in history['lineage']]
        _finish(self, history, lineages, g_rounds, NM, steps, B, smp)
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
    keyword extensions: `seed`, `labels`, `candidate_noise`, `guidance` ([N] guidance weights of the particles,
    guided sampler: a particle keeps its ancestor's weight at every resampling).  history: 'segments'; per
    resampling 'scores' (N), 'ancestors' (N particle ids) and 'ess'; 'lineage', the winner's particle id in every
    segment (lineage[0] is its x_T id); with `guidance` 'lineage_guidance', its weight in every segment (and
    `last_guidance` the winner's weight); 'unet_image_steps'.  `last_index` is the winner's x_T id, `last_seed` the search seed; `nfes` counts
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
        images, best, history = self._search(
            noise_shape, denoise_fn, verifier_fn, 1, labels=kwargs.get("labels"),
            candidate_noise=_one(kwargs.pop("candidate_noise", None)), seed=kwargs.pop("seed", None), device=device,
            guidance=kwargs.pop("guidance", None), batch=False)
        return images[0], best[0], _unwrap(self, history)

    def search_batch(self, noise_shape: Tuple[int, ...], denoise_fn: Callable, verifier_fn: Callable,
                     n_queries: int, *, labels: Optional[torch.Tensor] = None,
                     candidate_noise: Optional[torch.Tensor] = None, seed: Optional[int] = None,
                     device: str = 'cuda', guidance=None) -> Tuple[torch.Tensor, List[float], Dict[str, Any]]:
        """K = `n_queries` independent FK-steering searches evaluated as one population of K*N particles, resampled
        per query by one segmented kernel launch, with every query's winner selected on the device by one segmented
        top-k.  Population mode only.

        `labels` [K] or [K, B]: query q's labels (guided sampler; default: the denoiser's own for every query).
        `candidate_noise` [K, N, *noise_shape]: injected x_T.  Query q's particle j is global particle q*N + j
        (its x_T draw and step noise are keyed by that id, its resampling uniform by q, ancestors never cross
        queries), so K = 1 is `search`, query 0 is the single search with query 0's inputs, and a query's result
        does not depend on the other queries' inputs, the rank count or `max_images`.
        `guidance` [N] or [K, N] (guided sampler): particle j of query q starts at weight guidance[q, j] (or [j]) and
        every resampling hands a particle its ancestor's weight.
        Returns (best_images [K, *noise_shape], best_scores, history): 'segments' as in `search`; 'scores',
        'ancestors', 'ess' and 'lineage' (and with `guidance` 'lineage_guidance') are lists over the queries, with
        within-query ids; 'unet_image_steps' is the whole batch's.  `last_index` is the list of the winners' x_T ids,
        `last_guidance` of their weights.  A query none of whose particles can
        be weighted raises ValueError naming the query and the resampling round."""
        return self._search(noise_shape, denoise_fn, verifier_fn, n_queries, query_labels=labels,
                            candidate_noise=candidate_noise, seed=seed, device=device, guidance=guidance)

    def _search(self, noise_shape, denoise_fn, verifier_fn, K: int, *, labels=None, query_labels=None,
                candidate_noise=None, seed=None, device='cuda', guidance=None,
                batch: bool = True) -> Tuple[torch.Tensor, List[float], Dict[str, Any]]:
        """`search_batch`, and `search` with one query: K queries of N particles as one population sharded over the
        ranks.  `labels`: shared labels of every particle (a single search's); `query_labels`: one label row per
        query (`search_batch`'s `labels`); `guidance` ([N], or with `batch` [K, N]): the particles' weights, which
        follow their ancestors (`index_select` with the same device ancestor ids as the states).  Every argument,
        and the parameters against sampler.T, is checked before any device work."""
        K = _check_queries(K, noise_shape, query_labels)
        _refuse_ranks(verifier_fn, "FKSteering", "it weights particles by the change of their reward between "
                      "resamplings")
        ver = _require_population(denoise_fn, verifier_fn, "FKSteering")
        N = int(self.n_particles)
        if N < 1:
            raise ValueError(f"n_particles={self.n_particles} must be >= 1")
        if not (math.isfinite(float(self.lam)) and float(self.lam) >= 0.0):
            raise ValueError(f"lam={self.lam} must be finite and >= 0")
        smp = denoise_fn.sampler
        segments = fk_segments(smp.T, self.start_step, self.resample_interval)
        shape = tuple(noise_shape)
        _check_shape("candidate_noise", candidate_noise, (K, N) + shape)
        guidance = _guidance(guidance, K, N, denoise_fn, "FKSteering", device, batch)
        n = K * N
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
        g = guidance                                  # particle weights now,
        g_segments = None if guidance is None else []   # and in every segment
        with torch.no_grad():
            cand = None if candidate_noise is None else candidate_noise.reshape((n,) + shape)
            local = _x_T(cand, seed, lo, hi, shape, dev)
            for r, (t_start, t_stop) in enumerate(segments):
                if g is not None:
                    g_segments.append(g.tolist())
                local, scores = _evaluate(local, lo, n, denoise_fn, ver, t_start=t_start, t_stop=t_stop,
                                          cand_offset=r * ROUND_STRIDE, x0=True, seed=seed, labels=labels,
                                          cand_labels=_rows(rows, lo, hi), cand_guidance=_rows(g, lo, hi), n_seg=K)
                steps += n * (t_start - t_stop + 1)
                states = _gather_states(local.contiguous(), n)
                if t_stop == 0:
                    break
                anc, carried, ess = resample_systematic(scores, carried, self.lam, K, seed, r)
                ids, vals, ess_q = _per_query(anc.tolist(), K, N), scores.view(K, N).tolist(), ess.tolist()
                for q, own in enumerate(ids):
                    if own[0] < 0:
                        raise ValueError(f"{_query(K, q)}resampling round {r}: none of the {N} particles has a "
                                         "finite score to weight")
                    history['scores'][q].append(vals[q])
                    history['ancestors'][q].append(own)
                    history['ess'][q].append(ess_q[q])
                local = states.index_select(0, anc[lo:hi].long())
                if g is not None:
                    g = g.index_select(0, anc.long())
            idx, best = _topk_device(scores, 1, n_seg=K)
            winners = _per_query(idx.tolist(), K, N)
        history['lineage'] = []
        for q, own in enumerate(winners):
            if own[0] < 0:
                raise ValueError(f"{_query(K, q)}last segment: none of the {N} finished samples has a score that can "
                                 "be ranked")
            history['lineage'].append(_lineage(own[0], history['ancestors'][q]))
        self.last_index = [line[0] for line in history['lineage']]
        _finish(self, history, history['lineage'], g_segments, N, steps, B, smp)
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
