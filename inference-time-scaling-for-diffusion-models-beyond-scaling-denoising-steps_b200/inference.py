"""Inference driver of the sampling path: the callers on either side of the sampler in the
reference (SURVEY.md §8f rows 1 and 3), without Hydra.

  * load_config              — config/inference_config.yaml keys, `key=value` overrides
                               (abstract_metrics_from_pretrained_ddpm.py:649-694 reads them through Hydra)
  * load_checkpoint_state_dict, detect_checkpoint_T, extended_time_table, create_and_load_model,
    create_sampler           — abstract_metrics_from_pretrained_ddpm.py:126-379
  * sample_with_metrics_tracking — Diffusion/Train.py:25-166: the ancestral loop with the metric
    calculators called every `metric_interval` steps.  The reference drives `p_mean_variance` step by
    step from Python; here the steps between two metric points run as one device-resident segment of
    the sampler's step graph (`forward(..., t_start=a, t_stop=b)`), so tracking costs nothing between
    metric points.  Calculators are duck-typed (FID / IS / CLIP weights are third-party downloads the
    reference fetches at run time, SURVEY.md §8c): pass the reference's own objects, or None.
  * run_search               — config-driven search (random / zero_order / path / search_over_paths /
                               fk_steering) with the kernel verifiers
  * save_image_grid          — torchvision.utils.save_image grid as the reference writes it (:621-628)

    python -m its_b200.inference config/inference_config.yaml T=1000 img_size=32 batch_size=64
"""
from __future__ import annotations

import math
import os
import sys
from collections import OrderedDict
from typing import Any, Dict, Iterable, List, Optional, Tuple

import torch
from torch import nn


# --------------------------------------------------------------- config ------
def _parse_scalar(text: str) -> Any:
    import yaml
    return yaml.safe_load(text)


def load_config(path: Optional[str], overrides: Iterable[str] = ()) -> Dict[str, Any]:
    """YAML file + `key=value` overrides (dotted keys address nested dicts), the way the reference's
    Hydra entry point is invoked (`batch_size=32 metric_interval=20`, :656).  The `hydra:` block of the
    reference's config file is ignored."""
    import yaml
    cfg: Dict[str, Any] = {}
    if path is not None:
        with open(path) as f:
            cfg = yaml.safe_load(f) or {}
    cfg.pop("hydra", None)
    for ov in overrides:
        if "=" not in ov:
            raise ValueError(f"override {ov!r} is not key=value")
        key, val = ov.split("=", 1)
        node = cfg
        parts = key.split(".")
        for part in parts[:-1]:
            node = node.setdefault(part, {})
        node[parts[-1]] = _parse_scalar(val)
    # yaml reads 1e-4 as a string (no dot): the reference's OmegaConf does the same and the samplers
    # receive floats only because torch.linspace coerces; coerce here.
    for k in ("beta_1", "beta_T", "dropout", "w"):
        if isinstance(cfg.get(k), str):
            cfg[k] = float(cfg[k])
    return cfg


# ----------------------------------------------------------- checkpoints -----
def load_checkpoint_state_dict(checkpoint_path: str, device) -> "OrderedDict[str, torch.Tensor]":
    """State dict of a checkpoint file: a bare state dict, {'state_dict': ...}, or a pickled module;
    DataParallel's `module.` prefix is stripped (:126-159)."""
    if not os.path.exists(checkpoint_path):
        raise FileNotFoundError(f"Checkpoint not found: {checkpoint_path}")
    try:
        checkpoint = torch.load(checkpoint_path, map_location=device, weights_only=True)
    except Exception:
        checkpoint = torch.load(checkpoint_path, map_location=device, weights_only=False)
    if isinstance(checkpoint, dict) and "state_dict" in checkpoint:
        state_dict = checkpoint["state_dict"]
    elif isinstance(checkpoint, dict):
        state_dict = checkpoint
    elif hasattr(checkpoint, "state_dict"):
        state_dict = checkpoint.state_dict()
    else:
        raise ValueError("Could not extract state_dict from checkpoint")
    if any(k.startswith("module.") for k in state_dict.keys()):
        state_dict = OrderedDict((k[7:] if k.startswith("module.") else k, v) for k, v in state_dict.items())
    return state_dict


TIME_TABLE_KEY = "time_embedding.timembedding.0.weight"


def detect_checkpoint_T(state_dict: Dict[str, torch.Tensor]) -> Optional[int]:
    """T of a checkpoint whose time embedding is a [T, d_model] table (the conditional net,
    ModelCondition.py:24-46, and checkpoints of the older unconditional net); None for the functional
    embedding (Model.py:15-93), whose first tensor is a Linear weight [4ch, ch].  The rule is the
    reference's (:162-188): more than 500 rows means "table" — so a functional checkpoint with
    ch = 128 (4ch = 512) is reported as T = 512 there too; create_and_load_model compares shapes instead."""
    w = state_dict.get(TIME_TABLE_KEY)
    if w is not None and w.shape[0] > 500:
        return int(w.shape[0])
    return None


def _sinusoid_table(T: int, d_model: int) -> torch.Tensor:
    freq = torch.exp(-(torch.arange(0, d_model, step=2) / d_model * math.log(10000)))
    ang = torch.arange(T).float()[:, None] * freq[None, :]
    return torch.stack([torch.sin(ang), torch.cos(ang)], dim=-1).view(T, d_model)


def extended_time_table(checkpoint_T: int, current_T: int, d_model: int, strategy: str = "interpolate") -> torch.Tensor:
    """The [current_T, d_model] sinusoid table the reference installs when a T = checkpoint_T table
    checkpoint is sampled with a longer schedule (:191-262).  "interpolate": rows below checkpoint_T are
    the sinusoids scaled by checkpoint_T / current_T, the rest plain sinusoids; anything else: plain."""
    emb = _sinusoid_table(current_T, d_model)
    if strategy == "interpolate" and checkpoint_T < current_T:
        emb = emb.clone()
        emb[:checkpoint_T] = emb[:checkpoint_T] * (checkpoint_T / current_T)
    return emb


def install_time_table(model: nn.Module, table: torch.Tensor) -> None:
    """Replace the time-embedding table of a table-based net (ModelCondition.UNet) in place."""
    target = getattr(model, "module", model)
    seq = target.time_embedding.timembedding
    if not isinstance(seq[0], nn.Embedding):
        raise TypeError("this net has a functional time embedding (no table to extend): any T works as is")
    dev = seq[0].weight.device
    seq[0] = nn.Embedding.from_pretrained(table.to(dev), freeze=False)
    if hasattr(target, "invalidate_plans"):
        target.invalidate_plans()


def create_and_load_model(config: Dict[str, Any], device) -> nn.Module:
    """Build the UNet the config names and load `checkpoint_path` into it (:265-357).  `num_labels` in
    the config selects the conditional net.  A table checkpoint with a different T loses its
    time-embedding tensors (the rest loads non-strictly): the functional embedding of Model.UNet needs
    no table, the conditional net gets `extended_time_table`.  `checkpoint_path: null` keeps the
    random initialisation (synthetic runs)."""
    T = int(config["T"])
    if config.get("num_labels") is not None:
        from .DiffusionFreeGuidence import UNet as CondUNet
        model = CondUNet(T=T, num_labels=int(config["num_labels"]), ch=config["channel"], ch_mult=config["channel_mult"],
                         num_res_blocks=config["num_res_blocks"], dropout=config["dropout"])
    else:
        from .Diffusion import UNet
        model = UNet(T=T, ch=config["channel"], ch_mult=config["channel_mult"], attn=config["attn"],
                     num_res_blocks=config["num_res_blocks"], dropout=config["dropout"])
    model = model.to(device)
    path = config.get("checkpoint_path")
    if path:
        sd = load_checkpoint_state_dict(path, device)
        own = model.state_dict()
        ckpt_w, own_w = sd.get(TIME_TABLE_KEY), own.get(TIME_TABLE_KEY)
        # The reference decides "table checkpoint" by `rows > 500` (detect_checkpoint_T), which also fires
        # for the functional embedding's Linear [4ch, ch] at ch = 128 and then breaks that layer; here a
        # checkpoint tensor of the model's own shape is simply loaded, and only a differently shaped
        # first tensor (a table of another T, or a table for the functional net) is dropped.
        if ckpt_w is not None and own_w is not None and tuple(ckpt_w.shape) != tuple(own_w.shape):
            ckpt_T = int(ckpt_w.shape[0])
            for k in [k for k in sd if k.startswith("time_embedding")]:
                del sd[k]
            missing, unexpected = model.load_state_dict(sd, strict=False)
            if isinstance(model.time_embedding.timembedding[0], nn.Embedding):
                install_time_table(model, extended_time_table(ckpt_T, T, own_w.shape[1],
                                                              config.get("time_embedding_strategy", "interpolate")))
            missing = [k for k in missing if not k.startswith("time_embedding")]
        else:
            missing, unexpected = model.load_state_dict(sd, strict=False)
        if unexpected:
            print(f"Warning: Unexpected keys: {list(unexpected)}")
        if missing:
            print(f"Warning: Missing keys: {list(missing)}")
    # Raw feature maps in fp16 instead of bf16 (5x smaller error, DESIGN.md section 5) need bounded activations:
    # `residual_fp16: auto` (default) turns it on for loaded checkpoints (trained weights) and leaves random
    # initialisations, whose state can grow past fp16's range, on bf16; true / false force it.
    # `auto` never turns it on for schedules longer than the T = 1000 the checkpoints of this repository are trained
    # on (an untrained or mismatched net drives |x_t| to ~2e5 at T = 2000, past fp16's 65504: the overflow would
    # only surface as the sampler's "nan in tensor." assertion at the end of the trajectory).
    mode = config.get("residual_fp16", "auto")
    model.residual_fp16 = (bool(path) and int(config.get("T", 1000)) <= 1000) if mode == "auto" else bool(mode)
    # `precision`: 16bit (default: tensor-core path, samples within 2e-2 of the fp32 reference) | fp32 (CUDA-core
    # fp32 kernels, samples within 1e-4: the parity path)
    model.precision = str(config.get("precision", "16bit")).lower()
    print(f"its_b200: precision={model.precision} residual_fp16={model.residual_fp16} (residual_fp16: {mode})")
    return model.eval()


def create_sampler(model: nn.Module, config: Dict[str, Any], device):
    """GaussianDiffusionSampler for the model (:360-379); the guided one when the config has `w`."""
    if getattr(model, "is_conditional", False):
        from .DiffusionFreeGuidence import GaussianDiffusionSampler as Guided
        return Guided(model, config["beta_1"], config["beta_T"], int(config["T"]), w=float(config.get("w", 0.0))).to(device)
    from .Diffusion import GaussianDiffusionSampler
    return GaussianDiffusionSampler(model, config["beta_1"], config["beta_T"], int(config["T"])).to(device)


# ------------------------------------------------------ metrics tracking -----
def metric_points(T: int, metric_interval: int) -> List[int]:
    """Time steps after which the reference evaluates the metrics: time_step % interval == 0
    (Diffusion/Train.py:79), in loop order T-1 ... 0."""
    return [t for t in reversed(range(T)) if t % metric_interval == 0 or t == 0]


def sample_with_metrics_tracking(sampler, x_T: torch.Tensor, fid_calculator=None, is_calculator=None,
                                 clip_calculator=None, real_features: Optional[torch.Tensor] = None,
                                 real_clip_features: Optional[torch.Tensor] = None,
                                 mu_real: Optional[torch.Tensor] = None, sigma_real: Optional[torch.Tensor] = None,
                                 metric_interval: int = 5, device: str = "cuda", *, labels=None, noise=None,
                                 seed: Optional[int] = None
                                 ) -> Tuple[torch.Tensor, List[Tuple[int, float, float, float]]]:
    """Diffusion/Train.py:25-166 — returns (x_0 clipped to [-1, 1], [(time_step, fid, is, clip), ...]).
    Same calculator protocol: `fid_calculator.extract_features_from_tensor(x01)` /
    `.calculate_frechet_distance(mu_r, sigma_r, mu_f, sigma_f)`, `is_calculator.compute_is(x01) ->
    (mean, std)`, `clip_calculator.extract_features_from_tensor` / `.compute_clip_score_with_features`;
    a metric whose calculator is None (or raises) is recorded as NaN, as in the reference.
    Keyword-only extensions: `labels` (guided sampler), `noise` [T, *x_T.shape] (injected Gaussians,
    parity runs), `seed` (Philox stream)."""
    T = sampler.T
    if seed is None:
        seed = int(torch.randint(0, 2 ** 62, (1,)).item())
    history: List[Tuple[int, float, float, float]] = []
    x_t = x_T
    first = T - 1
    kw: Dict[str, Any] = dict(noise=noise, seed=seed, clip=False)
    with torch.no_grad():
        for t_metric in metric_points(T, metric_interval):
            # steps first ... t_metric as one device segment; the result is x after step t_metric
            x_t = sampler(x_t, labels, t_start=first, t_stop=t_metric, **kw) if labels is not None else \
                sampler(x_t, t_start=first, t_stop=t_metric, **kw)
            first = t_metric - 1
            x01 = torch.clamp(x_t * 0.5 + 0.5, 0, 1)
            fid_value = is_value = clip_value = float("nan")
            if fid_calculator is not None:
                try:
                    fake = fid_calculator.extract_features_from_tensor(x01)
                    if mu_real is None:
                        mu_real = real_features.mean(dim=0)
                        if real_features.shape[0] > 1:
                            sigma_real = torch.cov(real_features.T, correction=0)
                        else:
                            sigma_real = torch.eye(real_features.shape[1], dtype=torch.float64,
                                                   device=real_features.device) * 1e-6
                        mu_real, sigma_real = mu_real.to(device), sigma_real.to(device)
                    mu_fake = fake.mean(dim=0)
                    if fake.shape[0] > 1:
                        sigma_fake = torch.cov(fake.T, correction=0)
                    else:
                        sigma_fake = torch.eye(fake.shape[1], dtype=torch.float64, device=fake.device) * 1e-6
                    fid_value = fid_calculator.calculate_frechet_distance(mu_real, sigma_real, mu_fake, sigma_fake)
                except Exception as e:  # the reference reports and carries on (:104-105)
                    print(f"\nWarning: FID calculation failed at step {t_metric}: {e}")
            if is_calculator is not None:
                try:
                    is_value, _ = is_calculator.compute_is(x01)
                except Exception as e:
                    print(f"\nWarning: IS calculation failed at step {t_metric}: {e}")
            if clip_calculator is not None:
                try:
                    feats = clip_calculator.extract_features_from_tensor(x01)
                    clip_value = clip_calculator.compute_clip_score_with_features(real_clip_features, feats)
                except Exception as e:
                    print(f"\nWarning: CLIP Score calculation failed at step {t_metric}: {e}")
                    clip_value = float("nan")
            history.append((t_metric, fid_value, is_value, clip_value))
    return torch.clamp(x_t, -1, 1), history


# -------------------------------------------------------------- search -------
DENOISING_VERIFIERS = {"denoising": "likelihood", "diffusion_classifier": "class"}


def make_verifier(name: str, sampler=None, *, n_levels: int = 8, seed: int = 0, max_images: int = 256):
    """Verifier by config name.  `denoising` / `diffusion_classifier` are the sampler's own model scoring its
    samples (DenoisingVerifier, kinds likelihood / class) and need `sampler`; the class form needs the guided net."""
    from .search import verifier as V
    table = {"oracle": V.OracleVerifier, "self_supervised": V.SelfSupervisedVerifier, "aesthetic": V.AestheticPredictor}
    if name in DENOISING_VERIFIERS:
        if sampler is None:
            raise ValueError(f"verifier {name!r} scores with the diffusion model: pass the sampler")
        if name == "diffusion_classifier" and not getattr(sampler._unet(), "is_conditional", False):
            raise ValueError("verifier 'diffusion_classifier' needs the conditional net (num_labels in the config): "
                             "it compares the conditional and unconditional denoising errors")
        return V.DenoisingVerifier(sampler, DENOISING_VERIFIERS[name], n_levels=n_levels, seed=seed,
                                   max_images=max_images)
    if name not in table:
        raise ValueError(f"verifier {name!r}: choose one of {sorted(table)} (the CLIP-backed verifiers need "
                         "third-party weights that are not bundled)")
    return table[name]()


def run_search(sampler, config: Dict[str, Any], device, *, labels=None, seed: Optional[int] = None):
    """`search:` block of the config -> (best_noise, best_score, images of the best candidate).
    Keys: algorithm (random | zero_order | path | search_over_paths | fk_steering), verifier (oracle | self_supervised |
    aesthetic | denoising | diffusion_classifier; the last two score with the sampler's own model at score_levels
    (8) noise levels drawn from score_seed (0), in chunks of max_images UNet images), n_candidates / n_neighbors / n_iterations / lambda_radius / n_paths / injection_step / noise_scale
    (defaults: the reference constructors', search_algorithm.py:24,98-100,246-248), batch_size,
    img_size.  search_over_paths takes n_beams (4), n_children (4), start_step (800), delta_f (50) and
    delta_b (100), and returns the winner's initial x_T with the images the search itself finished (the winner's
    path is re-noised along the way: denoising its x_T again would not reproduce it).  fk_steering takes
    n_particles (4), start_step (800), resample_interval (100) and fk_lambda (10.0), and returns the same pair
    (a resampled particle's trajectory is not the one its x_T alone would give).
    `n_queries` (K, default 1) > 1 runs K independent random / search_over_paths / fk_steering searches as one
    population (`search_batch`): `labels` is then [K] or [K, B] (one row per query), and the results are stacked over the
    queries (best_noise and images [K, B, 3, H, W], a list of K scores).
    With torch.distributed initialised the candidates are sharded over the ranks."""
    from .search import search_algorithm as S
    sc = dict(config.get("search") or {})
    algo = sc.get("algorithm", "random")
    B, H = int(config.get("batch_size", 1)), int(config["img_size"])
    shape = (B, 3, H, H)
    ver = make_verifier(sc.get("verifier", "oracle"), sampler, n_levels=int(sc.get("score_levels", 8)),
                        seed=int(sc.get("score_seed", 0)), max_images=int(sc.get("max_images", 256)))
    K = int(sc.get("n_queries", 1))
    if K > 1:
        return _run_batch(sampler, sc, algo, K, shape, ver, device, labels=labels, seed=seed)
    den = S.make_denoise_fn(sampler, labels, max_images=int(sc.get("max_images", 256)), seed=seed)
    dev = str(device)
    if algo == "search_over_paths":
        search = S.SearchOverPaths(n_beams=int(sc.get("n_beams", 4)), n_children=int(sc.get("n_children", 4)),
                                   start_step=int(sc.get("start_step", 800)), delta_f=int(sc.get("delta_f", 50)),
                                   delta_b=int(sc.get("delta_b", 100)))
        images, score, _ = search.search(shape, den, ver.score, device=dev, verbose=False, seed=seed)
        best = S.philox_normal((1,) + shape, search.last_seed, search.last_index, S.TAG_X_T, torch.device(device))[0]
        return best, score, images
    if algo == "fk_steering":
        search = _fk_steering(sc)
        images, score, _ = search.search(shape, den, ver.score, device=dev, seed=seed)
        best = S.philox_normal((1,) + shape, search.last_seed, search.last_index, S.TAG_X_T, torch.device(device))[0]
        return best, score, images
    if algo == "random":
        search = S.RandomSearch(n_candidates=int(sc.get("n_candidates", 4)))
        best, score = search.search(shape, den, ver.score, device=dev, verbose=False, seed=seed)
    else:
        x0 = S.philox_normal((1,) + shape, 0 if seed is None else seed, 0, S.TAG_X_T, torch.device(device))[0]
        if algo == "zero_order":
            search = S.ZeroOrderSearch(n_neighbors=int(sc.get("n_neighbors", 4)),
                                       lambda_radius=float(sc.get("lambda_radius", 0.95)),
                                       n_iterations=int(sc.get("n_iterations", 10)))
            best, score, _ = search.search(x0, den, ver.score, device=dev, verbose=False, seed=seed)
        elif algo == "path":
            search = S.PathSearch(n_paths=int(sc.get("n_paths", 4)), injection_step=int(sc.get("injection_step", 400)),
                                  noise_scale=float(sc.get("noise_scale", 0.1)))
            best, score, _ = search.search(x0, den, ver.score, device=dev, verbose=False, seed=seed)
        else:
            raise ValueError(f"search.algorithm {algo!r}: random | zero_order | path | search_over_paths | "
                             "fk_steering")
    # the images of the winner: its own trajectory (the Philox stream of the candidate id it was scored under),
    # so that the returned images are the ones that produced the returned score
    images = None
    if best is not None:
        images = den.denoise_candidates(best.unsqueeze(0), max(0, int(getattr(search, "last_index", 0))),
                                        seed=getattr(search, "last_seed", seed))[0]
    return best, score, images


def _run_batch(sampler, sc: Dict[str, Any], algo: str, K: int, shape, ver, device, *, labels=None,
               seed: Optional[int] = None):
    """run_search for n_queries = K > 1: one `search_batch` over K queries."""
    from .search import search_algorithm as S
    batched = ("random", "search_over_paths", "fk_steering")
    if algo not in batched:
        raise ValueError(f"search.n_queries={K} needs search.algorithm in {list(batched)}, got {algo!r}")
    den = S.make_denoise_fn(sampler, max_images=int(sc.get("max_images", 256)), seed=seed)
    dev = torch.device(device)
    if algo == "search_over_paths":
        search = S.SearchOverPaths(n_beams=int(sc.get("n_beams", 4)), n_children=int(sc.get("n_children", 4)),
                                   start_step=int(sc.get("start_step", 800)), delta_f=int(sc.get("delta_f", 50)),
                                   delta_b=int(sc.get("delta_b", 100)))
        images, scores, _ = search.search_batch(shape, den, ver.score, K, labels=labels, seed=seed, device=str(dev))
        best = torch.stack([S.philox_normal((1,) + shape, search.last_seed, q * search.n_beams + p, S.TAG_X_T, dev)[0]
                            for q, p in enumerate(search.last_index)])
        return best, scores, images
    if algo == "fk_steering":
        search = _fk_steering(sc)
        images, scores, _ = search.search_batch(shape, den, ver.score, K, labels=labels, seed=seed, device=str(dev))
        best = torch.stack([S.philox_normal((1,) + shape, search.last_seed, q * search.n_particles + p, S.TAG_X_T,
                                            dev)[0] for q, p in enumerate(search.last_index)])
        return best, scores, images
    search = S.RandomSearch(n_candidates=int(sc.get("n_candidates", 4)))
    best, scores = search.search_batch(shape, den, ver.score, K, labels=labels, seed=seed, device=str(dev))
    # each winner's images from its own trajectory (the global candidate id it was scored under)
    images = torch.full_like(best, float("nan"))
    rows = None if labels is None else labels.to(dev, torch.int64).reshape(K, -1).expand(K, shape[0])
    for q, i in enumerate(search.last_index):
        if i >= 0:
            images[q] = den.denoise_candidates(best[q:q + 1], q * search.n_candidates + i, seed=search.last_seed,
                                               cand_labels=None if rows is None else rows[q:q + 1])[0]
    return best, scores, images


def _fk_steering(sc: Dict[str, Any]):
    from .search import search_algorithm as S
    return S.FKSteering(n_particles=int(sc.get("n_particles", 4)), start_step=int(sc.get("start_step", 800)),
                        resample_interval=int(sc.get("resample_interval", 100)), lam=float(sc.get("fk_lambda", 10.0)))


def save_image_grid(images: torch.Tensor, path: str, nrow: int = 8) -> str:
    """[-1, 1] samples -> [0, 1] PNG grid (abstract_metrics_from_pretrained_ddpm.py:621-628)."""
    from torchvision.utils import save_image
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    save_image((images.detach().float().cpu() * 0.5 + 0.5).clamp(0, 1), path, nrow=nrow)
    return path


def main(argv: Optional[List[str]] = None) -> int:
    argv = list(sys.argv[1:] if argv is None else argv)
    path = argv.pop(0) if argv and "=" not in argv[0] else None
    cfg = load_config(path, argv)
    device = torch.device(cfg.get("device", "cuda"))
    if device.type == "cuda" and device.index is None:
        device = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    if device.type == "cuda":
        torch.cuda.set_device(device)       # the library launches on the current device's current stream
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world > 1 and not torch.distributed.is_initialized():
        # one process per GPU: the searches shard their candidates over the ranks (scores all-gathered)
        torch.distributed.init_process_group("nccl" if device.type == "cuda" else "gloo",
                                             **({"device_id": device} if device.type == "cuda" else {}))
    model = create_and_load_model(cfg, device)
    sampler = create_sampler(model, cfg, device)
    sampler.print_steps = False
    labels = None
    K = int((cfg.get("search") or {}).get("n_queries", 1))
    if getattr(model, "is_conditional", False):
        # query q's labels are 1 + (q*B + arange(B)) % num_labels; a single search takes query 0's
        B = int(cfg.get("batch_size", 1))
        labels = (1 + torch.arange(K * B, device=device) % int(cfg["num_labels"])).to(torch.int64)
        labels = labels.view(K, B) if K > 1 else labels
    if cfg.get("search"):
        best, score, images = run_search(sampler, cfg, device, labels=labels, seed=cfg.get("seed"))
        if K > 1:
            print("search: best scores " + " ".join(f"{v:.6f}" for v in score))
            images = images.reshape(-1, *images.shape[2:])       # the grid holds all K*B winning images
        else:
            print(f"search: best score {score:.6f}")
    else:
        B, H = int(cfg.get("batch_size", 1)), int(cfg["img_size"])
        x_T = torch.randn(B, 3, H, H, device=device)
        images, history = sample_with_metrics_tracking(sampler, x_T, metric_interval=int(cfg.get("metric_interval", 5)),
                                                       device=str(device), labels=labels, seed=cfg.get("seed"))
        print(f"sampled {tuple(images.shape)}; {len(history)} metric points (no calculators configured)")
    out_dir = cfg.get("sampled_images_save_dir")
    if out_dir and images is not None:
        name = f"T{cfg['T']}_bs{cfg.get('batch_size', 1)}_size{cfg['img_size']}.png"
        print("saved", save_image_grid(images, os.path.join(out_dir, name), nrow=int(cfg.get("nrow", 8))))
    return 0


if __name__ == "__main__":
    raise SystemExit(main())
