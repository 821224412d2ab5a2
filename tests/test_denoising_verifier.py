"""Denoising verifier (DenoisingVerifier, its_level_inputs, its_denoise_scores): argument checks, levels, driver keys
and the oracle's zero class score on the CPU; the kernels, parity with tests/denoising_verifier_oracle.py, invariance,
graph reuse, the searches and the driver on the GPU."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import ddpm_oracle as O
from tests import cases
from tests import denoising_verifier_oracle as DV
from tests.path_search_oracle import search_over_paths
from tests.test_search_over_paths import SOP_CASES, _randn, _sampler, _sop_inputs
from tests.util import build_shell

# fp32 plan: per-pass forward parity 2.5e-6 relative (DESIGN §5) on eps_hat; a score is a mean of squared
# differences of O(1) values, so it inherits about twice that relative error: 2e-5 of the score's magnitude leaves
# a margin of 4x.
FP32_REL = 2e-5
# 16-bit plan (bf16 / fp16 operands, fp32 accumulation): measured at most 1.1e-4 of the mean squared error on these
# nets, and 8.7e-4 on 64 samples of config A's net (profiles/r05_denoising_verifier_bench.json); bound 2e-3.
BIT16_REL = 2e-3


def _lib_null_calls(L):
    p = ctypes.c_void_p(256)     # never dereferenced: validation returns first
    return [
        (L.its_level_inputs, (None, p, p, p, 2, 3, 16, None), b"null pointer"),
        (L.its_level_inputs, (p, None, p, p, 2, 3, 16, None), b"null pointer"),
        (L.its_level_inputs, (p, p, None, p, 2, 3, 16, None), b"null pointer"),
        (L.its_level_inputs, (p, p, p, None, 2, 3, 16, None), b"null pointer"),
        (L.its_level_inputs, (p, p, p, p, 0, 3, 16, None), b">= 1"),
        (L.its_level_inputs, (p, p, p, p, 2, 0, 16, None), b">= 1"),
        (L.its_level_inputs, (p, p, p, p, 2, 3, 0, None), b"multiple of 4"),
        (L.its_level_inputs, (p, p, p, p, 2, 3, 18, None), b"multiple of 4"),
        (L.its_denoise_scores, (None, p, None, p, 2, 1, 3, 16, None), b"null pointer"),
        (L.its_denoise_scores, (p, None, None, p, 2, 1, 3, 16, None), b"null pointer"),
        (L.its_denoise_scores, (p, p, None, None, 2, 1, 3, 16, None), b"null pointer"),
        (L.its_denoise_scores, (p, p, p, p, 0, 1, 3, 16, None), b">= 1"),
        (L.its_denoise_scores, (p, p, p, p, 2, 0, 3, 16, None), b">= 1"),
        (L.its_denoise_scores, (p, p, p, p, 2, 1, -1, 16, None), b">= 1"),
        (L.its_denoise_scores, (p, p, p, p, 2, 1, 3, 6, None), b"multiple of 4"),
    ]


# ------------------------------------------------------------------------------------------------ CPU --
def test_entry_points_validate_before_any_cuda_call(built_lib):
    for fn, args, msg in _lib_null_calls(built_lib):
        assert fn(*args) == 1, (fn.__name__, args)
        assert msg in built_lib.its_last_error_string(), (fn.__name__, args)


def test_levels_are_stratum_midpoints():
    from its_b200.search.verifier import score_levels
    assert score_levels(1000, 8) == [62, 187, 312, 437, 562, 687, 812, 937]
    assert score_levels(1000, 1) == [500]
    assert score_levels(6, 6) == [0, 1, 2, 3, 4, 5]
    assert score_levels(8, 3) == [1, 4, 6]
    for T, S in [(50, 32), (1000, 32), (7, 2)]:
        assert score_levels(T, S) == DV.levels(T, S)
    for bad in [(8, 0), (8, 9), (8, -1)]:
        with pytest.raises(ValueError):
            score_levels(*bad)


def test_score_tag_collides_with_no_other_stream():
    from its_b200.search import search_algorithm as S
    from its_b200.search import verifier as V
    assert V.TAG_SCORE == DV.TAG_SCORE
    assert V.TAG_SCORE >= 1 << 20          # above every time step a schedule can have
    assert V.TAG_SCORE not in (S.TAG_X_T, S.TAG_PATH, S.TAG_FORWARD) and V.TAG_SCORE < S.TAG_NEIGHBOR


def _cpu_sampler(name):
    cfg = cases.SEARCH_CASES[name]
    net, sd = build_shell(cfg)
    if cfg["kind"] == "uncond":
        from its_b200.Diffusion import GaussianDiffusionSampler
        return GaussianDiffusionSampler(net, cfg["beta_1"], cfg["beta_T"], cfg["T"]), sd
    from its_b200.DiffusionFreeGuidence import GaussianDiffusionSampler
    return GaussianDiffusionSampler(net, cfg["beta_1"], cfg["beta_T"], cfg["T"], w=cfg["w"]), sd


def test_constructor_validates():
    from its_b200.search.verifier import DenoisingVerifier
    u, _ = _cpu_sampler("u_search")
    c, _ = _cpu_sampler("c_search")
    with pytest.raises(ValueError, match="kind"):
        DenoisingVerifier(u, kind="clip")
    with pytest.raises(ValueError, match="guided"):
        DenoisingVerifier(u, kind="class")
    for n in (0, u.T + 1):
        with pytest.raises(ValueError, match="n_levels"):
            DenoisingVerifier(u, n_levels=n)
    v = DenoisingVerifier(c, kind="class", n_levels=c.T)
    assert v.levels == list(range(c.T)) and v.uses_labels and v.graph_captures == 0
    assert DenoisingVerifier(u, n_levels=2).levels == [2, 6]


def test_driver_keys():
    from its_b200 import inference as I
    from its_b200.search import verifier as V
    u, _ = _cpu_sampler("u_search")
    c, _ = _cpu_sampler("c_search")
    v = I.make_verifier("denoising", u, n_levels=4, seed=3, max_images=32)
    assert isinstance(v, V.DenoisingVerifier) and v.kind == "likelihood" and v.seed == 3 and v.max_images == 32
    assert v.levels == V.score_levels(u.T, 4)
    assert I.make_verifier("diffusion_classifier", c, n_levels=3).kind == "class"
    assert I.make_verifier("denoising", c, n_levels=3).kind == "likelihood"
    with pytest.raises(ValueError, match="diffusion_classifier"):
        I.make_verifier("diffusion_classifier", u)
    with pytest.raises(ValueError, match="denoising"):
        I.make_verifier("denoising")
    # run_search builds the verifier before any device work
    conf = dict(img_size=16, batch_size=2, search=dict(verifier="diffusion_classifier"))
    with pytest.raises(ValueError, match="diffusion_classifier"):
        I.run_search(u, conf, "cpu")
    with pytest.raises(ValueError, match="n_levels"):
        I.run_search(u, dict(conf, search=dict(verifier="denoising", score_levels=u.T + 1)), "cpu")
    assert isinstance(I.make_verifier("oracle"), V.OracleVerifier)


def _zero_label_net(sd):
    """The weight of cond_embedding.condEmbedding[3] zeroed: every label maps to the same cond_proj input."""
    sd = dict(sd)
    sd["cond_embedding.condEmbedding.3.weight"] = torch.zeros_like(sd["cond_embedding.condEmbedding.3.weight"])
    return sd


def test_oracle_class_score_is_zero_when_labels_carry_nothing():
    smp, sd = _cpu_sampler("c_search")
    sd = _zero_label_net(sd)
    imgs = _randn(61, (4, 3, 16, 16)).clamp(-1, 1)
    labels = torch.tensor([3, 7, 1, 10])
    with torch.no_grad():
        got = DV.denoise_scores(sd, smp.betas, imgs, 2, 3, 5, "class", labels)
        lik = DV.denoise_scores(sd, smp.betas, imgs, 2, 3, 5, "likelihood", labels)
    assert torch.equal(got, torch.zeros(2)) and bool((lik < 0).all())


# ------------------------------------------------------------------------------------------------ GPU --
def _raw_scores(L, eps_c, eps_u, tab, n_cand, per_cand, S):
    from its_b200 import _lib
    out = torch.empty(n_cand, dtype=torch.float32, device=eps_c.device)
    _lib.check(L.its_denoise_scores(out.data_ptr(), eps_c.data_ptr(), None if eps_u is None else eps_u.data_ptr(),
                                    tab.data_ptr(), n_cand, per_cand, S, tab[0].numel(), _lib.stream_ptr(eps_c.device)))
    return out


def _f64_scores(eps_c, eps_u, tab, n_cand, per_cand, S):
    n_per = tab[0].numel()
    e = tab.reshape(1, S, n_per)
    d_c = (eps_c.reshape(-1, S, n_per) - e).double().pow(2).reshape(n_cand, -1).sum(1)
    if eps_u is None:
        return (-d_c / (per_cand * S * n_per)).float()
    d_u = (eps_u.reshape(-1, S, n_per) - e).double().pow(2).reshape(n_cand, -1).sum(1)
    return ((d_u - d_c) / (per_cand * S * n_per)).float()


@pytest.mark.gpu
def test_level_inputs_bit_equal_to_torch(cuda_dev, built_lib):
    from its_b200 import _lib
    g = torch.Generator().manual_seed(3)
    for n_img, S, shape in [(1, 1, (3, 4, 4)), (5, 3, (3, 16, 16)), (7, 8, (3, 32, 32))]:
        x = (torch.randn((n_img,) + shape, generator=g) * 2).to(cuda_dev)
        eps = torch.randn((S,) + shape, generator=g).to(cuda_dev)
        abar = torch.rand(S, generator=g, dtype=torch.float64)
        coef = torch.stack([abar.sqrt(), (1 - abar).sqrt()], 1).float().to(cuda_dev).contiguous()
        out = torch.empty((n_img * S,) + shape, device=cuda_dev)
        _lib.check(built_lib.its_level_inputs(out.data_ptr(), x.data_ptr(), eps.data_ptr(), coef.data_ptr(), n_img, S,
                                              x[0].numel(), _lib.stream_ptr(cuda_dev)))
        want = coef[:, 0].view(1, S, 1, 1, 1) * x.unsqueeze(1) + coef[:, 1].view(1, S, 1, 1, 1) * eps.unsqueeze(0)
        assert torch.equal(out, want.reshape(out.shape)), (n_img, S)


@pytest.mark.gpu
@pytest.mark.parametrize("per_cand", [1, 2])
@pytest.mark.parametrize("kind", ["likelihood", "class"])
def test_denoise_scores_match_a_float64_reduction(cuda_dev, built_lib, per_cand, kind):
    g = torch.Generator().manual_seed(4)
    S, n_cand, shape = 3, 5, (3, 16, 16)
    rows = n_cand * per_cand * S
    tab = torch.randn((S,) + shape, generator=g).to(cuda_dev)
    eps_c = (tab.repeat(n_cand * per_cand, 1, 1, 1) + 0.3 * torch.randn((rows,) + shape, generator=g).to(cuda_dev))
    eps_u = (tab.repeat(n_cand * per_cand, 1, 1, 1) + 0.4 * torch.randn((rows,) + shape, generator=g).to(cuda_dev)) \
        if kind == "class" else None
    got = _raw_scores(built_lib, eps_c, eps_u, tab, n_cand, per_cand, S)
    want = _f64_scores(eps_c, eps_u, tab, n_cand, per_cand, S)
    assert torch.allclose(got, want, rtol=1e-6, atol=0), (got, want)
    # a NaN in one image makes its candidate's score NaN and leaves the others alone
    bad = eps_c.clone()
    bad[per_cand * S + 1, 0, 2, 3] = float("nan")
    got_nan = _raw_scores(built_lib, bad, eps_u, tab, n_cand, per_cand, S)
    assert torch.isnan(got_nan[1]) and not torch.isnan(got_nan[torch.arange(n_cand) != 1]).any()
    assert torch.equal(got_nan[torch.arange(n_cand) != 1], got[torch.arange(n_cand) != 1])


def _gpu_net(name, dev, precision, zero_labels=False):
    cfg = cases.SEARCH_CASES[name]
    net, sd = build_shell(cfg)
    if zero_labels:
        sd = _zero_label_net(sd)
        net.load_state_dict(sd)
    net = net.to(dev)
    net.precision = precision
    return cfg, net, sd, _sampler(cfg, net, dev)


def _images(n, seed=71):
    return _randn(seed, (n, 3, 16, 16)).clamp(-1, 1)


def _labels(n, cfg, seed=72):
    if cfg["kind"] != "cond":
        return None
    return torch.from_numpy(np.random.default_rng(seed).integers(1, cfg["num_labels"] + 1, n)).long()


def _device_eps(ver, dev):
    return ver._tables_for(dev, 3 * 16 * 16)[0].view(-1, 3, 16, 16).cpu()


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "16bit"])
@pytest.mark.parametrize("name,kind", [("u_search", "likelihood"), ("c_search", "likelihood"), ("c_search", "class")])
def test_scores_match_the_oracle(cuda_dev, name, kind, precision):
    from its_b200.search.verifier import DenoisingVerifier
    cfg, net, sd, smp = _gpu_net(name, cuda_dev, precision)
    S, B, n_cand = 4, 2, 3
    imgs, labels = _images(n_cand * B), _labels(n_cand * B, cfg)
    ver = DenoisingVerifier(smp, kind, n_levels=S, seed=9)
    got = ver.score_candidates(imgs.to(cuda_dev), B, None if labels is None else labels.to(cuda_dev)).cpu()
    eps = _device_eps(ver, cuda_dev)
    ph = torch.from_numpy(DV.philox.normal(9, 0, DV.TAG_SCORE, S, 3 * 16 * 16)).view_as(eps)
    assert (eps - ph).abs().max() <= 1e-5            # the same draws as oracle.philox, up to fast-math bits
    with torch.no_grad():
        ref = DV.denoise_scores(sd, smp.betas.cpu(), imgs, B, S, 9, kind, labels, eps=eps)
        # errors relative to the mean squared error itself: a class score is a difference of two of them
        scale = DV.denoise_scores(sd, smp.betas.cpu(), imgs, B, S, 9, "likelihood", labels, eps=eps).abs() \
            if kind == "class" else ref.abs()
    err = float(((got - ref).abs() / scale).max())
    print(f"{name} {kind} {precision}: scores {got.tolist()} oracle {ref.tolist()} max rel err {err:.3e}")
    assert err <= (FP32_REL if precision == "fp32" else BIT16_REL)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "16bit"])
def test_class_score_is_exactly_zero_when_labels_carry_nothing(cuda_dev, precision):
    """Both halves of the plan see the same cond_proj; an image's arithmetic does not depend on its batch position
    (DESIGN §3.1), so D_u == D_c bit for bit."""
    from its_b200.search.verifier import DenoisingVerifier
    cfg, net, sd, smp = _gpu_net("c_search", cuda_dev, precision, zero_labels=True)
    imgs, labels = _images(6), _labels(6, cfg)
    ver = DenoisingVerifier(smp, "class", n_levels=3, seed=2)
    got = ver.score_candidates(imgs.to(cuda_dev), 2, labels.to(cuda_dev))
    assert torch.equal(got, torch.zeros_like(got))


@pytest.mark.gpu
@pytest.mark.parametrize("name,kind", [("u_search", "likelihood"), ("c_search", "class")])
def test_scores_do_not_depend_on_chunking_position_or_population(cuda_dev, name, kind):
    from its_b200.search.verifier import DenoisingVerifier
    cfg, net, _, smp = _gpu_net(name, cuda_dev, "16bit")
    S, B, n_cand = 3, 2, 5
    imgs = _images(n_cand * B).to(cuda_dev)
    labels = _labels(n_cand * B, cfg)
    labels = None if labels is None else labels.to(cuda_dev)
    halves = 2 if kind == "class" else 1
    whole = DenoisingVerifier(smp, kind, n_levels=S, seed=5).score_candidates(imgs, B, labels)
    assert torch.isfinite(whole).all() and whole.unique().numel() == n_cand
    for max_images in (halves * B * S, 2 * halves * B * S, 1):
        ver = DenoisingVerifier(smp, kind, n_levels=S, seed=5, max_images=max_images)
        assert torch.equal(ver.score_candidates(imgs, B, labels), whole), max_images
    # reversed population, and every candidate alone
    rev = torch.arange(n_cand - 1, -1, -1, device=cuda_dev)
    r_imgs = imgs.view(n_cand, B, 3, 16, 16)[rev].reshape_as(imgs)
    r_lab = None if labels is None else labels.view(n_cand, B)[rev].reshape(-1)
    ver = DenoisingVerifier(smp, kind, n_levels=S, seed=5)
    assert torch.equal(ver.score_candidates(r_imgs, B, r_lab), whole[rev])
    for c in range(n_cand):
        one = ver.score(imgs[c * B:(c + 1) * B], None if labels is None else labels[c * B:(c + 1) * B])
        assert one == float(whole[c]), c
    # the seed
    again = DenoisingVerifier(smp, kind, n_levels=S, seed=5).score_candidates(imgs, B, labels)
    other = DenoisingVerifier(smp, kind, n_levels=S, seed=6).score_candidates(imgs, B, labels)
    assert torch.equal(again, whole) and not torch.equal(other, whole)


@pytest.mark.gpu
def test_scoring_graph_is_captured_once_per_plan(cuda_dev):
    from its_b200.search.verifier import DenoisingVerifier
    cfg, net, _, smp = _gpu_net("c_search", cuda_dev, "16bit")
    imgs, labels = _images(8).to(cuda_dev), _labels(8, cfg).to(cuda_dev)
    ver = DenoisingVerifier(smp, "class", n_levels=2, seed=1, max_images=3 * 2 * 2 * 2)   # 3 candidates per pass
    a = ver.score_candidates(imgs, 2, labels)            # chunks of 3 and 1 candidates: two plans
    assert ver.graph_captures == 2
    b = ver.score_candidates(imgs, 2, labels)
    assert ver.graph_captures == 2 and torch.equal(a, b)
    # the likelihood plan of 16 UNet images is UNet.forward's plan for a batch of 16: a forward call in between
    # leaves the scores alone (t_idx and labels are restated for every chunk)
    lik = DenoisingVerifier(smp, "likelihood", n_levels=2, seed=1)
    c = lik.score_candidates(imgs, 2, labels)
    net(torch.zeros(16, 3, 16, 16, device=cuda_dev), torch.full((16,), 5, dtype=torch.long, device=cuda_dev),
        torch.zeros(16, dtype=torch.long, device=cuda_dev))
    assert torch.equal(lik.score_candidates(imgs, 2, labels), c) and lik.graph_captures == 1
    net.invalidate_plans()                               # rebuilt plans: the stale graphs are dropped
    assert torch.equal(ver.score_candidates(imgs, 2, labels), a) and ver.graph_captures == 4
    assert len(ver._graphs) == 2


def _den(smp, **kw):
    from its_b200.search import search_algorithm as S
    return S.make_denoise_fn(smp, **kw)


@pytest.mark.gpu
def test_random_searches_report_the_scores_of_their_images(cuda_dev):
    """Guided net, class kind: the single search (shared labels) and the batched one (per-query labels) return
    scores equal to re-scoring the winners' images with their labels."""
    from its_b200.search import search_algorithm as S
    from its_b200.search.verifier import DenoisingVerifier
    cfg, net, _, smp = _gpu_net("c_search", cuda_dev, "16bit")
    shape = tuple(cfg["noise_shape"])
    B = shape[0]
    ver = DenoisingVerifier(smp, "class", n_levels=3, seed=4)
    lab = torch.tensor([2, 9], device=cuda_dev)
    den = _den(smp, labels=lab, seed=7)
    rs = S.RandomSearch(n_candidates=4)
    best, score = rs.search(shape, den, ver.score, device=str(cuda_dev), seed=13)
    img = den.denoise_candidates(best.unsqueeze(0), rs.last_index, seed=13)[0]
    assert score == ver.score(img, lab)
    K = 3
    q_lab = torch.tensor([[1, 2], [5, 5], [10, 3]], device=cuda_dev)
    den = _den(smp, seed=7)
    rb = S.RandomSearch(n_candidates=4)
    bests, scores = rb.search_batch(shape, den, ver.score, K, labels=q_lab, seed=13, device=str(cuda_dev))
    assert rb.last_scores.unique().numel() == K * 4
    for q in range(K):
        img = den.denoise_candidates(bests[q:q + 1], q * 4 + rb.last_index[q], seed=13, cand_labels=q_lab[q:q + 1])[0]
        assert scores[q] == ver.score(img, q_lab[q]), q
    # callable mode (labels through **kwargs) scores the same candidates the same way
    cands = S.philox_normal((4,) + shape, 13, 0, S.TAG_X_T, cuda_dev)
    den = _den(smp, seed=7)
    best_c, score_c = S.RandomSearch(n_candidates=4).search(shape, den, lambda x, **k: ver.score(x, **k),
                                                            device=str(cuda_dev), candidate_noise=cands, labels=lab)
    assert score_c == score and torch.equal(best_c, best)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["u_sop", "c_sop"])
def test_search_over_paths_vs_oracle(cuda_dev, name):
    """fp32 plan, injected noise: the search with the denoising verifier against the oracle's search with the
    restated verifier; the returned score equals re-scoring the returned image."""
    from its_b200.search import search_algorithm as S
    from its_b200.search.verifier import DenoisingVerifier
    from tests.test_search_over_paths import _compare_with_oracle
    cfg = SOP_CASES[name]
    net, sd = build_shell(cfg, cuda_dev)
    net.precision = "fp32"
    smp = _sampler(cfg, net, cuda_dev)
    x_T, fwd, step_noise, labels = _sop_inputs(cfg)
    kind = "class" if cfg["kind"] == "cond" else "likelihood"
    S_lv = 3
    ver = DenoisingVerifier(smp, kind, n_levels=S_lv, seed=8)
    den = S.make_denoise_fn(smp, None if labels is None else labels.to(cuda_dev), step_noise=step_noise.to(cuda_dev))
    sop = S.SearchOverPaths(n_beams=cfg["n_beams"], n_children=cfg["n_children"], start_step=cfg["start_step"],
                            delta_f=cfg["delta_f"], delta_b=cfg["delta_b"])
    extra = {} if labels is None else {"labels": labels.to(cuda_dev)}
    img, score, h = sop.search(tuple(cfg["noise_shape"]), den, ver.score, device=str(cuda_dev), seed=3,
                               candidate_noise=x_T.to(cuda_dev), forward_noise=fwd.to(cuda_dev), **extra)
    assert score == ver.score(img, None if labels is None else labels.to(cuda_dev))
    eps = _device_eps(ver, cuda_dev)
    sched = O.schedule(cfg["beta_1"], cfg["beta_T"], cfg["T"])
    betas = smp.betas.cpu()

    def vfn(images):
        return float(DV.denoise_scores(sd, betas, images, images.shape[0], S_lv, 8, kind, labels, eps=eps)[0])

    with torch.no_grad():
        ref_img, ref_score, ref_h = search_over_paths(sd, sched, x_T, lambda t: step_noise[t], fwd, cfg["n_beams"],
                                                      cfg["n_children"], cfg["start_step"], cfg["delta_f"],
                                                      cfg["delta_b"], vfn, labels, cfg.get("w", 0.0))
    tol = 1e-3 * max(abs(v) for row in ref_h["scores"] for v in row)
    if _compare_with_oracle(h, ref_h, cfg["n_beams"], tol, False):
        last = np.sort(np.array(ref_h["scores"][-1]))[::-1]
        if last[0] - last[1] > 2 * tol:
            assert h["lineage"] == ref_h["lineage"] and abs(score - ref_score) <= tol


@pytest.mark.gpu
@pytest.mark.parametrize("verifier,K", [("denoising", 1), ("diffusion_classifier", 1), ("diffusion_classifier", 3)])
def test_run_search_with_the_denoising_verifiers(cuda_dev, verifier, K):
    from its_b200 import inference as I
    from its_b200.search.verifier import DenoisingVerifier
    name = "c_search" if verifier == "diffusion_classifier" else "u_search"
    cfg, net, _, smp = _gpu_net(name, cuda_dev, "16bit")
    B, H = cfg["noise_shape"][0], cfg["noise_shape"][2]
    sc = dict(algorithm="random", verifier=verifier, n_candidates=4, n_queries=K, score_levels=3, score_seed=2)
    labels = None
    if cfg["kind"] == "cond":
        labels = (1 + torch.arange(K * B, device=cuda_dev) % cfg["num_labels"]).view(K, B) if K > 1 else \
            (1 + torch.arange(B, device=cuda_dev))
    best, score, images = I.run_search(smp, dict(img_size=H, batch_size=B, search=sc), cuda_dev, labels=labels,
                                       seed=5)
    ver = DenoisingVerifier(smp, "class" if verifier == "diffusion_classifier" else "likelihood", n_levels=3, seed=2)
    if K == 1:
        assert score == ver.score(images, labels)
    else:
        for q in range(K):
            assert score[q] == ver.score(images[q], labels[q]), q
