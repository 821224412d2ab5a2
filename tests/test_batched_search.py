"""Batched searches (RandomSearch.search_batch, SearchOverPaths.search_batch) and the segmented top-k kernel they
select with: argument checks and the selection rule on the CPU; the kernel, equivalence with single searches,
stream keying, invariance, unrankable queries, the driver and step-graph reuse on the GPU."""
import ctypes
import math

import numpy as np
import pytest
import torch

from tests import cases
from tests.test_search_over_paths import SOP_CASES, _FakeSampler, _randn, _sampler, _verifier
from tests.util import build_shell


def topk_segmented_rule(scores, n_seg, k):
    """The selection its_topk_first_segmented implements: per segment, the k best by (score descending, index
    ascending); NaN and -inf never rank; flat indices; -1 / -inf past a segment's eligible scores."""
    scores = np.asarray(scores, dtype=np.float32)
    seg = scores.size // n_seg
    idx = np.full((n_seg, k), -1, dtype=np.int32)
    val = np.full((n_seg, k), -np.inf, dtype=np.float32)
    for s in range(n_seg):
        loc = scores[s * seg:(s + 1) * seg]
        ranked = sorted((i for i in range(seg) if loc[i] > -np.inf), key=lambda i: (-loc[i], i))[:k]
        for r, i in enumerate(ranked):
            idx[s, r], val[s, r] = s * seg + i, loc[i]
    return idx.reshape(-1), val.reshape(-1)


# ------------------------------------------------------------------------------------------------ CPU --
def test_segmented_rule_ties_nan_inf_and_short_segments():
    nan, inf = float("nan"), float("inf")
    s = [0.5, nan, 0.7, 0.7,          # tie: first index first, NaN never ranks
         -inf, 2.0, -inf, 1.0,        # -inf never ranks
         nan, nan, nan, nan]          # all NaN: nothing ranks
    idx, val = topk_segmented_rule(s, 3, 3)
    assert idx.tolist() == [2, 3, 0, 5, 7, -1, -1, -1, -1]
    assert val.tolist() == [np.float32(0.7), np.float32(0.7), 0.5, 2.0, 1.0, -inf, -inf, -inf, -inf]
    idx, _ = topk_segmented_rule([3.0, 1.0], 2, 4)         # k > seg_len
    assert idx.tolist() == [0, -1, -1, -1, 1, -1, -1, -1]


def test_segmented_topk_validates_before_any_cuda_call(built_lib):
    L = built_lib
    p = ctypes.c_void_p(256)     # never dereferenced: validation returns first
    for args in [(None, p, p, 2, 4, 1), (p, None, p, 2, 4, 1), (p, p, None, 2, 4, 1)]:
        assert L.its_topk_first_segmented(*args, None) == 1
        assert b"null pointer" in L.its_last_error_string()
    for n_seg, seg_len, k in [(0, 4, 1), (2, 0, 1), (2, 4, 0), (-1, 4, 1)]:
        assert L.its_topk_first_segmented(p, p, p, n_seg, seg_len, k, None) == 1
        assert b">= 1" in L.its_last_error_string()
    assert L.its_topk_first_segmented(p, p, p, 1 << 16, 1 << 15, 1, None) == 1
    assert b"exceeds int32" in L.its_last_error_string()


def _bad_batch_calls():
    """(algorithm, search_batch keyword overrides) that must raise ValueError; noise shape (2, 3, 8, 8)."""
    shape = (2, 3, 8, 8)
    return [
        ("random", dict(n_queries=0)),
        ("random", dict(labels=torch.zeros(3, dtype=torch.int64))),
        ("random", dict(labels=torch.zeros(2, 3, dtype=torch.int64))),
        ("random", dict(candidate_noise=torch.zeros((2, 3) + shape))),
        ("random", dict(candidate_noise=torch.zeros((4,) + shape))),
        ("random", dict(callable_mode=True)),
        ("sop", dict(n_queries=0)),
        ("sop", dict(labels=torch.zeros(2, 1, dtype=torch.int64))),
        ("sop", dict(candidate_noise=torch.zeros((2, 3) + shape))),
        ("sop", dict(forward_noise=torch.zeros((1, 2, 4) + shape))),          # too few rounds
        ("sop", dict(forward_noise=torch.zeros((8, 2, 3) + shape))),          # N*M = 4 children per query
        ("sop", dict(callable_mode=True)),
        ("sop", dict(n_beams=0)),
    ]


@pytest.mark.parametrize("algo,kw", _bad_batch_calls())
def test_search_batch_rejects_bad_arguments(algo, kw):
    """Every check runs before any device work (the fake sampler has no device at all)."""
    from its_b200.search import search_algorithm as S
    from its_b200.search import verifier as V
    kw = dict(kw)
    K = kw.pop("n_queries", 2)
    den, ver = S.SamplerDenoiser(_FakeSampler()), V.OracleVerifier().score
    if kw.pop("callable_mode", False):
        den, ver = (lambda x, **k: x), (lambda x, **k: 0.0)
    if algo == "random":
        search = S.RandomSearch(n_candidates=2)
    else:
        search = S.SearchOverPaths(n_beams=kw.pop("n_beams", 2), n_children=2, start_step=12, delta_f=2, delta_b=4)
    with pytest.raises(ValueError):
        search.search_batch((2, 3, 8, 8), den, ver, K, device="cpu", **kw)


# ------------------------------------------------------------------------------------------------ GPU --
def _topk_raw(L, scores, n_seg, k, segmented=True):
    from its_b200 import _lib
    idx = torch.empty(n_seg * k, dtype=torch.int32, device=scores.device)
    val = torch.empty(n_seg * k, dtype=torch.float32, device=scores.device)
    if segmented:
        rc = L.its_topk_first_segmented(idx.data_ptr(), val.data_ptr(), scores.data_ptr(), n_seg,
                                        scores.numel() // n_seg, k, _lib.stream_ptr(scores.device))
    else:
        rc = L.its_topk_first(idx.data_ptr(), val.data_ptr(), scores.data_ptr(), scores.numel(), k,
                              _lib.stream_ptr(scores.device))
    _lib.check(rc)
    return idx.cpu().numpy(), val.cpu().numpy()


@pytest.mark.gpu
def test_segmented_topk_matches_the_rule_and_per_segment_topk(cuda_dev, built_lib):
    L = built_lib
    rng = np.random.default_rng(17)
    shapes = [(1, 1, 1), (1, 1, 3), (5, 1, 1), (5, 1, 2), (3, 7, 1), (3, 7, 9), (16, 4, 1), (8, 8, 2), (8, 64, 8),
              (4, 200, 16), (2, 1500, 5), (1, 3000, 40)]
    shapes += [(int(rng.integers(1, 40)), int(rng.integers(1, 300)), int(rng.integers(1, 12))) for _ in range(12)]
    for n_seg, seg_len, k in shapes:
        v = np.round(rng.standard_normal(n_seg * seg_len) * 3).astype(np.float32)     # many ties
        v[rng.random(v.size) < 0.1] = np.nan
        v[rng.random(v.size) < 0.05] = -np.inf
        if n_seg > 2:
            v[seg_len:2 * seg_len] = np.nan                                            # one unrankable segment
        s = torch.from_numpy(v).to(cuda_dev)
        want_i, want_v = topk_segmented_rule(v, n_seg, k)
        got_i, got_v = _topk_raw(L, s, n_seg, k)
        assert np.array_equal(got_i, want_i), (n_seg, seg_len, k)
        assert np.array_equal(got_v, want_v), (n_seg, seg_len, k)
        for q in range(n_seg):                        # its_topk_first on each segment, indices shifted by the base
            one_i, one_v = _topk_raw(L, s[q * seg_len:(q + 1) * seg_len].contiguous(), 1, k, segmented=False)
            one_i = np.where(one_i >= 0, one_i + q * seg_len, -1)
            assert np.array_equal(got_i[q * k:(q + 1) * k], one_i) and np.array_equal(got_v[q * k:(q + 1) * k], one_v)
        # its_topk_first over the whole array is the rule with one segment
        all_i, all_v = _topk_raw(L, s, 1, k, segmented=False)
        want_i, want_v = topk_segmented_rule(v, 1, k)
        assert np.array_equal(all_i, want_i) and np.array_equal(all_v, want_v)


def _den(smp, cuda_dev, *, step_noise=None, max_images=256, seed=None):
    from its_b200.search import search_algorithm as S
    return S.make_denoise_fn(smp, max_images=max_images, seed=seed,
                             step_noise=None if step_noise is None else step_noise.to(cuda_dev))


def _sop(cfg, **over):
    from its_b200.search import search_algorithm as S
    kw = dict(n_beams=cfg["n_beams"], n_children=cfg["n_children"], start_step=cfg["start_step"],
              delta_f=cfg["delta_f"], delta_b=cfg["delta_b"])
    kw.update(over)
    return S.SearchOverPaths(**kw)


def _n_rounds(cfg, smp):
    from its_b200.search.search_algorithm import path_rounds
    return len(path_rounds(smp.T, cfg["start_step"], cfg["delta_f"], cfg["delta_b"]))


def _query_labels(cfg, K):
    B = cfg["noise_shape"][0]
    return (1 + (torch.arange(K * B) * 3 + torch.arange(K * B) // B) % cfg["num_labels"]).view(K, B)


@pytest.mark.gpu
def test_unguided_random_batch_is_the_flat_population(cuda_dev):
    """K = 3 queries of N = 4 candidates draw and score exactly RandomSearch(12)'s population; each winner is the
    first-index argmax of its block."""
    from its_b200.search import search_algorithm as S
    cfg = cases.SEARCH_CASES["u_search"]
    net, _ = build_shell(cfg, cuda_dev)
    smp = _sampler(cfg, net, cuda_dev)
    shape, ver = tuple(cfg["noise_shape"]), _verifier(cfg["verifier"])
    flat = S.RandomSearch(n_candidates=12)
    flat.search(shape, _den(smp, cuda_dev), ver.score, device=str(cuda_dev), verbose=False, seed=71)
    rs = S.RandomSearch(n_candidates=4)
    best, scores = rs.search_batch(shape, _den(smp, cuda_dev), ver.score, 3, seed=71, device=str(cuda_dev))
    assert rs.last_scores.shape == (3, 4) and torch.equal(rs.last_scores.flatten(), flat.last_scores)
    assert best.shape == (3,) + shape and rs.last_seed == 71
    for q in range(3):
        i, v = S.argmax_first(flat.last_scores[4 * q:4 * q + 4])
        assert rs.last_index[q] == i and scores[q] == v
        assert torch.equal(best[q], S.philox_normal((1,) + shape, 71, 4 * q + i, S.TAG_X_T, cuda_dev)[0])


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["u_search", "c_search"])
def test_one_query_random_batch_is_search(cuda_dev, name):
    from its_b200.search import search_algorithm as S
    cfg = cases.SEARCH_CASES[name]
    net, _ = build_shell(cfg, cuda_dev)
    smp = _sampler(cfg, net, cuda_dev)
    shape, ver = tuple(cfg["noise_shape"]), _verifier(cfg["verifier"])
    labels = cases.search_labels(cfg)
    kw = {} if labels is None else {"labels": labels.to(cuda_dev)}
    one = S.RandomSearch(n_candidates=cfg["n_candidates"])
    noise, score = one.search(shape, _den(smp, cuda_dev), ver.score, device=str(cuda_dev), verbose=False, seed=5, **kw)
    rs = S.RandomSearch(n_candidates=cfg["n_candidates"])
    best, scores = rs.search_batch(shape, _den(smp, cuda_dev), ver.score, 1, seed=5, device=str(cuda_dev),
                                   labels=None if labels is None else labels.view(1, -1))
    assert torch.equal(best[0], noise) and scores == [score]
    assert torch.equal(rs.last_scores[0], one.last_scores) and rs.last_index == [one.last_index]
    assert rs.nfes == one.nfes


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["u_sop", "c_sop"])
def test_one_query_path_batch_is_search(cuda_dev, name):
    cfg = SOP_CASES[name]
    net, _ = build_shell(cfg, cuda_dev)
    smp = _sampler(cfg, net, cuda_dev)
    shape, ver = tuple(cfg["noise_shape"]), _verifier(cfg["verifier"])
    labels = cases.search_labels(cfg)
    kw = {} if labels is None else {"labels": labels.to(cuda_dev)}
    one = _sop(cfg)
    img, score, h = one.search(shape, _den(smp, cuda_dev), ver.score, device=str(cuda_dev), seed=6, **kw)
    sop = _sop(cfg)
    imgs, scores, hb = sop.search_batch(shape, _den(smp, cuda_dev), ver.score, 1, seed=6, device=str(cuda_dev),
                                        labels=None if labels is None else labels.view(1, -1))
    assert torch.equal(imgs[0], img) and scores == [score]
    assert hb["rounds"] == h["rounds"] and hb["unet_image_steps"] == h["unet_image_steps"]
    for key in ("scores", "survivors", "lineage"):
        assert hb[key] == [h[key]], key
    assert sop.last_index == [one.last_index] and sop.nfes == one.nfes and sop.last_seed == one.last_seed


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["16bit", "fp32"])
@pytest.mark.parametrize("algo", ["random", "sop"])
def test_guided_queries_equal_standalone_searches(cuda_dev, algo, precision):
    """Different labels per query, every draw injected: query q of the batch is the standalone search with query
    q's labels and noise, bit for bit."""
    from its_b200.search import search_algorithm as S
    cfg = SOP_CASES["c_sop"] if algo == "sop" else cases.SEARCH_CASES["c_search"]
    net, _ = build_shell(cfg, cuda_dev)
    net.precision = precision
    smp = _sampler(cfg, net, cuda_dev)
    shape, ver = tuple(cfg["noise_shape"]), _verifier(cfg["verifier"])
    step_noise = cases.search_noise(cfg)
    K = 3
    labels = _query_labels(cfg, K).to(cuda_dev)
    if algo == "random":
        N = cfg["n_candidates"]
        x_T = _randn(811, (K, N) + shape).to(cuda_dev)
        rs = S.RandomSearch(n_candidates=N)
        best, scores = rs.search_batch(shape, _den(smp, cuda_dev, step_noise=step_noise), ver.score, K, labels=labels,
                                       candidate_noise=x_T, seed=9, device=str(cuda_dev))
        for q in range(K):
            one = S.RandomSearch(n_candidates=N)
            noise, score = one.search(shape, _den(smp, cuda_dev, step_noise=step_noise), ver.score,
                                      device=str(cuda_dev), verbose=False, seed=9, candidate_noise=x_T[q],
                                      labels=labels[q])
            assert torch.equal(rs.last_scores[q], one.last_scores), q
            assert rs.last_index[q] == one.last_index and scores[q] == score and torch.equal(best[q], noise), q
        return
    N, NM = cfg["n_beams"], cfg["n_beams"] * cfg["n_children"]
    R = _n_rounds(cfg, smp)
    x_T = _randn(812, (K, N) + shape).to(cuda_dev)
    fwd = _randn(813, (R, K, NM) + shape).to(cuda_dev)
    sop = _sop(cfg)
    imgs, scores, hb = sop.search_batch(shape, _den(smp, cuda_dev, step_noise=step_noise), ver.score, K,
                                        labels=labels, candidate_noise=x_T, forward_noise=fwd, seed=9,
                                        device=str(cuda_dev))
    for q in range(K):
        one = _sop(cfg)
        img, score, h = one.search(shape, _den(smp, cuda_dev, step_noise=step_noise), ver.score,
                                   device=str(cuda_dev), seed=9, candidate_noise=x_T[q], forward_noise=fwd[:, q],
                                   labels=labels[q])
        assert torch.equal(imgs[q], img) and scores[q] == score, q
        for key in ("scores", "survivors", "lineage"):
            assert hb[key][q] == h[key], (q, key)
        assert sop.last_index[q] == one.last_index


@pytest.mark.gpu
@pytest.mark.parametrize("algo", ["random", "sop"])
def test_batch_results_do_not_depend_on_chunking_and_follow_the_seed(cuda_dev, algo):
    """Chunks of one candidate, and chunks of three that straddle the queries, give the unchunked results."""
    from its_b200.search import search_algorithm as S
    cfg = SOP_CASES["u_sop"]
    net, _ = build_shell(cfg, cuda_dev)
    smp = _sampler(cfg, net, cuda_dev)
    shape, ver = tuple(cfg["noise_shape"]), _verifier(cfg["verifier"])
    B = shape[0]

    def run(seed, max_images):
        search = S.RandomSearch(n_candidates=4) if algo == "random" else _sop(cfg)
        out = search.search_batch(shape, _den(smp, cuda_dev, max_images=max_images), ver.score, 3, seed=seed,
                                  device=str(cuda_dev))
        return out, search.last_index

    (a, ia), (b, ib), (c, ic), (d, _) = run(41, B), run(41, 3 * B), run(41, 256), run(42, 256)
    for other, io in ((b, ib), (c, ic)):
        assert torch.equal(a[0], other[0]) and a[1] == other[1] and ia == io
        if algo == "sop":
            assert a[2] == other[2]
    assert not torch.equal(a[0], d[0]) and a[1] != d[1]


def _nan_query_verifier(per_query, q):
    """An OracleVerifier whose scores are NaN for every candidate of query `q` (`per_query` candidates each)."""
    from its_b200.search import verifier as V

    class NaNQuery(V.OracleVerifier):
        def score_candidates(self, images, per_cand):
            s = super().score_candidates(images, per_cand).clone()
            s[q * per_query:(q + 1) * per_query] = float("nan")
            return s
    return NaNQuery()


@pytest.mark.gpu
def test_unrankable_query(cuda_dev):
    """Random search: the query gets -1 / -inf / a NaN row and the others keep their winners.  Search over paths:
    ValueError naming the query and the round."""
    from its_b200.search import search_algorithm as S
    cfg = SOP_CASES["u_sop"]
    net, _ = build_shell(cfg, cuda_dev)
    smp = _sampler(cfg, net, cuda_dev)
    shape, ver = tuple(cfg["noise_shape"]), _verifier(cfg["verifier"])
    rs = S.RandomSearch(n_candidates=4)
    best, scores = rs.search_batch(shape, _den(smp, cuda_dev), ver.score, 3, seed=12, device=str(cuda_dev))
    bad = S.RandomSearch(n_candidates=4)
    b_best, b_scores = bad.search_batch(shape, _den(smp, cuda_dev), _nan_query_verifier(4, 1).score, 3, seed=12,
                                        device=str(cuda_dev))
    assert bad.last_index[1] == -1 and b_scores[1] == -math.inf and torch.isnan(b_best[1]).all()
    for q in (0, 2):
        assert bad.last_index[q] == rs.last_index[q] and b_scores[q] == scores[q] and torch.equal(b_best[q], best[q])
    assert bad.search(shape, _den(smp, cuda_dev), _nan_query_verifier(4, 0).score, device=str(cuda_dev),
                      seed=12) == (None, -math.inf) and bad.last_index == -1
    NM = cfg["n_beams"] * cfg["n_children"]
    with pytest.raises(ValueError, match="query 2, round 0: only 0 of %d children" % NM):
        _sop(cfg).search_batch(shape, _den(smp, cuda_dev), _nan_query_verifier(NM, 2).score, 3, seed=12, device=str(cuda_dev))


@pytest.mark.gpu
@pytest.mark.parametrize("algo", ["random", "search_over_paths"])
def test_run_search_with_several_queries(cuda_dev, algo):
    from its_b200 import inference as I
    from its_b200.search import search_algorithm as S
    cfg = SOP_CASES["u_sop"]
    net, _ = build_shell(cfg, cuda_dev)
    smp = _sampler(cfg, net, cuda_dev)
    B, H = cfg["noise_shape"][0], cfg["noise_shape"][2]
    shape, ver = (B, 3, H, H), _verifier("oracle")
    search = dict(algorithm=algo, verifier="oracle", n_queries=3, n_candidates=4, n_beams=2, n_children=3,
                  start_step=6, delta_f=1, delta_b=3)
    best, scores, images = I.run_search(smp, dict(img_size=H, batch_size=B, search=search), cuda_dev, seed=8)
    assert best.shape == images.shape == (3,) + shape and len(scores) == 3
    if algo == "random":
        rs = S.RandomSearch(n_candidates=4)
        ref_best, ref_scores = rs.search_batch(shape, _den(smp, cuda_dev, seed=8), ver.score, 3, seed=8,
                                               device=str(cuda_dev))
        assert torch.equal(best, ref_best) and scores == ref_scores
        for q, i in enumerate(rs.last_index):          # a re-run of each winner gives its images and its score
            again = _den(smp, cuda_dev, seed=8).denoise_candidates(best[q:q + 1], 4 * q + i)[0]
            assert torch.equal(images[q], again) and ver.score(again) == scores[q]
        with pytest.raises(ValueError, match="n_queries"):
            I.run_search(smp, dict(img_size=H, batch_size=B, search=dict(search, algorithm="zero_order")), cuda_dev)
        return
    sop = _sop(SOP_CASES["u_sop"])
    ref_imgs, ref_scores, _ = sop.search_batch(shape, _den(smp, cuda_dev, seed=8), ver.score, 3, seed=8,
                                               device=str(cuda_dev))
    assert torch.equal(images, ref_imgs) and scores == ref_scores
    for q, p in enumerate(sop.last_index):
        assert ver.score(images[q]) == scores[q]
        assert torch.equal(best[q], S.philox_normal((1,) + shape, 8, 2 * q + p, S.TAG_X_T, cuda_dev)[0])


@pytest.mark.gpu
def test_batched_search_captures_stage_0_and_round_graphs_once(cuda_dev):
    cfg = SOP_CASES["u_sop"]
    net, _ = build_shell(cfg, cuda_dev)
    smp = _sampler(cfg, net, cuda_dev)
    shape, ver = tuple(cfg["noise_shape"]), _verifier(cfg["verifier"])
    _, _, h = _sop(cfg, start_step=4).search_batch(shape, _den(smp, cuda_dev), ver.score, 3, seed=4,
                                                   device=str(cuda_dev))
    assert len(h["rounds"]) > 1 and smp.graph_captures == 2
    _sop(cfg, start_step=4).search_batch(shape, _den(smp, cuda_dev), ver.score, 3, seed=4, device=str(cuda_dev))
    assert smp.graph_captures == 2
