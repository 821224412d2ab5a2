"""Feynman-Kac steering (FKSteering, its_resample_systematic): segment schedule, argument checks, the resampling rule
and the oracle on the CPU; the kernel against the rule, parity with the oracle, equivalences, invariance, errors,
step-graph reuse and the driver on the GPU."""
import ctypes
import math

import numpy as np
import pytest
import torch

from oracle import ddpm_oracle as O
from tests import cases
from tests.fk_steering_oracle import fk_steering, resample, uniform
from tests.test_batched_search import _nan_query_verifier, _query_labels
from tests.test_search_over_paths import _FakeSampler, _randn, _sampler, _verifier
from tests.util import build_shell

SCORE_TOL = 1e-3

# small search cases: the search-parity nets of tests/cases.py with a few resamplings
FK_CASES = {
    "u_fk": dict(cases.SEARCH_CASES["u_search"], n_particles=4, start_step=5, resample_interval=2, lam=200.0,
                 x_T_seed=4201),
    "c_fk": dict(cases.SEARCH_CASES["c_search"], n_particles=3, start_step=3, resample_interval=1, lam=100.0,
                 x_T_seed=4202),
}


def _fk_inputs(cfg):
    shape = tuple(cfg["noise_shape"])
    return _randn(cfg["x_T_seed"], (cfg["n_particles"],) + shape), cases.search_noise(cfg), cases.search_labels(cfg)


def _oracle(cfg, sd, x_T, step_noise, labels, seed, verifier_fn=None, **over):
    kw = dict(N=cfg["n_particles"], start_step=cfg["start_step"], interval=cfg["resample_interval"], lam=cfg["lam"])
    kw.update(over)
    sched = O.schedule(cfg["beta_1"], cfg["beta_T"], cfg["T"])
    with torch.no_grad():
        return fk_steering(sd, sched, x_T, lambda t: step_noise[t], seed=seed,
                           verifier_fn=verifier_fn or O.VERIFIERS[cfg["verifier"]], labels=labels,
                           w=cfg.get("w", 0.0), **kw)


# ------------------------------------------------------------------------------------------------ CPU --
def test_segment_schedule():
    from its_b200.search.search_algorithm import fk_segments
    assert fk_segments(20, 12, 4) == [(19, 12), (11, 8), (7, 4), (3, 0)]
    assert fk_segments(20, 0, 4) == [(19, 0)]
    assert fk_segments(20, 19, 7) == [(19, 19), (18, 12), (11, 5), (4, 0)]
    assert fk_segments(5, 4, 1) == [(4, 4), (3, 3), (2, 2), (1, 1), (0, 0)]
    assert fk_segments(1000, 800, 50)[-1] == (49, 0) and len(fk_segments(1000, 800, 50)) == 17
    for bad in [(20, 20, 4), (20, -1, 4), (20, 12, 0), (20, 12, -3), (0, 0, 1)]:
        with pytest.raises(ValueError):
            fk_segments(*bad)


def _bad_calls():
    """(constructor overrides, search_batch keyword overrides) that must raise ValueError; noise shape (2, 3, 8, 8)."""
    shape = (2, 3, 8, 8)
    return [
        (dict(n_particles=0), {}),
        (dict(lam=-1.0), {}),
        (dict(lam=float("nan")), {}),
        (dict(lam=float("inf")), {}),
        (dict(start_step=20), {}),
        (dict(start_step=-1), {}),
        (dict(resample_interval=0), {}),
        ({}, dict(n_queries=0)),
        ({}, dict(labels=torch.zeros(3, dtype=torch.int64))),
        ({}, dict(labels=torch.zeros(2, 3, dtype=torch.int64))),
        ({}, dict(candidate_noise=torch.zeros((2, 3) + shape))),
        ({}, dict(candidate_noise=torch.zeros((4,) + shape))),
        ({}, dict(callable_mode=True)),
    ]


@pytest.mark.parametrize("ctor,kw", _bad_calls())
def test_search_rejects_bad_arguments(ctor, kw):
    """Every check runs before any device work (the fake sampler has no device at all)."""
    from its_b200.search import search_algorithm as S
    from its_b200.search import verifier as V
    kw = dict(kw)
    K = kw.pop("n_queries", 2)
    den, ver = S.SamplerDenoiser(_FakeSampler()), V.OracleVerifier().score
    if kw.pop("callable_mode", False):
        den, ver = (lambda x, **k: x), (lambda x, **k: 0.0)
    args = dict(n_particles=2, start_step=12, resample_interval=4, lam=10.0)
    args.update(ctor)
    with pytest.raises(ValueError):
        S.FKSteering(**args).search_batch((2, 3, 8, 8), den, ver, K, device="cpu", **kw)
    if K == 2 and not kw:
        with pytest.raises(ValueError):
            S.FKSteering(**args).search((2, 3, 8, 8), den, ver, device="cpu")
    if "candidate_noise" in kw:
        with pytest.raises(ValueError):
            S.FKSteering(**args).search((2, 3, 8, 8), den, ver, device="cpu", candidate_noise=kw["candidate_noise"])


def test_resample_validates_before_any_cuda_call(built_lib):
    L = built_lib
    p = ctypes.c_void_p(256)     # never dereferenced: validation returns first
    for args in [(None, p, p, p), (p, None, p, p), (p, p, None, p), (p, p, p, None)]:
        assert L.its_resample_systematic(*args, None, 1.0, 2, 4, 0, 0, 0, None) == 1
        assert b"null pointer" in L.its_last_error_string()
    for n_seg, seg_len in [(0, 4), (2, 0), (-1, 4), (2, -5)]:
        assert L.its_resample_systematic(p, p, p, p, None, 1.0, n_seg, seg_len, 0, 0, 0, None) == 1
        assert b">= 1" in L.its_last_error_string()
    assert L.its_resample_systematic(p, p, p, p, p, 1.0, 1 << 16, 1 << 15, 0, 0, 0, None) == 1
    assert b"exceeds int32" in L.its_last_error_string()
    for lam in (-0.5, float("nan"), float("inf")):
        assert L.its_resample_systematic(p, p, p, p, None, lam, 2, 4, 0, 0, 0, None) == 1
        assert b"lam" in L.its_last_error_string()


def test_uniform_is_53_bits_of_the_library_philox():
    from oracle import philox
    seen = set()
    for seed, seg, rnd in [(0, 0, 0), (1, 0, 0), (1, 1, 0), (1, 0, 1), (2 ** 40 + 3, 7, 2 ** 33 + 1)]:
        u = uniform(seed, seg, rnd)
        assert 0.0 <= u < 1.0 and u not in seen
        seen.add(u)
        c = philox.philox4x32_10(np.array([seg, rnd & 0xFFFFFFFF, 0x40000002, rnd >> 32], dtype=np.uint32),
                                 np.array([seed & 0xFFFFFFFF, seed >> 32], dtype=np.uint32))
        assert u * 2.0 ** 53 == (int(c[0]) >> 5) * 2 ** 26 + (int(c[1]) >> 6)


def test_resampling_rule():
    nan, inf = float("nan"), float("inf")
    rng = np.random.default_rng(3)
    r = rng.standard_normal(12).astype(np.float32)
    anc, out, ess, _ = resample(r, None, 0.0, 3, 5, 0)          # lam = 0: equal weights, identity
    assert anc.tolist() == list(range(12)) and np.array_equal(out, r) and np.allclose(ess, 4.0)
    anc, out, _, _ = resample(r, r, 7.0, 3, 5, 1)                # reward = carried: identity again
    assert anc.tolist() == list(range(12))
    dom = np.zeros(8, dtype=np.float32)
    dom[5] = 10.0                                                # one dominant weight (exp(-100) next to 1)
    anc, out, ess, _ = resample(dom, None, 10.0, 2, 9, 0)
    assert anc[:4].tolist() == [0, 1, 2, 3]                      # equal weights in the first segment
    assert anc[4:].tolist() == [5] * 4 and out[4:].tolist() == [10.0] * 4 and abs(ess[1] - 1.0) < 1e-12
    bad = np.array([nan, 0.3, inf, -inf, 0.1, nan, 0.2, -inf, nan, nan, nan, nan], dtype=np.float32)
    for seed in range(20):
        anc, out, ess, _ = resample(bad, None, 3.0, 3, seed, 0)
        assert set(anc[:4].tolist()) == {1} and set(anc[4:8].tolist()) <= {4, 6}
        assert anc[8:].tolist() == [-1] * 4 and np.isnan(out[8:]).all() and ess[2] == 0.0
    # a non-finite carried reward or log-potential weighs 0 as well
    anc, _, _, _ = resample(np.array([1, 2, 3, 4], dtype=np.float32), np.array([0, nan, 0, 0], dtype=np.float32),
                            1.0, 1, 4, 2)
    assert 1 not in anc.tolist()


@pytest.mark.parametrize("name", ["u_fk", "c_fk"])
def test_oracle_single_particle_is_the_plain_sampler(name):
    """N = 1: every resampling keeps the one particle, so the search is the ancestral loop cut into segments and
    returns O.sample's image exactly."""
    cfg = FK_CASES[name]
    _, sd = build_shell(cfg)
    x_T, step_noise, labels = _fk_inputs(cfg)
    img, score, h = _oracle(cfg, sd, x_T[:1], step_noise, labels, seed=3, N=1)
    sched = O.schedule(cfg["beta_1"], cfg["beta_T"], cfg["T"])
    with torch.no_grad():
        ref = O.sample(sd, sched, x_T[0], lambda t: step_noise[t], labels, cfg.get("w", 0.0))
    assert torch.equal(img, ref)
    assert score == float(np.float32(O.VERIFIERS[cfg["verifier"]](ref)))
    assert h["ancestors"] == [[0]] * (len(h["segments"]) - 1) and h["lineage"] == [0] * len(h["segments"])


# ------------------------------------------------------------------------------------------------ GPU --
def _resample_raw(L, reward, carried, lam, n_seg, seed, rnd):
    from its_b200 import _lib
    n = reward.numel()
    anc = torch.empty(n, dtype=torch.int32, device=reward.device)
    out = torch.empty(n, dtype=torch.float32, device=reward.device)
    ess = torch.empty(n_seg, dtype=torch.float32, device=reward.device)
    _lib.check(L.its_resample_systematic(anc.data_ptr(), out.data_ptr(), ess.data_ptr(), reward.data_ptr(),
                                         None if carried is None else carried.data_ptr(), lam, n_seg, n // n_seg,
                                         seed, rnd, 0x40000002, _lib.stream_ptr(reward.device)))
    return anc.cpu().numpy(), out.cpu().numpy(), ess.cpu().numpy()


@pytest.mark.gpu
def test_resample_kernel_matches_the_rule(cuda_dev, built_lib):
    L = built_lib
    rng = np.random.default_rng(29)
    shapes = [(1, 1, 1.0), (4, 1, 3.0), (1, 3, 10.0), (5, 3, 0.0), (3, 64, 2.0), (2, 64, 40.0), (1, 1000, 5.0),
              (3, 1000, 0.5), (1, 5000, 3.0), (2, 5000, 20.0), (7, 37, 1e3), (4, 300, 0.0)]
    for k, (n_seg, seg_len, lam) in enumerate(shapes):
        n = n_seg * seg_len
        r = np.round(rng.standard_normal(n) * 4) / 4                  # many ties
        r = r.astype(np.float32)
        r[rng.random(n) < 0.05] = np.nan
        r[rng.random(n) < 0.03] = np.inf
        r[rng.random(n) < 0.03] = -np.inf
        if n_seg > 2:
            r[seg_len:2 * seg_len] = np.nan                            # one segment with nothing to weigh
        c = None if k % 2 else (rng.standard_normal(n) * 0.5).astype(np.float32)
        seed, rnd = int(rng.integers(0, 2 ** 62)), int(rng.integers(0, 2 ** 40))
        want_a, want_c, want_e, margin = resample(r, c, lam, n_seg, seed, rnd)
        assert margin > 1e-9, (n_seg, seg_len, lam)                    # exact equality is a fair demand
        rt = torch.from_numpy(r).to(cuda_dev)
        ct = None if c is None else torch.from_numpy(c).to(cuda_dev)
        got_a, got_c, got_e = _resample_raw(L, rt, ct, lam, n_seg, seed, rnd)
        assert np.array_equal(got_a, want_a), (n_seg, seg_len, lam)
        assert np.array_equal(got_c, want_c, equal_nan=True), (n_seg, seg_len, lam)
        assert np.all(np.abs(got_e - want_e) <= 1e-6 * np.abs(want_e)), (n_seg, seg_len, lam)
        again = _resample_raw(L, rt, ct, lam, n_seg, seed, rnd)
        assert all(np.array_equal(x, y, equal_nan=True) for x, y in zip(again, (got_a, got_c, got_e)))


def _den(smp, dev, *, labels=None, step_noise=None, max_images=256, seed=None):
    from its_b200.search import search_algorithm as S
    return S.make_denoise_fn(smp, None if labels is None else labels.to(dev), max_images=max_images, seed=seed,
                             step_noise=None if step_noise is None else step_noise.to(dev))


def _fk(cfg, **over):
    from its_b200.search import search_algorithm as S
    kw = dict(n_particles=cfg["n_particles"], start_step=cfg["start_step"], resample_interval=cfg["resample_interval"],
              lam=cfg["lam"])
    kw.update(over)
    return S.FKSteering(**kw)


def _compare_with_oracle(h, ref_h, lam, tol, strict):
    """True when every resampling drew the oracle's ancestors.  A different draw is accepted (non-strict) only where
    the oracle's positions lie within what a score error of `tol` can move them; later rounds then differ."""
    assert h["segments"] == ref_h["segments"]
    for r, (got, ref) in enumerate(zip(h["scores"], ref_h["scores"])):
        got, ref = np.array(got), np.array(ref)
        print("round %d: scores %s vs oracle %s, ancestors %s vs %s, oracle margin %.3g" %
              (r, got, ref, h["ancestors"][r], ref_h["ancestors"][r], ref_h["margin"][r]))
        assert np.abs(got - ref).max() <= tol, r
        if h["ancestors"][r] == ref_h["ancestors"][r]:
            assert abs(h["ess"][r] - ref_h["ess"][r]) <= 1e-3 * ref_h["ess"][r] + 4 * lam * tol * len(got), r
            continue
        assert not strict, r
        assert ref_h["margin"][r] <= 4 * lam * tol, r
        return False
    return True


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["16bit", "fp32"])
@pytest.mark.parametrize("name", ["u_fk", "c_fk"])
def test_fk_steering_vs_oracle(cuda_dev, name, precision):
    cfg = FK_CASES[name]
    net, sd = build_shell(cfg, cuda_dev)
    net.precision = precision
    smp = _sampler(cfg, net, cuda_dev)
    x_T, step_noise, labels = _fk_inputs(cfg)
    fk = _fk(cfg)
    extra = {} if labels is None else {"labels": labels.to(cuda_dev)}
    img, score, h = fk.search(tuple(cfg["noise_shape"]), _den(smp, cuda_dev, labels=labels, step_noise=step_noise),
                              _verifier(cfg["verifier"]).score, device=str(cuda_dev), seed=3,
                              candidate_noise=x_T.to(cuda_dev), **extra)
    ref_img, ref_score, ref_h = _oracle(cfg, sd, x_T, step_noise, labels, seed=3)
    assert any(a != list(range(cfg["n_particles"])) for a in ref_h["ancestors"])     # the case does resample
    strict = precision == "fp32"
    tol = 1e-4 if strict else SCORE_TOL
    if _compare_with_oracle(h, ref_h, cfg["lam"], tol, strict):
        last = np.sort(np.array(ref_h["final_scores"]))[::-1]
        if strict or last[0] - last[1] > 2 * tol:
            assert h["lineage"] == ref_h["lineage"] and fk.last_index == ref_h["lineage"][0]
            assert abs(score - ref_score) <= tol
            assert (img.cpu() - ref_img).abs().max().item() <= (1e-3 if strict else 5e-2)
    assert fk.nfes == cfg["n_particles"] * cfg["T"]
    assert h["unet_image_steps"] == fk.nfes * cfg["noise_shape"][0] * (2 if cfg["kind"] == "cond" else 1)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["u_fk", "c_fk"])
def test_no_resampling_is_random_search(cuda_dev, name):
    """start_step = 0: one segment from x_T to step 0 on RandomSearch's streams, the same winners, scores and
    images bit for bit."""
    from its_b200.search import search_algorithm as S
    cfg = FK_CASES[name]
    net, _ = build_shell(cfg, cuda_dev)
    smp = _sampler(cfg, net, cuda_dev)
    shape, ver = tuple(cfg["noise_shape"]), _verifier(cfg["verifier"])
    K, N = 3, cfg["n_particles"]
    labels = _query_labels(cfg, K).to(cuda_dev) if cfg["kind"] == "cond" else None
    fk = _fk(cfg, start_step=0)
    imgs, scores, h = fk.search_batch(shape, _den(smp, cuda_dev), ver.score, K, labels=labels, seed=21,
                                      device=str(cuda_dev))
    assert h["segments"] == [(cfg["T"] - 1, 0)] and h["ancestors"] == [[]] * K
    rs = S.RandomSearch(n_candidates=N)
    best, rs_scores = rs.search_batch(shape, _den(smp, cuda_dev), ver.score, K, labels=labels, seed=21,
                                      device=str(cuda_dev))
    assert fk.last_index == rs.last_index and scores == rs_scores and fk.nfes == K * N * cfg["T"]
    for q, i in enumerate(rs.last_index):
        rows = None if labels is None else labels[q:q + 1]
        again = _den(smp, cuda_dev).denoise_candidates(best[q:q + 1], q * N + i, seed=21, cand_labels=rows)[0]
        assert torch.equal(imgs[q], again), q


@pytest.mark.gpu
def test_zero_lambda_keeps_every_particle(cuda_dev):
    cfg = FK_CASES["u_fk"]
    net, _ = build_shell(cfg, cuda_dev)
    smp = _sampler(cfg, net, cuda_dev)
    _, _, h = _fk(cfg, lam=0.0).search_batch(tuple(cfg["noise_shape"]), _den(smp, cuda_dev),
                                             _verifier(cfg["verifier"]).score, 2, seed=5, device=str(cuda_dev))
    N = cfg["n_particles"]
    assert len(h["ancestors"][0]) == len(h["segments"]) - 1 > 1
    for q in range(2):
        assert h["ancestors"][q] == [list(range(N))] * (len(h["segments"]) - 1)
        assert all(abs(e - N) < 1e-5 for e in h["ess"][q])


@pytest.mark.gpu
def test_copies_of_one_particle_diverge(cuda_dev):
    """A verifier under which particle 2 dominates: every child descends from it, yet the finished images differ,
    because each copy continues on its own step-noise stream."""
    from its_b200.search import verifier as V
    cfg = FK_CASES["u_fk"]
    net, _ = build_shell(cfg, cuda_dev)
    smp = _sampler(cfg, net, cuda_dev)
    N = cfg["n_particles"]

    class OneWins(V.OracleVerifier):
        def __init__(self):
            super().__init__()
            self.seen = []

        def score_candidates(self, images, per_cand):
            self.seen.append(images.clone())
            s = super().score_candidates(images, per_cand).clone()
            if len(self.seen) == 1:
                s[2] = s[2] + 10.0          # lam * 10 = 2000: the other weights underflow to 0
            return s

    ver = OneWins()
    fk = _fk(cfg)
    _, _, h = fk.search(tuple(cfg["noise_shape"]), _den(smp, cuda_dev), ver.score, device=str(cuda_dev), seed=8)
    assert h["ancestors"][0] == [2] * N and h["ess"][0] == 1.0
    assert h["lineage"][0] == 2 and fk.last_index == 2
    assert len(ver.seen) == len(h["segments"])
    final = ver.seen[-1].view(N, -1)                # the finished samples of all N particles
    assert all(not torch.equal(final[a], final[b]) for a in range(N) for b in range(a + 1, N))


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["16bit", "fp32"])
def test_batched_queries_are_independent_searches(cuda_dev, precision):
    """Different labels per query, x_T and step noise injected.  Query 0 of the batch is the single search with its
    labels and x_T, bit for bit (a query's resampling uniform is keyed by its index in the batch, as a single
    search's is by 0); query 1 does not change when the other queries get other labels and x_T; and nothing depends
    on max_images."""
    cfg = FK_CASES["c_fk"]
    net, _ = build_shell(cfg, cuda_dev)
    net.precision = precision
    smp = _sampler(cfg, net, cuda_dev)
    shape, ver = tuple(cfg["noise_shape"]), _verifier(cfg["verifier"])
    step_noise = cases.search_noise(cfg)
    K, N, B = 3, cfg["n_particles"], shape[0]
    labels = _query_labels(cfg, K).to(cuda_dev)
    x_T = _randn(911, (K, N) + shape).to(cuda_dev)

    def batch(lab, x, max_images=256):
        fk = _fk(cfg)
        out = fk.search_batch(shape, _den(smp, cuda_dev, step_noise=step_noise, max_images=max_images), ver.score, K,
                              labels=lab, candidate_noise=x, seed=9, device=str(cuda_dev))
        return out, fk.last_index

    (imgs, scores, hb), last = batch(labels, x_T)
    assert any(a != list(range(N)) for q in range(K) for a in hb["ancestors"][q])
    one = _fk(cfg)
    img, score, h = one.search(shape, _den(smp, cuda_dev, step_noise=step_noise), ver.score, device=str(cuda_dev),
                               seed=9, candidate_noise=x_T[0], labels=labels[0])
    assert torch.equal(imgs[0], img) and scores[0] == score and last[0] == one.last_index
    for key in ("scores", "ancestors", "ess", "lineage"):
        assert hb[key][0] == h[key], key
    other_labels = labels.clone()
    other_labels[0], other_labels[2] = labels[2], labels[0]
    other_x = x_T.clone()
    other_x[0], other_x[2] = _randn(912, (2, N) + shape).to(cuda_dev)
    (o_imgs, o_scores, o_h), o_last = batch(other_labels, other_x)
    assert torch.equal(o_imgs[1], imgs[1]) and o_scores[1] == scores[1] and o_last[1] == last[1]
    for key in ("scores", "ancestors", "ess", "lineage"):
        assert o_h[key][1] == hb[key][1], key
    for max_images in (B, 2 * B):
        (c_imgs, c_scores, c_h), c_last = batch(labels, x_T, max_images)
        assert torch.equal(c_imgs, imgs) and c_scores == scores and c_h == hb and c_last == last


@pytest.mark.gpu
def test_results_follow_the_seed_and_not_the_chunking(cuda_dev):
    cfg = FK_CASES["u_fk"]
    net, _ = build_shell(cfg, cuda_dev)
    smp = _sampler(cfg, net, cuda_dev)
    shape, ver = tuple(cfg["noise_shape"]), _verifier(cfg["verifier"])
    B = shape[0]

    def run(seed, max_images):
        fk = _fk(cfg)
        out = fk.search_batch(shape, _den(smp, cuda_dev, max_images=max_images), ver.score, 3, seed=seed,
                              device=str(cuda_dev))
        return out, fk.last_index, fk.last_seed

    (a, ia, sa), (b, ib, _), (c, _, _) = run(41, B), run(41, 3 * B), run(42, 256)
    assert torch.equal(a[0], b[0]) and a[1] == b[1] and a[2] == b[2] and ia == ib and sa == 41
    assert not torch.equal(a[0], c[0]) and a[1] != c[1]


@pytest.mark.gpu
def test_unweighable_query_raises(cuda_dev):
    cfg = FK_CASES["u_fk"]
    net, _ = build_shell(cfg, cuda_dev)
    smp = _sampler(cfg, net, cuda_dev)
    N = cfg["n_particles"]
    with pytest.raises(ValueError, match="query 1, resampling round 0: none of the %d particles" % N):
        _fk(cfg).search_batch(tuple(cfg["noise_shape"]), _den(smp, cuda_dev), _nan_query_verifier(N, 1).score, 3,
                              seed=12, device=str(cuda_dev))


@pytest.mark.gpu
def test_second_search_captures_no_step_graph(cuda_dev):
    cfg = FK_CASES["u_fk"]
    net, _ = build_shell(cfg, cuda_dev)
    smp = _sampler(cfg, net, cuda_dev)
    shape, ver = tuple(cfg["noise_shape"]), _verifier(cfg["verifier"])
    _, _, h = _fk(cfg).search_batch(shape, _den(smp, cuda_dev), ver.score, 3, seed=4, device=str(cuda_dev))
    assert len(h["segments"]) > 2
    captured = smp.graph_captures
    _fk(cfg).search_batch(shape, _den(smp, cuda_dev), ver.score, 3, seed=4, device=str(cuda_dev))
    assert captured >= 1 and smp.graph_captures == captured


@pytest.mark.gpu
@pytest.mark.parametrize("K", [1, 3])
def test_run_search_returns_the_search_images(cuda_dev, K):
    from its_b200 import inference as I
    from its_b200.search import search_algorithm as S
    cfg = FK_CASES["u_fk"]
    net, _ = build_shell(cfg, cuda_dev)
    smp = _sampler(cfg, net, cuda_dev)
    B, H = cfg["noise_shape"][0], cfg["noise_shape"][2]
    shape, ver, N = (B, 3, H, H), _verifier("oracle"), cfg["n_particles"]
    search = dict(algorithm="fk_steering", verifier="oracle", n_queries=K, n_particles=N,
                  start_step=cfg["start_step"], resample_interval=cfg["resample_interval"], fk_lambda=cfg["lam"])
    best, scores, images = I.run_search(smp, dict(img_size=H, batch_size=B, search=search), cuda_dev, seed=8)
    fk = _fk(cfg)
    if K == 1:
        img, score, h = fk.search(shape, _den(smp, cuda_dev, seed=8), ver.score, device=str(cuda_dev), seed=8)
        assert torch.equal(images, img) and scores == score
        assert torch.equal(best, S.philox_normal((1,) + shape, 8, fk.last_index, S.TAG_X_T, cuda_dev)[0])
        return
    ref_imgs, ref_scores, _ = fk.search_batch(shape, _den(smp, cuda_dev, seed=8), ver.score, K, seed=8,
                                              device=str(cuda_dev))
    assert best.shape == images.shape == (K,) + shape
    assert torch.equal(images, ref_imgs) and scores == ref_scores
    for q, p in enumerate(fk.last_index):
        assert ver.score(images[q]) == scores[q]
        assert torch.equal(best[q], S.philox_normal((1,) + shape, 8, q * N + p, S.TAG_X_T, cuda_dev)[0])


@pytest.mark.gpu
def test_denoising_verifier_scores_the_returned_images(cuda_dev):
    from its_b200.search.verifier import DenoisingVerifier
    cfg = FK_CASES["c_fk"]
    net, _ = build_shell(cfg, cuda_dev)
    smp = _sampler(cfg, net, cuda_dev)
    shape = tuple(cfg["noise_shape"])
    ver = DenoisingVerifier(smp, "class", n_levels=3, seed=4)
    K = 3
    labels = _query_labels(cfg, K).to(cuda_dev)
    fk = _fk(cfg)
    imgs, scores, h = fk.search_batch(shape, _den(smp, cuda_dev, seed=7), ver.score, K, labels=labels, seed=13,
                                      device=str(cuda_dev))
    for q in range(K):
        assert scores[q] == ver.score(imgs[q], labels[q]), q
        assert all(math.isfinite(v) for row in h["scores"][q] for v in row)
    lab = torch.tensor([2, 9], device=cuda_dev)
    img, score, _ = _fk(cfg).search(shape, _den(smp, cuda_dev, labels=lab, seed=7), ver.score, device=str(cuda_dev),
                                    seed=13)
    assert score == ver.score(img, lab)
