"""Rank-ensemble verifier (EnsembleVerifier, its_rank_ensemble): the rule against scipy, argument checks, the searches
that refuse it and the [n, V] score gather on the CPU; the kernel against tests/verifier_ensemble_oracle.py bit for bit,
its invariances, the searches that use it, the driver and graph reuse on the GPU."""
import ctypes
import os

import numpy as np
import pytest
import torch
from scipy.stats import rankdata

from tests import cases
from tests.test_batched_search import _query_labels
from tests.test_denoising_verifier import _cpu_sampler
from tests.test_search_over_paths import SOP_CASES, _FakeSampler, _free_port, _randn, _sampler
from tests.util import build_shell
from tests.verifier_ensemble_oracle import average_ranks, eligible, rank_ensemble

NAN, INF = float("nan"), float("inf")


def _bits(a):
    return np.asarray(a, dtype=np.float32).view(np.int32)


# ------------------------------------------------------------------------------------------------ CPU --
def test_oracle_ranks_are_scipys_average_ranks():
    rng = np.random.default_rng(5)
    for n, V, n_seg in [(12, 1, 1), (40, 3, 4), (64, 8, 2), (7, 2, 7)]:
        s = np.round(rng.standard_normal((n, V)) * 3).astype(np.float32)     # integer values: many ties
        s[rng.random((n, V)) < 0.05] = INF
        w = rng.uniform(0.1, 3.0, V).astype(np.float32)
        out = rank_ensemble(s, w, n_seg)
        L = n // n_seg
        for q in range(n_seg):
            seg = s[q * L:(q + 1) * L]
            for v in range(V):
                assert np.array_equal(average_ranks(seg[:, v]), rankdata(seg[:, v], method="average") - 1)
            if L == 1:
                assert out[q] == 1.0
                continue
            ranks = np.stack([rankdata(seg[:, v], method="average") - 1 for v in range(V)], axis=1)
            want = (ranks @ w.astype(np.float64)) / (w.astype(np.float64).sum() * (L - 1))
            assert np.allclose(out[q * L:(q + 1) * L], want, rtol=1e-6, atol=0)
            assert out[q * L:(q + 1) * L].min() >= 0.0 and out[q * L:(q + 1) * L].max() <= 1.0


def test_oracle_hand_made_cases():
    s = np.array([[1, 5], [1, NAN], [2, 5], [-INF, 0], [INF, 3], [INF, 3],        # segment 0
                  [NAN, 1], [4, 4], [-INF, 2], [0, -INF], [NAN, NAN], [7, NAN],    # segment 1: one eligible
                  [NAN, 1], [1, NAN], [-INF, INF], [0, -INF], [NAN, NAN], [2, -INF]],  # segment 2: none
                 dtype=np.float32)
    out = rank_ensemble(s, [1.0, 3.0], 3)
    # segment 0: eligible rows 0, 2, 4, 5; member 0 ranks 0, 1, 2.5, 2.5 (+inf ties with +inf), member 1 ranks
    # 2.5, 2.5, 0.5, 0.5; the denominator is (1 + 3) * (4 - 1)
    want0 = [(0 + 3 * 2.5) / 12, NAN, (1 + 3 * 2.5) / 12, NAN, (2.5 + 3 * 0.5) / 12, (2.5 + 3 * 0.5) / 12]
    assert np.array_equal(_bits(out[:6]), _bits(want0))
    assert eligible(s[6:12]).tolist() == [False, True, False, False, False, False]
    assert np.array_equal(_bits(out[6:12]), _bits([NAN, 1.0, NAN, NAN, NAN, NAN]))
    assert not eligible(s[12:]).any() and np.array_equal(_bits(out[12:]), _bits([NAN] * 6))
    one = np.array([[NAN], [3.0], [-INF]], dtype=np.float32)
    assert _bits(rank_ensemble(one, [2.0], 1)).tolist() == _bits([NAN, 1.0, NAN]).tolist()


def test_entry_point_validates_before_any_cuda_call(built_lib):
    L = built_lib
    p = ctypes.c_void_p(256)     # never dereferenced: validation returns first
    for args in [(None, p, p), (p, None, p), (p, p, None)]:
        assert L.its_rank_ensemble(*args, 2, 3, 4, None) == 1
        assert b"null pointer" in L.its_last_error_string()
    for V in (0, 9, -1):
        assert L.its_rank_ensemble(p, p, p, V, 3, 4, None) == 1
        assert b"outside [1, 8]" in L.its_last_error_string()
    for n_seg, seg_len in [(0, 4), (2, 0), (-1, 4), (2, -5)]:
        assert L.its_rank_ensemble(p, p, p, 2, n_seg, seg_len, None) == 1
        assert b">= 1" in L.its_last_error_string()
    assert L.its_rank_ensemble(p, p, p, 2, 1 << 16, 1 << 15, None) == 1
    assert b"exceeds int32" in L.its_last_error_string()


def test_ensemble_rejects_bad_members_and_weights():
    from its_b200.search import verifier as V
    a, o = V.AestheticPredictor(), V.OracleVerifier()
    ok = V.EnsembleVerifier([a, o])
    assert ok.weights == [1.0, 1.0] and not ok.uses_labels and ok.ranks_population
    bad = [([], None), ([a] * 9, None), ([a, ok], None), ([a, object()], None),
           ([a, V.OracleVerifier(dataset_stats={"mean": np.zeros(3)})], None),
           ([a, o], [1.0]), ([a, o], [1.0, 2.0, 3.0]), ([a, o], [1.0, 0.0]), ([a, o], [-1.0, 1.0]),
           ([a, o], [NAN, 1.0]), ([a, o], [1.0, INF])]
    for members, weights in bad:
        with pytest.raises(ValueError):
            V.EnsembleVerifier(members, weights)
    assert V.EnsembleVerifier([a] * 8, [0.5] * 8).weights == [0.5] * 8
    u, _ = _cpu_sampler("u_search")
    assert V.EnsembleVerifier([V.DenoisingVerifier(u, n_levels=2), a]).uses_labels
    with pytest.raises(ValueError, match="population"):
        ok.score(torch.zeros(1, 3, 8, 8))
    assert not hasattr(o, "combine") and not hasattr(V.DenoisingVerifier(u, n_levels=2), "combine")


def test_driver_builds_and_rejects_ensembles():
    from its_b200 import inference as I
    from its_b200.search import verifier as V
    u, _ = _cpu_sampler("u_search")
    v = I.make_verifier("ensemble", u, n_levels=3, seed=4, max_images=32, ensemble=["denoising", "aesthetic"],
                        ensemble_weights=[2.0, 0.5])
    assert isinstance(v, V.EnsembleVerifier) and v.weights == [2.0, 0.5]
    assert isinstance(v.members[0], V.DenoisingVerifier) and isinstance(v.members[1], V.AestheticPredictor)
    d = v.members[0]
    assert d.kind == "likelihood" and d.seed == 4 and d.max_images == 32 and d.n_levels == 3
    for ens, w, msg in [(None, None, "non-empty list"), ([], None, "non-empty list"), ("aesthetic", None, "list"),
                        (["aesthetic", "ensemble"], None, "nest"), (["aesthetic", "clip"], None, "clip"),
                        (["diffusion_classifier"], None, "conditional"), (["aesthetic", "oracle"], [1.0], "weights"),
                        (["aesthetic", "oracle"], [1.0, 0.0], "weights"), (["aesthetic", "oracle"], [1.0, -2.0], "weights"),
                        (["aesthetic"], 1.0, "list of floats")]:
        with pytest.raises(ValueError, match=msg):
            I.make_verifier("ensemble", u, ensemble=ens, ensemble_weights=w)
    # run_search builds the verifier before any device work; fk_steering refuses the ensemble before any device work
    conf = dict(img_size=16, batch_size=2, search=dict(verifier="ensemble", ensemble=["aesthetic", "aesthetic"],
                                                       ensemble_weights=[1.0]))
    with pytest.raises(ValueError, match="weights"):
        I.run_search(u, conf, "cpu")
    conf["search"] = dict(algorithm="fk_steering", verifier="ensemble", ensemble=["aesthetic", "oracle"])
    with pytest.raises(ValueError, match="FKSteering cannot use a rank ensemble"):
        I.run_search(u, conf, "cpu")


def test_zero_order_and_fk_steering_refuse_an_ensemble():
    """Both compare scores of different populations; the check runs before any device work (the fake sampler has
    no device at all), in population and callable mode alike."""
    from its_b200.search import search_algorithm as S
    from its_b200.search import verifier as V
    ens = V.EnsembleVerifier([V.AestheticPredictor(), V.OracleVerifier()])
    shape = (2, 3, 8, 8)
    for den in (S.SamplerDenoiser(_FakeSampler()), lambda x, **k: x):
        with pytest.raises(ValueError, match="ZeroOrderSearch cannot use a rank ensemble: it compares"):
            S.ZeroOrderSearch(n_neighbors=2, n_iterations=1).search(torch.zeros(shape), den, ens.score, device="cpu")
        with pytest.raises(ValueError, match="FKSteering cannot use a rank ensemble: it weights"):
            S.FKSteering(n_particles=2, start_step=12, resample_interval=4).search(shape, den, ens.score, device="cpu")
    with pytest.raises(ValueError, match="FKSteering cannot use a rank ensemble"):
        S.FKSteering(n_particles=2, start_step=12, resample_interval=4).search_batch(
            shape, S.SamplerDenoiser(_FakeSampler()), ens.score, 2, device="cpu")


def test_callable_mode_has_no_population_to_rank():
    from its_b200.search import search_algorithm as S
    from its_b200.search import verifier as V
    ens = V.EnsembleVerifier([V.AestheticPredictor()])
    with pytest.raises(ValueError, match="population"):
        S.RandomSearch(n_candidates=2).search((1, 3, 8, 8), lambda x, **k: x, ens.score, device="cpu")


def test_other_verifiers_pass_through_unchanged():
    from its_b200.search import search_algorithm as S
    from its_b200.search import verifier as V
    t = torch.arange(6, dtype=torch.float32)
    for ver in (V.OracleVerifier(), V.AestheticPredictor(), V.SelfSupervisedVerifier()):
        assert S._combine(ver, t, 3) is t
        assert S._no_scores(ver, torch.device("cpu")).shape == (0,)
    ens = V.EnsembleVerifier([V.AestheticPredictor(), V.OracleVerifier(), V.SelfSupervisedVerifier()])
    assert S._no_scores(ens, torch.device("cpu")).shape == (0, 3)


def _gather_worker(rank, world, port, n, out_dir):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from its_b200.search import search_algorithm as S
        from its_b200.search import verifier as V
        ens = V.EnsembleVerifier([V.AestheticPredictor(), V.OracleVerifier(), V.AestheticPredictor()])
        full = torch.arange(n * 3, dtype=torch.float32).view(n, 3) * 0.25 - 2.0
        full[0, 1] = -INF
        lo, hi = S._shard(n, rank, world)
        local = full[lo:hi].clone() if hi > lo else S._no_scores(ens, torch.device("cpu"))
        torch.save({"got": S._gather_scores(local, n), "full": full}, os.path.join(out_dir, f"rank{rank}.pt"))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("n", [9, 4, 1])
def test_member_scores_gather_to_the_flat_matrix(tmp_path, n):
    """gloo, world size 2: the [n_local, V] member blocks (and the empty [0, V] one of a rank without candidates,
    n = 1) gather to the [n, V] matrix on every rank."""
    import torch.multiprocessing as mp
    mp.spawn(_gather_worker, args=(2, _free_port(), n, str(tmp_path)), nprocs=2, join=True)
    for r in range(2):
        res = torch.load(os.path.join(tmp_path, f"rank{r}.pt"))
        assert res["got"].shape == (n, 3) and torch.equal(res["got"], res["full"])


# ------------------------------------------------------------------------------------------------ GPU --
def _kernel(scores, weights, n_seg):
    from its_b200.search.verifier import rank_ensemble as dev_rank_ensemble
    return dev_rank_ensemble(scores, weights, n_seg).cpu().numpy()


def _int_scores(rng, n, V, spread=6):
    s = rng.integers(-spread, spread + 1, (n, V)).astype(np.float32)
    s[rng.random((n, V)) < 0.03] = NAN
    s[rng.random((n, V)) < 0.03] = INF
    s[rng.random((n, V)) < 0.03] = -INF
    return s


@pytest.mark.gpu
def test_kernel_matches_the_oracle_bit_for_bit(cuda_dev):
    rng = np.random.default_rng(17)
    for seg_len in (1, 2, 31, 33, 256, 1000, 5000):
        for V in (1, 2, 3, 8):
            n_seg = {1: 1000, 2: 700, 31: 300, 33: 64, 256: 9, 1000: 3, 5000: 2}[seg_len]
            s = _int_scores(rng, n_seg * seg_len, V, spread=3 if seg_len < 100 else 40)
            if n_seg > 2:
                s[seg_len:2 * seg_len, rng.integers(V)] = NAN            # a segment with nothing eligible
                s[2 * seg_len:3 * seg_len - 1, 0] = -INF                   # a segment with one eligible candidate
            w = rng.uniform(0.05, 4.0, V).astype(np.float32)
            got = _kernel(torch.from_numpy(s).to(cuda_dev), torch.from_numpy(w).to(cuda_dev), n_seg)
            want = rank_ensemble(s, w, n_seg)
            assert np.array_equal(_bits(got), _bits(want)), (seg_len, V)
    # real-valued scores, unit weights
    s = rng.standard_normal((4 * 97, 5)).astype(np.float32)
    w = np.ones(5, dtype=np.float32)
    assert np.array_equal(_bits(_kernel(torch.from_numpy(s).to(cuda_dev), torch.from_numpy(w).to(cuda_dev), 4)),
                          _bits(rank_ensemble(s, w, 4)))


@pytest.mark.gpu
def test_kernel_invariances(cuda_dev):
    rng = np.random.default_rng(23)
    n_seg, seg_len, V = 5, 300, 3
    s = _int_scores(rng, n_seg * seg_len, V, spread=20)
    w = torch.tensor([1.0, 2.5, 0.75], device=cuda_dev)
    base = _kernel(torch.from_numpy(s).to(cuda_dev), w, n_seg)
    for v, f in [(0, lambda x: x * 2), (1, lambda x: x + 7), (2, lambda x: x * 4 - 3)]:   # exact on these integers
        t = s.copy()
        t[:, v] = f(t[:, v])
        assert np.array_equal(_bits(_kernel(torch.from_numpy(t).to(cuda_dev), w, n_seg)), _bits(base)), v
    perm = rng.permutation(seg_len)
    t = s.copy()
    t[seg_len:2 * seg_len] = s[seg_len:2 * seg_len][perm]
    got = _kernel(torch.from_numpy(t).to(cuda_dev), w, n_seg)
    assert np.array_equal(_bits(got[seg_len:2 * seg_len]), _bits(base[seg_len:2 * seg_len][perm]))
    assert np.array_equal(_bits(np.delete(got, np.s_[seg_len:2 * seg_len])),
                          _bits(np.delete(base, np.s_[seg_len:2 * seg_len])))
    t = s.copy()
    t[3 * seg_len:4 * seg_len] = _int_scores(rng, seg_len, V)
    got = _kernel(torch.from_numpy(t).to(cuda_dev), w, n_seg)
    assert not np.array_equal(_bits(got[3 * seg_len:4 * seg_len]), _bits(base[3 * seg_len:4 * seg_len]))
    assert np.array_equal(_bits(np.delete(got, np.s_[3 * seg_len:4 * seg_len])),
                          _bits(np.delete(base, np.s_[3 * seg_len:4 * seg_len])))


class _Recording:
    """Mixin: keep every [n, V] member matrix the ensemble hands to a search."""

    def score_candidates(self, images, per_cand, labels=None):
        m = super().score_candidates(images, per_cand, labels)
        self.seen.append(m.clone())
        return m


def _ensemble(members, weights=None):
    from its_b200.search import verifier as V

    class Recording(_Recording, V.EnsembleVerifier):
        pass
    ens = Recording(members, weights)
    ens.seen = []
    return ens


def _members(smp, names):
    from its_b200.search import verifier as V
    make = {"denoising": lambda: V.DenoisingVerifier(smp, "likelihood", n_levels=3, seed=2, max_images=16),
            "diffusion_classifier": lambda: V.DenoisingVerifier(smp, "class", n_levels=3, seed=2, max_images=16),
            "aesthetic": V.AestheticPredictor, "oracle": V.OracleVerifier}
    return [make[n]() for n in names]


def _member_matrix(members, imgs, B, labels=None):
    """[n, V] scores of the candidates imgs [n, B, C, H, W], each member scoring them on its own."""
    flat = imgs.reshape(-1, *imgs.shape[2:])
    cols = [m.score_candidates(flat, B, labels=labels) if m.uses_labels else m.score_candidates(flat, B)
            for m in members]
    return torch.stack(cols, dim=1).cpu().numpy()


def _first_best(x):
    x = np.asarray(x, dtype=np.float32)
    ok = np.flatnonzero(~np.isnan(x) & (x > -np.inf))
    return int(ok[np.argmax(x[ok])]) if ok.size else -1


RANDOM_CASES = [("u_search", ["denoising", "aesthetic"], [1.0, 1.0]),
                ("c_search", ["diffusion_classifier", "denoising"], [2.0, 0.5])]


@pytest.mark.gpu
@pytest.mark.parametrize("name,names,weights", RANDOM_CASES)
def test_random_search_ranks_the_member_scores(cuda_dev, name, names, weights):
    """last_scores is the rule over the member scores of the same candidates' images, the winner follows, and
    nothing changes with the denoiser's or the members' chunking."""
    from its_b200.search import search_algorithm as S
    cfg = cases.SEARCH_CASES[name]
    net, _ = build_shell(cfg, cuda_dev)
    smp = _sampler(cfg, net, cuda_dev)
    shape, N = tuple(cfg["noise_shape"]), 6
    B = shape[0]
    lab = torch.tensor([2, 9], device=cuda_dev) if cfg["kind"] == "cond" else None
    results = []
    for max_images in (256, B):
        ens = _ensemble(_members(smp, names), weights)
        for m in ens.members:
            if hasattr(m, "max_images"):
                m.max_images = max_images * 3 * (2 if m.kind == "class" else 1)
        den = S.make_denoise_fn(smp, lab, max_images=max_images, seed=7)
        rs = S.RandomSearch(n_candidates=N)
        best, score = rs.search(shape, den, ens.score, device=str(cuda_dev), seed=13)
        results.append((rs.last_scores.cpu().numpy(), rs.last_index, score, best))
    (scores, idx, score, best), again = results
    assert np.array_equal(_bits(again[0]), _bits(scores)) and again[1] == idx and again[2] == score
    assert torch.equal(again[3], best)
    den = S.make_denoise_fn(smp, lab, seed=7)
    cands = S.philox_normal((N,) + shape, 13, 0, S.TAG_X_T, cuda_dev)
    imgs = den.denoise_candidates(cands, 0, seed=13)
    members = _members(smp, names)
    mat = _member_matrix(members, imgs, B, den.image_labels(N))
    want = rank_ensemble(mat, weights, 1)
    assert np.array_equal(_bits(scores), _bits(want))
    assert idx == _first_best(want) and score == float(want[idx]) and torch.equal(best, cands[idx])


@pytest.mark.gpu
@pytest.mark.parametrize("name,names,weights", RANDOM_CASES)
def test_batched_random_queries_equal_standalone_searches(cuda_dev, name, names, weights):
    from its_b200.search import search_algorithm as S
    cfg = cases.SEARCH_CASES[name]
    net, _ = build_shell(cfg, cuda_dev)
    smp = _sampler(cfg, net, cuda_dev)
    shape, N, K = tuple(cfg["noise_shape"]), 5, 3
    step_noise = cases.search_noise(cfg).to(cuda_dev)
    labels = _query_labels(cfg, K).to(cuda_dev) if cfg["kind"] == "cond" else None
    x = _randn(77, (K, N) + shape).to(cuda_dev)
    ens = _ensemble(_members(smp, names), weights)
    rb = S.RandomSearch(n_candidates=N)
    best, scores = rb.search_batch(shape, S.make_denoise_fn(smp, step_noise=step_noise), ens.score, K, labels=labels,
                                   candidate_noise=x, seed=3, device=str(cuda_dev))
    assert len(ens.seen) == 1 and ens.seen[0].shape == (K * N, len(names))
    want = rank_ensemble(ens.seen[0].cpu().numpy(), weights, K).reshape(K, N)
    assert np.array_equal(_bits(rb.last_scores.cpu().numpy()), _bits(want))
    for q in range(K):
        one = S.RandomSearch(n_candidates=N)
        den = S.make_denoise_fn(smp, None if labels is None else labels[q], step_noise=step_noise)
        b, s = one.search(shape, den, ens.score, device=str(cuda_dev), seed=3, candidate_noise=x[q])
        assert np.array_equal(_bits(one.last_scores.cpu().numpy()), _bits(rb.last_scores[q].cpu().numpy())), q
        assert one.last_index == rb.last_index[q] and s == scores[q] and torch.equal(b, best[q]), q


@pytest.mark.gpu
@pytest.mark.parametrize("name,names,K", [("u_sop", ["denoising", "aesthetic"], 1),
                                          ("c_sop", ["diffusion_classifier", "denoising"], 2)])
def test_search_over_paths_ranks_each_rounds_children(cuda_dev, name, names, K):
    from its_b200.search import search_algorithm as S
    cfg = SOP_CASES[name]
    net, _ = build_shell(cfg, cuda_dev)
    smp = _sampler(cfg, net, cuda_dev)
    shape, NM = tuple(cfg["noise_shape"]), cfg["n_beams"] * cfg["n_children"]
    weights = [1.0, 3.0]
    ens = _ensemble(_members(smp, names), weights)
    sop = S.SearchOverPaths(n_beams=cfg["n_beams"], n_children=cfg["n_children"], start_step=cfg["start_step"],
                            delta_f=cfg["delta_f"], delta_b=cfg["delta_b"])
    if K == 1:
        img, score, h = sop.search(shape, S.make_denoise_fn(smp, seed=4), ens.score, device=str(cuda_dev), seed=5)
        per_query = [h["scores"]]
    else:
        labels = _query_labels(cfg, K).to(cuda_dev)
        img, score, h = sop.search_batch(shape, S.make_denoise_fn(smp, seed=4), ens.score, K, labels=labels, seed=5,
                                         device=str(cuda_dev))
        per_query = h["scores"]
    assert len(ens.seen) == len(h["rounds"]) > 1
    for r, mat in enumerate(ens.seen):
        assert mat.shape == (K * NM, len(names))
        want = rank_ensemble(mat.cpu().numpy(), weights, K)
        for q in range(K):
            assert np.array_equal(_bits(per_query[q][r]), _bits(want[q * NM:(q + 1) * NM])), (r, q)
    for q in range(K):
        final = np.asarray(per_query[q][-1], dtype=np.float32)
        best = score if K == 1 else score[q]
        assert best == float(final[_first_best(final)])


@pytest.mark.gpu
@pytest.mark.parametrize("restart", [False, True])
def test_path_search_ranks_one_population(cuda_dev, restart):
    from its_b200.search import search_algorithm as S
    cfg = cases.SEARCH_CASES["u_search"]
    net, _ = build_shell(cfg, cuda_dev)
    smp = _sampler(cfg, net, cuda_dev)
    shape = tuple(cfg["noise_shape"])
    ens = _ensemble(_members(smp, ["denoising", "aesthetic", "oracle"]), [1.0, 0.5, 0.25])
    ps = S.PathSearch(n_paths=7, injection_step=4, noise_scale=0.5)
    x0 = _randn(31, shape).to(cuda_dev)
    best, score, h = ps.search(x0, S.make_denoise_fn(smp, seed=2), ens.score, device=str(cuda_dev), seed=6,
                               restart=restart)
    want = rank_ensemble(ens.seen[0].cpu().numpy(), ens.weights, 1)
    assert len(ens.seen) == 1 and np.array_equal(_bits(h["scores"]), _bits(want))
    assert ps.last_index == _first_best(want) and score == float(want[ps.last_index])


@pytest.mark.gpu
def test_one_member_ensemble_selects_the_members_winner(cuda_dev):
    from its_b200.search import search_algorithm as S
    from its_b200.search import verifier as V
    cfg = cases.SEARCH_CASES["u_search"]
    net, _ = build_shell(cfg, cuda_dev)
    smp = _sampler(cfg, net, cuda_dev)
    shape, K, N = tuple(cfg["noise_shape"]), 4, 6
    alone, ens = S.RandomSearch(n_candidates=N), S.RandomSearch(n_candidates=N)
    b0, _ = alone.search_batch(shape, S.make_denoise_fn(smp, seed=1), V.AestheticPredictor().score, K, seed=9,
                               device=str(cuda_dev))
    b1, s1 = ens.search_batch(shape, S.make_denoise_fn(smp, seed=1), V.EnsembleVerifier([V.AestheticPredictor()]).score,
                              K, seed=9, device=str(cuda_dev))
    member = alone.last_scores.cpu().numpy()
    for q in range(K):
        top = np.sort(member[q])[::-1]
        assert top[0] > top[1], q                                   # a unique winner: the claim is exact
        assert ens.last_index[q] == alone.last_index[q] and s1[q] == 1.0 and torch.equal(b0[q], b1[q]), q


@pytest.mark.gpu
@pytest.mark.parametrize("algo,K", [("random", 1), ("random", 3), ("search_over_paths", 1)])
def test_run_search_with_an_ensemble(cuda_dev, monkeypatch, algo, K):
    """The driver builds the ensemble from search.ensemble; the winner's images (re-run from its trajectory for
    random search, the search's own finished samples for search over paths) reproduce its member scores."""
    from its_b200 import inference as I
    from its_b200.search import verifier as V
    seen = []
    orig = V.EnsembleVerifier.score_candidates

    def record(self, images, per_cand, labels=None):
        m = orig(self, images, per_cand, labels)
        seen.append((self, m.clone(), None if labels is None else labels.clone()))
        return m
    monkeypatch.setattr(V.EnsembleVerifier, "score_candidates", record)
    guided = algo == "random" and K == 3
    cfg = dict(cases.SEARCH_CASES["c_search" if guided else "u_search"])
    if algo == "search_over_paths":
        cfg = SOP_CASES["u_sop"]
    net, _ = build_shell(cfg, cuda_dev)
    smp = _sampler(cfg, net, cuda_dev)
    B, H = cfg["noise_shape"][0], cfg["noise_shape"][2]
    names = ["diffusion_classifier", "denoising"] if guided else ["denoising", "aesthetic"]
    sc = dict(algorithm=algo, verifier="ensemble", ensemble=names, ensemble_weights=[1.5, 1.0], n_candidates=4,
              n_queries=K, score_levels=3, score_seed=2, n_beams=cfg.get("n_beams", 4),
              n_children=cfg.get("n_children", 4), start_step=cfg.get("start_step", 800),
              delta_f=cfg.get("delta_f", 50), delta_b=cfg.get("delta_b", 100))
    labels = (1 + torch.arange(K * B, device=cuda_dev) % cfg["num_labels"]).view(K, B) if guided else None
    best, score, images = I.run_search(smp, dict(img_size=H, batch_size=B, search=sc), cuda_dev, labels=labels,
                                       seed=5)
    ens, mat, _ = seen[-1]
    mat = mat.cpu().numpy()
    n_seg = K
    want = rank_ensemble(mat, ens.weights, n_seg)
    per = want.size // n_seg
    scores = [score] if K == 1 else score
    imgs = images.unsqueeze(0) if K == 1 else images
    for q in range(K):
        i = q * per + _first_best(want[q * per:(q + 1) * per])
        assert scores[q] == float(want[i]), q
        lab = None if labels is None else labels[q]
        again = _member_matrix(ens.members, imgs[q:q + 1], B, lab)[0]
        assert np.array_equal(_bits(again), _bits(mat[i])), q
    for bad in ("zero_order", "fk_steering"):
        with pytest.raises(ValueError, match="cannot use a rank ensemble"):
            I.run_search(smp, dict(img_size=H, batch_size=B, search=dict(sc, algorithm=bad, n_queries=1)), cuda_dev,
                         seed=5)


@pytest.mark.gpu
def test_ensemble_adds_no_graph_captures(cuda_dev):
    """The sampler's step graphs and the denoising member's scoring graphs are those of the member-only search."""
    from its_b200.search import search_algorithm as S
    from its_b200.search import verifier as V
    cfg = cases.SEARCH_CASES["u_search"]
    shape = tuple(cfg["noise_shape"])
    counts = []
    for ensemble in (False, True):
        net, _ = build_shell(cfg, cuda_dev)
        smp = _sampler(cfg, net, cuda_dev)
        d = V.DenoisingVerifier(smp, "likelihood", n_levels=3, seed=2)
        ver = V.EnsembleVerifier([d, V.AestheticPredictor()]) if ensemble else d
        for _ in range(2):
            S.RandomSearch(n_candidates=5).search_batch(shape, S.make_denoise_fn(smp, seed=1), ver.score, 2, seed=9,
                                                        device=str(cuda_dev))
            sop = S.SearchOverPaths(n_beams=2, n_children=2, start_step=5, delta_f=1, delta_b=3)
            sop.search(shape, S.make_denoise_fn(smp, seed=1), ver.score, device=str(cuda_dev), seed=9)
        counts.append((smp.graph_captures, d.graph_captures))
    assert counts[0] == counts[1] and counts[0][0] >= 1 and counts[0][1] >= 1
