"""Search over the guidance weight (`guidance=` of the guided sampler's segment / forward and of RandomSearch,
SearchOverPaths and FKSteering; its_ddpm_step_x0_w): argument checks, the driver's refusals and the C-ABI checks on
the CPU; the kernel, the sampler, the searches, the oracle and the driver on the GPU."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import ddpm_oracle as O
from tests import cases
from tests import guidance_search_oracle as GO
from tests.test_fk_steering import FK_CASES, _compare_with_oracle
from tests.test_search_over_paths import SOP_CASES, _randn, _sampler, _verifier
from tests.util import build_shell

RS_CASE = dict(cases.SEARCH_CASES["c_search"], n_candidates=6)
GRID = [0.0, 1.8, 4.0, -0.5, 1.0, 2.5]        # weights of members 0, 1, ... (negative weights are allowed)


def _grid(n, K=None, shift=0):
    """[n] (or [K, n]) weights from GRID, query q shifted by q + shift."""
    rows = [[GRID[(i + q + shift) % len(GRID)] for i in range(n)] for q in range(K or 1)]
    return torch.tensor(rows if K else rows[0], dtype=torch.float64)


def _query_labels(K, B=2):
    return (1 + (torch.arange(K * B) * 3 + torch.arange(K * B) // B) % 10).view(K, B)


class _FakeSampler:
    T = 20
    guided = False


class _FakeGuided:
    T = 20
    guided = True


# ------------------------------------------------------------------------------------------------ CPU --
def _searches():
    from its_b200.search import search_algorithm as S
    return {"random": (lambda: S.RandomSearch(n_candidates=3)),
            "sop": (lambda: S.SearchOverPaths(n_beams=3, n_children=2, start_step=12, delta_f=2, delta_b=4)),
            "fk": (lambda: S.FKSteering(n_particles=3, start_step=12, resample_interval=4))}


@pytest.mark.parametrize("algo", ["random", "sop", "fk"])
@pytest.mark.parametrize("case", ["shape", "batch_shape", "nan", "inf", "unguided", "callable"])
def test_searches_reject_bad_guidance(algo, case):
    """Every check runs before any device work (the fake samplers have no device at all)."""
    from its_b200.search import search_algorithm as S
    from its_b200.search import verifier as V
    shape = (2, 3, 8, 8)
    den, ver = S.SamplerDenoiser(_FakeGuided()), V.OracleVerifier().score
    g, gb = torch.zeros(3), torch.zeros(2, 3)
    if case == "shape":
        g, gb = torch.zeros(4), torch.zeros(3, 3)
    elif case == "batch_shape":
        g, gb = torch.zeros(2, 3), torch.zeros(2, 3, 1)         # search takes [N] only
    elif case in ("nan", "inf"):
        g = torch.tensor([0.0, float(case), 1.0])
        gb = torch.stack([g, g])
    elif case == "unguided":
        den = S.SamplerDenoiser(_FakeSampler())
    else:
        den, ver = (lambda x, **k: x), (lambda x, **k: 0.0)
    name = {"random": "RandomSearch", "sop": "SearchOverPaths", "fk": "FKSteering"}[algo]
    with pytest.raises(ValueError, match=name if case != "callable" or algo == "random" else "population mode"):
        _searches()[algo]().search(shape, den, ver, device="cpu", guidance=g)
    with pytest.raises(ValueError):
        _searches()[algo]().search_batch(shape, den, ver, 2, device="cpu", guidance=gb)


@pytest.mark.parametrize("algo", ["zero_order", "path"])
def test_zero_order_and_path_search_refuse_guidance(algo):
    from its_b200.search import search_algorithm as S
    from its_b200.search import verifier as V
    x = torch.zeros(2, 3, 8, 8)
    search = S.ZeroOrderSearch(n_neighbors=2, n_iterations=1) if algo == "zero_order" else S.PathSearch(n_paths=2)
    for den in (S.SamplerDenoiser(_FakeGuided()), lambda x, **k: x):
        with pytest.raises(ValueError, match="ZeroOrderSearch" if algo == "zero_order" else "PathSearch"):
            search.search(x, den, V.OracleVerifier().score, device="cpu", guidance=torch.zeros(2))


def test_denoiser_and_unguided_sampler_reject_guidance():
    from its_b200.Diffusion import GaussianDiffusionSampler
    from its_b200.search import search_algorithm as S
    with pytest.raises(ValueError, match="guided sampler"):
        S.SamplerDenoiser(_FakeSampler()).denoise_segment(torch.zeros(2, 1, 3, 8, 8), 0, t_start=3, t_stop=0,
                                                          cand_guidance=torch.zeros(2))
    with pytest.raises(ValueError, match=r"\[2\]"):
        S.SamplerDenoiser(_FakeGuided()).denoise_segment(torch.zeros(2, 1, 3, 8, 8), 0, t_start=3, t_stop=0,
                                                         cand_guidance=torch.zeros(3))
    smp = GaussianDiffusionSampler(torch.nn.Identity(), 1e-4, 0.02, 10)
    with pytest.raises(ValueError, match="guided sampler"):
        smp.segment(torch.zeros(1, 3, 8, 8), t_start=3, t_stop=0, seed=1, guidance=[1.0])


def test_guidance_pairs_round_like_the_scalar_path():
    """{w, 1 + w} formed in float64 and rounded once to fp32, as its_ddpm_step_x0 forms float(w), float(1.0 + w)."""
    from its_b200._sampler_base import guidance_pairs
    ws = [0.0, 1.8, -0.5, 1e-8, 3.3, 1 / 3]
    got = guidance_pairs(ws, len(ws), "cpu")
    want = np.array([[np.float32(w), np.float32(1.0 + w)] for w in ws], dtype=np.float32)
    assert got.dtype == torch.float32 and np.array_equal(got.numpy(), want)
    for bad in ([1.0, float("nan")], [float("inf"), 0.0]):
        with pytest.raises(ValueError, match="finite"):
            guidance_pairs(bad, 2, "cpu")
    with pytest.raises(ValueError, match="one weight per image"):
        guidance_pairs([1.0, 2.0, 3.0], 2, "cpu")


def test_config_key_parses():
    from its_b200 import inference as I
    cfg = I.load_config(None, ["search.guidance_weights=[0,1.8,4]", "search.algorithm=random"])
    assert cfg["search"]["guidance_weights"] == [0, 1.8, 4]
    assert I._guidance_weights(cfg["search"], "random", _FakeGuided()) == [0.0, 1.8, 4.0]
    g = I._grid([0.0, 1.8, 4.0], 7)["guidance"]
    assert g.tolist() == [0.0, 1.8, 4.0, 0.0, 1.8, 4.0, 0.0] and g.dtype == torch.float64
    assert I._grid(None, 7) == {}


@pytest.mark.parametrize("algo,gw,sampler,match", [
    ("zero_order", [1.0], _FakeGuided(), "algorithm"),
    ("path", [1.0], _FakeGuided(), "algorithm"),
    ("random", [1.0], _FakeSampler(), "guided net"),
    ("fk_steering", [1.0, 2.0], _FakeSampler(), "guided net"),
    ("random", [], _FakeGuided(), "non-empty"),
    ("random", 1.8, _FakeGuided(), "list"),
    ("random", [1.0, "a"], _FakeGuided(), "list"),
    ("search_over_paths", [1.0, float("nan")], _FakeGuided(), "finite"),
])
def test_driver_refuses_guidance_weights(algo, gw, sampler, match):
    from its_b200 import inference as I
    for K in (1, 2):
        cfg = dict(img_size=8, batch_size=1, search=dict(algorithm=algo, guidance_weights=gw, n_queries=K))
        with pytest.raises(ValueError, match=match):
            I.run_search(sampler, cfg, "cpu")


def test_abi_validates_before_any_cuda_call(built_lib):
    L = built_lib
    p = ctypes.c_void_p(256)     # never dereferenced: validation returns first
    odd = ctypes.c_void_p(260)
    good = [p, p, p, p, None, 0, 1, 4, p, p, p, p, 0, p, p, 1, None]
    # x, eps_c, eps_u, coef, t_dev, w_img, cand_dev, nan_flag are required
    for i in (0, 2, 3, 8, 10, 11, 13, 14):
        args = list(good)
        args[i] = None
        assert L.its_ddpm_step_x0_w(*args) == 1, i
        assert b"null pointer" in L.its_last_error_string()
    args = list(good)
    args[9] = None                                    # x0_out without x0_coef
    assert L.its_ddpm_step_x0_w(*args) == 1 and b"x0_coef" in L.its_last_error_string()
    args = list(good)
    args[11] = odd
    assert L.its_ddpm_step_x0_w(*args) == 1 and b"aligned" in L.its_last_error_string()
    for n_img, n_per in [(0, 4), (1, 0), (1, 6), (-1, 4)]:
        args = list(good)
        args[6], args[7] = n_img, n_per
        assert L.its_ddpm_step_x0_w(*args) == 1 and b"multiple of 4" in L.its_last_error_string()
    args = list(good)
    args[5] = 6
    assert L.its_ddpm_step_x0_w(*args) == 1 and b"noise_t_stride" in L.its_last_error_string()


# ------------------------------------------------------------------------------------------------ GPU --
def _step_inputs(dev, n_img, n_per, T, nan):
    g = torch.Generator().manual_seed(17)
    x = (torch.randn(n_img, n_per, generator=g) * 2).to(dev)
    e_c = torch.randn(n_img, n_per, generator=g).to(dev)
    e_u = torch.randn(n_img, n_per, generator=g).to(dev)
    noise = torch.randn(T, n_img, n_per, generator=g).to(dev)
    if nan:
        e_u[1, 5] = float("nan")
    return x, e_c, e_u, noise


@pytest.mark.gpu
@pytest.mark.parametrize("injected", [False, True])
@pytest.mark.parametrize("clip", [0, 1])
@pytest.mark.parametrize("nan", [False, True])
def test_kernel_matches_scalar_launches_and_torch(cuda_dev, built_lib, injected, clip, nan):
    """Every pair equal to w: its_ddpm_step_x0's state, x0 and NaN flag bit for bit.  Distinct pairs: each image
    equals a scalar launch at its own w.  With injected noise both equal the fp32 torch restatement."""
    from its_b200 import _lib
    from its_b200._sampler_base import guidance_pairs
    from its_b200.Diffusion import GaussianDiffusionSampler
    dev, L = cuda_dev, built_lib
    T, n_img, n_per, seed, cand = 12, 5, 3 * 8 * 8, 77, 1234
    smp = GaussianDiffusionSampler(torch.nn.Identity(), 1e-4, 0.02, T).to(dev)
    coef, x0tab = smp._coef_table(dev), smp._x0_table(dev)
    x, e_c, e_u, noise = _step_inputs(dev, n_img, n_per, T, nan)
    cand_dev = torch.tensor([cand], dtype=torch.int64, device=dev)
    s = _lib.stream_ptr(dev)
    stride = n_img * n_per if injected else 0
    nz = noise.data_ptr() if injected else None
    ws = [0.0, 1.8, -0.5, 4.0, 1 / 3]

    def scalar(xs, w, t_dev):
        out, x0, f = xs.clone(), torch.empty_like(xs), torch.zeros(1, dtype=torch.int32, device=dev)
        _lib.check(L.its_ddpm_step_x0(out.data_ptr(), x0.data_ptr(), e_c.data_ptr(), e_u.data_ptr(), nz, stride,
                                      n_img, n_per, coef.data_ptr(), x0tab.data_ptr(), t_dev.data_ptr(), w, seed,
                                      cand_dev.data_ptr(), f.data_ptr(), clip, s))
        return out, x0, int(f.item())

    def per_image(xs, weights, t_dev):
        pairs = guidance_pairs(weights, n_img, dev)
        out, x0, f = xs.clone(), torch.empty_like(xs), torch.zeros(1, dtype=torch.int32, device=dev)
        _lib.check(L.its_ddpm_step_x0_w(out.data_ptr(), x0.data_ptr(), e_c.data_ptr(), e_u.data_ptr(), nz, stride,
                                        n_img, n_per, coef.data_ptr(), x0tab.data_ptr(), t_dev.data_ptr(),
                                        pairs.data_ptr(), seed, cand_dev.data_ptr(), f.data_ptr(), clip, s))
        return out, x0, int(f.item())

    for t in (T - 1, 5, 0):
        t_dev = torch.tensor([t], dtype=torch.int32, device=dev)
        for w in (1.8, -0.5):
            a, b = scalar(x, w, t_dev), per_image(x, [w] * n_img, t_dev)
            assert torch.equal(a[0].nan_to_num(), b[0].nan_to_num()) and torch.equal(a[0].isnan(), b[0].isnan()), t
            assert torch.equal(a[1].nan_to_num(), b[1].nan_to_num()) and a[2] == b[2] == int(nan), t
        got, got_x0, flag = per_image(x, ws, t_dev)
        assert flag == int(nan)
        for i, w in enumerate(ws):
            ref, ref_x0, _ = scalar(x, w, t_dev)
            assert torch.equal(got[i].nan_to_num(), ref[i].nan_to_num()), (t, i)
            assert torch.equal(got_x0[i].nan_to_num(), ref_x0[i].nan_to_num()), (t, i)
        # the fp32 torch restatement: separately rounded mul / mul / sub for the mix
        pairs = guidance_pairs(ws, n_img, dev)
        eps = pairs[:, 1:] * e_c - pairs[:, :1] * e_u
        want_x0 = torch.clip(x0tab[t, 0] * x - x0tab[t, 1] * eps, -1, 1)
        assert torch.equal(got_x0.nan_to_num(), want_x0.nan_to_num()), t
        if injected:
            c1, c2, sig = coef[t, 0], coef[t, 1], (coef[t, 2] if t > 0 else torch.zeros((), device=dev))
            want = (c1 * x - c2 * eps) + sig * noise[t] if t > 0 else c1 * x - c2 * eps
            if t == 0 and clip:
                want = torch.clamp(want, -1, 1)
            ok = torch.isfinite(want)              # the final clip sends NaN to -1, torch.clamp keeps it
            assert torch.equal(got[ok], want[ok]) and (t == 0 and clip or torch.equal(ok, torch.isfinite(got))), t


def _guided(cfg, dev, precision="16bit"):
    net, sd = build_shell(cfg, dev)
    net.precision = precision
    return _sampler(cfg, net, dev), sd


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["16bit", "fp32"])
def test_segment_with_guidance_equals_scalar_runs(cuda_dev, precision):
    """segment(guidance=g) over B images equals, image by image, scalar-w runs; new weights replay the same graph
    and the scalar path's graph stays as it was."""
    cfg = RS_CASE
    smp, _ = _guided(cfg, cuda_dev, precision)
    B = 4
    x = _randn(5, (B, 3, 16, 16)).to(cuda_dev)
    lab = torch.tensor([1, 4, 7, 2], device=cuda_dev)
    kw = dict(t_start=cfg["T"] - 1, t_stop=2, seed=9, cand_id0=40, x0=True)
    w0 = smp.w
    ref0 = smp.segment(x, lab, **kw)
    scalar_captures = smp.graph_captures
    assert smp.segment(x, lab, **kw)[0].equal(ref0[0]) and smp.graph_captures == scalar_captures
    for weights in ([0.0, 1.8, 4.0, -0.5], [2.5, 2.5, 0.0, 1.0]):
        got, got_x0 = smp.segment(x, lab, **kw, guidance=torch.tensor(weights, dtype=torch.float64))
        for i, w in enumerate(weights):
            smp.w = w
            ref, ref_x0 = smp.segment(x, lab, **kw)
            assert torch.equal(got[i], ref[i]) and torch.equal(got_x0[i], ref_x0[i]), (weights, i)
        smp.w = w0
    # one capture for the per-image path, whatever the weights; the scalar path recaptures only on a new w
    captures = smp.graph_captures
    smp.segment(x, lab, **kw, guidance=[3.0, -1.0, 0.5, 1.8])
    assert smp.graph_captures == captures
    every = smp.segment(x, lab, **kw, guidance=[w0] * B)
    assert torch.equal(every[0], ref0[0]) and torch.equal(every[1], ref0[1])
    # forward() of the guided sampler takes the same keyword
    full = smp(x, lab, seed=9, guidance=[0.0, 1.8, 4.0, -0.5])
    smp.w = 4.0
    assert torch.equal(full[2], smp(x, lab, seed=9)[2])
    smp.w = w0


def _den(smp, dev, *, step_noise=None, max_images=256, seed=None):
    from its_b200.search import search_algorithm as S
    return S.make_denoise_fn(smp, max_images=max_images, seed=seed,
                             step_noise=None if step_noise is None else step_noise.to(dev))


def _sop(cfg, **over):
    from its_b200.search import search_algorithm as S
    kw = dict(n_beams=cfg["n_beams"], n_children=cfg["n_children"], start_step=cfg["start_step"],
              delta_f=cfg["delta_f"], delta_b=cfg["delta_b"])
    kw.update(over)
    return S.SearchOverPaths(**kw)


def _fk(cfg, **over):
    from its_b200.search import search_algorithm as S
    kw = dict(n_particles=cfg["n_particles"], start_step=cfg["start_step"], resample_interval=cfg["resample_interval"],
              lam=cfg["lam"])
    kw.update(over)
    return S.FKSteering(**kw)


def _make(algo):
    from its_b200.search import search_algorithm as S
    if algo == "random":
        return RS_CASE, (lambda cfg: S.RandomSearch(n_candidates=cfg["n_candidates"])), "n_candidates"
    if algo == "sop":
        return SOP_CASES["c_sop"], _sop, "n_beams"
    return FK_CASES["c_fk"], _fk, "n_particles"


def _run(algo, smp, dev, K, *, guidance=None, labels=None, seed=31, max_images=256):
    cfg, ctor, key = _make(algo)
    search = ctor(cfg)
    shape = tuple(cfg["noise_shape"])
    out = search.search_batch(shape, _den(smp, dev, max_images=max_images), _verifier(cfg["verifier"]).score, K,
                              labels=labels, seed=seed, device=str(dev), guidance=guidance)
    return out, search


@pytest.mark.gpu
@pytest.mark.parametrize("algo", ["random", "sop", "fk"])
def test_equal_weights_reproduce_the_plain_search(cuda_dev, algo):
    cfg, _, key = _make(algo)
    smp, _ = _guided(cfg, cuda_dev)
    K, N = 2, cfg[key]
    labels = _query_labels(K).to(cuda_dev)
    plain, ps = _run(algo, smp, cuda_dev, K, labels=labels)
    captures = smp.graph_captures
    same, gs = _run(algo, smp, cuda_dev, K, labels=labels,
                    guidance=torch.full((N,), smp.w, dtype=torch.float64))
    assert torch.equal(plain[0], same[0]) and plain[1] == same[1] and ps.last_index == gs.last_index
    assert gs.last_guidance == [smp.w] * K and getattr(ps, "last_guidance", None) is None
    if algo != "random":
        assert all(all(v == smp.w for v in lg) for lg in same[2].pop("lineage_guidance"))
        assert plain[2] == same[2]
    else:
        assert torch.equal(ps.last_scores, gs.last_scores)
    _run(algo, smp, cuda_dev, K, labels=labels)
    assert smp.graph_captures > captures       # the per-image path has graphs of its own ...
    again = smp.graph_captures
    _run(algo, smp, cuda_dev, K, labels=labels, guidance=_grid(N, K))
    _run(algo, smp, cuda_dev, K, labels=labels)
    assert smp.graph_captures == again         # ... which serve every weight vector; the scalar ones stay


@pytest.mark.gpu
def test_random_search_scores_are_scalar_reruns(cuda_dev):
    """Mixed grid: each candidate's score is that of a scalar-w run of the candidate; the winner's images re-run at
    last_guidance reproduce its score."""
    from its_b200.search import search_algorithm as S
    cfg = RS_CASE
    smp, _ = _guided(cfg, cuda_dev)
    K, N, shape = 2, cfg["n_candidates"], tuple(cfg["noise_shape"])
    labels = _query_labels(K).to(cuda_dev)
    grid = _grid(N, K)
    (best, scores), rs = _run("random", smp, cuda_dev, K, labels=labels, guidance=grid)
    ver, w0 = _verifier(cfg["verifier"]), smp.w
    for q in range(K):
        for i in range(N):
            smp.w = float(grid[q, i])
            x = S.philox_normal((1,) + shape, 31, q * N + i, S.TAG_X_T, cuda_dev)
            img = _den(smp, cuda_dev).denoise_candidates(x, q * N + i, seed=31, cand_labels=labels[q:q + 1])[0]
            assert ver.score(img) == float(rs.last_scores[q, i]), (q, i)
        smp.w = w0
        i = rs.last_index[q]
        assert rs.last_guidance[q] == float(grid[q, i]) and scores[q] == float(rs.last_scores[q].max())
        img = _den(smp, cuda_dev).denoise_candidates(best[q:q + 1], q * N + i, seed=31, cand_labels=labels[q:q + 1],
                                                     cand_guidance=torch.tensor([rs.last_guidance[q]]))[0]
        assert ver.score(img) == scores[q]


@pytest.mark.gpu
@pytest.mark.parametrize("algo", ["random", "sop", "fk"])
def test_results_do_not_depend_on_batch_chunking_or_other_queries(cuda_dev, algo):
    cfg, ctor, key = _make(algo)
    smp, _ = _guided(cfg, cuda_dev)
    K, N, B = 3, cfg[key], cfg["noise_shape"][0]
    labels = _query_labels(K).to(cuda_dev)
    grid = _grid(N, K)
    (out, s) = _run(algo, smp, cuda_dev, K, labels=labels, guidance=grid)
    # another query's weights
    other = grid.clone()
    other[0], other[2] = _grid(N, 2, shift=3)
    o_out, o_s = _run(algo, smp, cuda_dev, K, labels=labels, guidance=other)
    assert torch.equal(o_out[0][1], out[0][1]) and o_out[1][1] == out[1][1]
    assert o_s.last_index[1] == s.last_index[1] and o_s.last_guidance[1] == s.last_guidance[1]
    # chunking
    c_out, c_s = _run(algo, smp, cuda_dev, K, labels=labels, guidance=grid, max_images=B)
    assert torch.equal(c_out[0], out[0]) and c_out[1] == out[1] and c_s.last_guidance == s.last_guidance
    if algo != "random":
        assert c_out[2] == out[2]
    # K = 1: query 0 is the single search
    search = ctor(cfg)
    one = search.search(tuple(cfg["noise_shape"]), _den(smp, cuda_dev), _verifier(cfg["verifier"]).score,
                        device=str(cuda_dev), seed=31, labels=labels[0], guidance=grid[0])
    assert torch.equal(one[0], out[0][0]) and one[1] == out[1][0] and search.last_guidance == s.last_guidance[0]
    if algo != "random":
        assert one[2]["lineage_guidance"] == out[2]["lineage_guidance"][0]
        # a weight follows its lineage: the winner's weight is that of the path / particle it started from
        for q in range(K):
            start = s.last_index[q]
            assert out[2]["lineage_guidance"][q] == [float(grid[q, start])] * len(out[2]["lineage_guidance"][q])
            assert s.last_guidance[q] == float(grid[q, start])


@pytest.mark.gpu
def test_sop_children_inherit_their_parents_weights(cuda_dev):
    """A search over paths whose grid gives paths of one query very different weights: every round's survivors carry
    the weight of the initial path they descend from (checked through the lineage of every query's winner and the
    score of the finished winner re-scored)."""
    cfg = SOP_CASES["c_sop"]
    smp, _ = _guided(cfg, cuda_dev)
    K, N = 2, cfg["n_beams"]
    grid = torch.tensor([[0.0, 6.0], [-0.8, 3.0]], dtype=torch.float64)[:, :N]
    (imgs, scores, h), sop = _run("sop", smp, cuda_dev, K, labels=_query_labels(K).to(cuda_dev), guidance=grid)
    for q in range(K):
        assert h["lineage_guidance"][q] == [float(grid[q, h["lineage"][q]["path"]])] * len(h["rounds"])
        assert _verifier(cfg["verifier"]).score(imgs[q]) == scores[q]


def _oracle_inputs(cfg, N):
    shape = tuple(cfg["noise_shape"])
    return _randn(4301, (N,) + shape), cases.search_noise(cfg), cases.search_labels(cfg)


@pytest.mark.gpu
def test_random_search_vs_oracle_fp32(cuda_dev):
    from its_b200.search import search_algorithm as S
    cfg = RS_CASE
    smp, sd = _guided(cfg, cuda_dev, "fp32")
    N = cfg["n_candidates"]
    x_T, step_noise, labels = _oracle_inputs(cfg, N)
    g = _grid(N)
    rs = S.RandomSearch(n_candidates=N)
    _, score = rs.search(tuple(cfg["noise_shape"]), _den(smp, cuda_dev, step_noise=step_noise),
                         _verifier(cfg["verifier"]).score, device=str(cuda_dev), seed=3,
                         candidate_noise=x_T.to(cuda_dev), labels=labels.to(cuda_dev), guidance=g)
    sched = O.schedule(cfg["beta_1"], cfg["beta_T"], cfg["T"])
    with torch.no_grad():
        ref_i, ref_score, ref_scores = GO.random_search(sd, sched, x_T, lambda t: step_noise[t], g.tolist(),
                                                        O.VERIFIERS[cfg["verifier"]], labels)
    got = rs.last_scores.cpu().numpy()
    assert np.abs(got - np.array(ref_scores)).max() <= 1e-4
    assert len(set(np.round(ref_scores, 6))) == N                 # the weights do change the samples
    assert rs.last_index == ref_i and abs(score - ref_score) <= 1e-4 and rs.last_guidance == g[ref_i].item()


@pytest.mark.gpu
def test_fk_steering_vs_oracle_fp32(cuda_dev):
    cfg = FK_CASES["c_fk"]
    smp, sd = _guided(cfg, cuda_dev, "fp32")
    N = cfg["n_particles"]
    x_T, step_noise, labels = _oracle_inputs(cfg, N)
    g = torch.tensor([0.0, 4.0, -0.5], dtype=torch.float64)[:N]
    fk = _fk(cfg)
    img, score, h = fk.search(tuple(cfg["noise_shape"]), _den(smp, cuda_dev, step_noise=step_noise),
                              _verifier(cfg["verifier"]).score, device=str(cuda_dev), seed=3,
                              candidate_noise=x_T.to(cuda_dev), labels=labels.to(cuda_dev), guidance=g)
    sched = O.schedule(cfg["beta_1"], cfg["beta_T"], cfg["T"])
    with torch.no_grad():
        ref_img, ref_score, ref_h = GO.fk_steering(sd, sched, x_T, lambda t: step_noise[t], g.tolist(),
                                                   cfg["start_step"], cfg["resample_interval"], cfg["lam"], 3,
                                                   O.VERIFIERS[cfg["verifier"]], labels)
    assert _compare_with_oracle(h, ref_h, cfg["lam"], 1e-4, strict=True)
    assert h["lineage"] == ref_h["lineage"] and h["lineage_guidance"] == ref_h["lineage_guidance"]
    assert fk.last_guidance == ref_h["lineage_guidance"][-1]
    assert abs(score - ref_score) <= 1e-4 and (img.cpu() - ref_img).abs().max().item() <= 1e-3


@pytest.mark.gpu
@pytest.mark.parametrize("K", [1, 3])
def test_run_search_with_guidance_weights(cuda_dev, K, capsys):
    from its_b200 import inference as I
    from its_b200.search import search_algorithm as S
    cfg = RS_CASE
    smp, _ = _guided(cfg, cuda_dev)
    B, H = cfg["noise_shape"][0], cfg["noise_shape"][2]
    shape, ver, N = (B, 3, H, H), _verifier(cfg["verifier"]), cfg["n_candidates"]
    gw = [0.0, 1.8, 4.0, -0.5]
    labels = _query_labels(K).to(cuda_dev) if K > 1 else _query_labels(1)[0].to(cuda_dev)
    for algo in ("random", "fk_steering", "search_over_paths"):
        search = dict(algorithm=algo, verifier=cfg["verifier"], n_queries=K, n_candidates=N, n_particles=3,
                      start_step=3, resample_interval=1, fk_lambda=50.0, n_beams=2, n_children=2, delta_f=1,
                      delta_b=2, guidance_weights=gw)
        info = {}
        best, scores, images = I.run_search(smp, dict(img_size=H, batch_size=B, search=search), cuda_dev,
                                            labels=labels, seed=8, info=info)
        chosen = info["guidance"] if K > 1 else [info["guidance"]]
        sc = scores if K > 1 else [scores]
        imgs = images if K > 1 else images.unsqueeze(0)
        assert len(chosen) == K and all(c in gw for c in chosen), algo
        for q in range(K):
            assert ver.score(imgs[q]) == sc[q], (algo, q)      # the images that produced the score
        if algo == "random":
            rs = S.RandomSearch(n_candidates=N)
            grid = torch.tensor([gw[i % len(gw)] for i in range(N)], dtype=torch.float64)
            if K > 1:
                ref_best, ref_scores = rs.search_batch(shape, _den(smp, cuda_dev, seed=8), ver.score, K, labels=labels,
                                                       seed=8, device=str(cuda_dev), guidance=grid)
            else:
                ref_best, ref_scores = rs.search(shape, S.make_denoise_fn(smp, labels, seed=8), ver.score,
                                                 device=str(cuda_dev), seed=8, guidance=grid)
            assert torch.equal(best, ref_best) and scores == ref_scores
            last = rs.last_index if K > 1 else [rs.last_index]
            assert chosen == [gw[i % len(gw)] for i in last]
