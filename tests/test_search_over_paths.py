"""Search over paths (SearchOverPaths): round schedule, oracle, state exchange and C-ABI checks on the CPU;
kernels, segment graph, parity with the oracle, determinism and the driver on the GPU."""
import ctypes
import os
import socket

import numpy as np
import pytest
import torch

from oracle import ddpm_oracle as O
from tests import cases
from tests.path_search_oracle import search_over_paths
from tests.util import build_shell

SCORE_TOL = 1e-3

# small search cases: the search-parity nets of tests/cases.py with a beam schedule of a few rounds
SOP_CASES = {
    "u_sop": dict(cases.SEARCH_CASES["u_search"], n_beams=2, n_children=3, start_step=6, delta_f=1, delta_b=3,
                  forward_seed=4101),
    "c_sop": dict(cases.SEARCH_CASES["c_search"], n_beams=2, n_children=2, start_step=4, delta_f=1, delta_b=2,
                  forward_seed=4102),
}


def _randn(seed, shape):
    return torch.from_numpy(np.random.default_rng(seed).standard_normal(shape).astype(np.float32))


def _sop_inputs(cfg):
    from its_b200.search.search_algorithm import path_rounds
    shape = tuple(cfg["noise_shape"])
    N, M = cfg["n_beams"], cfg["n_children"]
    R = len(path_rounds(cfg["T"], cfg["start_step"], cfg["delta_f"], cfg["delta_b"]))
    x_T = _randn(cfg["forward_seed"] + 1, (N,) + shape)
    fwd = _randn(cfg["forward_seed"], (R, N * M) + shape)
    return x_T, fwd, cases.search_noise(cfg), cases.search_labels(cfg)


# ------------------------------------------------------------------------------------------------ CPU --
def test_round_schedule():
    from its_b200.search.search_algorithm import path_rounds
    assert path_rounds(20, 12, 2, 4) == [(12, 14, 11), (10, 12, 9), (8, 10, 7), (6, 8, 5), (4, 6, 3), (2, 4, 1),
                                         (0, 2, 0)]
    assert path_rounds(20, 19, 5, 10) == [(19, 19, 10), (9, 14, 5), (4, 9, 0)]    # s' capped at T - 1
    assert path_rounds(8, 0, 0, 1) == [(0, 0, 0)]
    assert path_rounds(8, 7, 0, 1) == [(t, t, t) for t in range(7, -1, -1)]
    for bad in [(20, 12, 2, 2), (20, 12, 3, 2), (20, 20, 0, 1), (20, -1, 0, 1), (20, 5, -1, 1)]:
        with pytest.raises(ValueError):
            path_rounds(*bad)


class _FakeSampler:
    T = 20
    guided = False


@pytest.mark.parametrize("kw", [dict(n_beams=0), dict(n_children=0), dict(delta_b=2), dict(delta_f=3, delta_b=3),
                                dict(start_step=20), dict(start_step=-1)])
def test_search_rejects_bad_parameters(kw):
    """Parameters are validated against sampler.T when `search` runs, before any device work."""
    from its_b200.search import search_algorithm as S
    from its_b200.search import verifier as V
    args = dict(n_beams=2, n_children=2, start_step=12, delta_f=2, delta_b=4)
    args.update(kw)
    sop = S.SearchOverPaths(**args)
    with pytest.raises(ValueError):
        sop.search((1, 3, 8, 8), S.SamplerDenoiser(_FakeSampler()), V.OracleVerifier().score, device="cpu")


def test_search_needs_population_mode():
    from its_b200.search import search_algorithm as S
    with pytest.raises(ValueError, match="population mode"):
        S.SearchOverPaths().search((1, 3, 8, 8), lambda x, **k: x, lambda x, **k: 0.0, device="cpu")


@pytest.mark.parametrize("name", ["u_sop", "c_sop"])
def test_oracle_single_path_is_the_plain_sampler(name):
    """N = M = 1, delta_f = 0: every round continues the one path unchanged (a = 1, b = 0), so the search is the
    ancestral loop cut into segments and returns O.sample's image exactly."""
    cfg = SOP_CASES[name]
    _, sd = build_shell(cfg)
    sched = O.schedule(cfg["beta_1"], cfg["beta_T"], cfg["T"])
    _, _, step_noise, labels = _sop_inputs(cfg)
    shape = tuple(cfg["noise_shape"])
    x_T = _randn(7, (1,) + shape)
    fwd = _randn(8, (cfg["T"], 1) + shape)
    w = cfg.get("w", 0.0)
    with torch.no_grad():
        img, score, h = search_over_paths(sd, sched, x_T, lambda t: step_noise[t], fwd, 1, 1, cfg["start_step"], 0,
                                          2, O.VERIFIERS[cfg["verifier"]], labels, w)
        ref = O.sample(sd, sched, x_T[0], lambda t: step_noise[t], labels, w)
    assert torch.equal(img, ref)
    assert score == O.VERIFIERS[cfg["verifier"]](ref)
    assert h["lineage"] == {"path": 0, "children": [0] * len(h["rounds"])}


def _free_port() -> int:
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _gather_worker(rank, world, port, n, out_dir):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from its_b200.search import search_algorithm as S
        full = torch.arange(n * 2 * 3 * 4, dtype=torch.float32).view(n, 2, 3, 4) * 0.5 - 7.0
        lo, hi = S._shard(n, rank, world)
        got = S._gather_states(full[lo:hi].clone(), n)
        torch.save({"got": got, "full": full}, os.path.join(out_dir, f"rank{rank}.pt"))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("n", [9, 4, 1])
def test_state_exchange_returns_the_population_in_global_order(tmp_path, n):
    """gloo, world size 2: ragged shards (and an empty one for n = 1) gather to all n states on every rank."""
    import torch.multiprocessing as mp
    mp.spawn(_gather_worker, args=(2, _free_port(), n, str(tmp_path)), nprocs=2, join=True)
    for r in range(2):
        res = torch.load(os.path.join(tmp_path, f"rank{r}.pt"))
        assert torch.equal(res["got"], res["full"])


def test_new_entry_points_validate_before_any_cuda_call(built_lib):
    L = built_lib
    p = ctypes.c_void_p(256)     # never dereferenced: validation returns first
    rc = L.its_ddpm_step_x0(None, None, None, None, None, 0, 1, 4, None, None, None, 0.0, 0, None, None, 0, None)
    assert rc == 1 and b"null pointer" in L.its_last_error_string()
    rc = L.its_ddpm_step_x0(p, p, p, None, None, 0, 1, 4, p, None, p, 0.0, 0, p, p, 1, None)
    assert rc == 1 and b"x0_coef" in L.its_last_error_string()
    rc = L.its_ddpm_step_x0(p, None, p, None, None, 0, 1, 6, p, None, p, 0.0, 0, p, p, 1, None)
    assert rc == 1 and b"multiple of 4" in L.its_last_error_string()
    rc = L.its_path_expand(None, p, p, 2, 3, 0, 6, 6, 16, 1.0, 0.0, None, 0, 0, 0, None)
    assert rc == 1 and b"null pointer" in L.its_last_error_string()
    rc = L.its_path_expand(p, p, p, 2, 3, 0, 6, 6, 18, 1.0, 0.0, None, 0, 0, 0, None)
    assert rc == 1 and b"multiple of 4" in L.its_last_error_string()
    rc = L.its_path_expand(p, p, p, 2, 3, 4, 3, 6, 16, 1.0, 0.0, None, 0, 0, 0, None)
    assert rc == 1 and b"exceed" in L.its_last_error_string()
    rc = L.its_path_expand(p, p, p, 2, 0, 0, 1, 6, 16, 1.0, 0.0, None, 0, 0, 0, None)
    assert rc == 1


# ------------------------------------------------------------------------------------------------ GPU --
def _sampler(cfg, net, dev):
    if cfg["kind"] == "uncond":
        from its_b200.Diffusion import GaussianDiffusionSampler
        smp = GaussianDiffusionSampler(net, cfg["beta_1"], cfg["beta_T"], cfg["T"])
    else:
        from its_b200.DiffusionFreeGuidence import GaussianDiffusionSampler
        smp = GaussianDiffusionSampler(net, cfg["beta_1"], cfg["beta_T"], cfg["T"], w=cfg["w"])
    smp = smp.to(dev)
    smp.print_steps = False
    return smp


def _verifier(name):
    from its_b200.search import verifier as V
    return {"oracle": V.OracleVerifier(), "aesthetic": V.AestheticPredictor(),
            "self_supervised": V.SelfSupervisedVerifier()}[name]


def _search(cfg, smp, dev, *, step_noise=None, fwd=None, x_T=None, labels=None, seed=3, max_images=256, **over):
    from its_b200.search import search_algorithm as S
    den = S.make_denoise_fn(smp, None if labels is None else labels.to(dev), max_images=max_images,
                            step_noise=None if step_noise is None else step_noise.to(dev))
    kw = dict(n_beams=cfg["n_beams"], n_children=cfg["n_children"], start_step=cfg["start_step"],
              delta_f=cfg["delta_f"], delta_b=cfg["delta_b"])
    kw.update(over)
    sop = S.SearchOverPaths(**kw)
    extra = {}
    if x_T is not None:
        extra["candidate_noise"] = x_T.to(dev)
    if fwd is not None:
        extra["forward_noise"] = fwd.to(dev)
    if labels is not None:
        extra["labels"] = labels.to(dev)
    img, score, h = sop.search(tuple(cfg["noise_shape"]), den, _verifier(cfg["verifier"]).score, device=str(dev),
                               seed=seed, **extra)
    return img, score, h, sop


@pytest.mark.gpu
@pytest.mark.parametrize("guided", [False, True])
@pytest.mark.parametrize("injected", [False, True])
def test_ddpm_step_x0_matches_ddpm_step(cuda_dev, built_lib, guided, injected):
    """The state update is bit-identical to its_ddpm_step (Philox and injected noise, guided and not, the clip of
    step 0); x0 equals the fp32 torch expression of the same formula."""
    from its_b200 import _lib
    from its_b200.Diffusion import GaussianDiffusionSampler
    dev = cuda_dev
    T, n_img, n_per, w, seed, cand = 12, 5, 3 * 8 * 8, 1.8 if guided else 0.0, 77, 1234
    smp = GaussianDiffusionSampler(torch.nn.Identity(), 1e-4, 0.02, T).to(dev)
    coef, x0tab = smp._coef_table(dev), smp._x0_table(dev)
    g = torch.Generator().manual_seed(5)
    x = (torch.randn(n_img, n_per, generator=g) * 2).to(dev)
    e_c = torch.randn(n_img, n_per, generator=g).to(dev)
    e_u = torch.randn(n_img, n_per, generator=g).to(dev) if guided else None
    noise = torch.randn(T, n_img, n_per, generator=g).to(dev) if injected else None
    cand_dev = torch.tensor([cand], dtype=torch.int64, device=dev)
    L = _lib.lib()
    s = _lib.stream_ptr(dev)
    ptr = lambda t: None if t is None else t.data_ptr()
    for t in (T - 1, 5, 0):
        t_dev = torch.tensor([t], dtype=torch.int32, device=dev)
        a, b, x0 = x.clone(), x.clone(), torch.empty_like(x)
        fa, fb = torch.zeros(1, dtype=torch.int32, device=dev), torch.zeros(1, dtype=torch.int32, device=dev)
        _lib.check(L.its_ddpm_step(a.data_ptr(), e_c.data_ptr(), ptr(e_u), ptr(noise), n_img * n_per if injected
                                   else 0, n_img, n_per, coef.data_ptr(), t_dev.data_ptr(), w, seed, cand,
                                   fa.data_ptr(), 1, s))
        _lib.check(L.its_ddpm_step_x0(b.data_ptr(), x0.data_ptr(), e_c.data_ptr(), ptr(e_u), ptr(noise),
                                      n_img * n_per if injected else 0, n_img, n_per, coef.data_ptr(),
                                      x0tab.data_ptr(), t_dev.data_ptr(), w, seed, cand_dev.data_ptr(), fb.data_ptr(),
                                      1, s))
        assert torch.equal(a, b), t
        eps = e_c
        if guided:
            eps = torch.tensor(1.0 + w, dtype=torch.float32, device=dev) * e_c - \
                torch.tensor(w, dtype=torch.float32, device=dev) * e_u
        ref = torch.clip(x0tab[t, 0] * x - x0tab[t, 1] * eps, -1, 1)
        assert torch.equal(x0, ref), t
        if t == 0:
            assert float(b.abs().max()) <= 1.0
        # x0_out = NULL leaves the state update as it is
        c = x.clone()
        _lib.check(L.its_ddpm_step_x0(c.data_ptr(), None, e_c.data_ptr(), ptr(e_u), ptr(noise),
                                      n_img * n_per if injected else 0, n_img, n_per, coef.data_ptr(), None,
                                      t_dev.data_ptr(), w, seed, cand_dev.data_ptr(), fb.data_ptr(), 1, s))
        assert torch.equal(a, c), t


@pytest.mark.gpu
def test_path_expand_matches_torch(cuda_dev, built_lib):
    from its_b200.search import search_algorithm as S
    dev = cuda_dev
    shape = (2, 3, 8, 8)
    g = torch.Generator().manual_seed(9)
    x = torch.randn((6,) + shape, generator=g).to(dev)
    parent = torch.tensor([4, 4, 1], dtype=torch.int32, device=dev)       # repeated parent
    M, a, b = 3, float(np.sqrt(0.93)), float(np.sqrt(0.07))
    af, bf = torch.tensor(a, dtype=torch.float32, device=dev), torch.tensor(b, dtype=torch.float32, device=dev)
    par_of = parent.long()[torch.arange(9, device=dev) // M]
    z = torch.randn((9,) + shape, generator=g).to(dev)
    got = S.path_expand(x, parent, M, 0, 9, a, b, z=z.reshape(9, -1)).view((9,) + shape)
    assert torch.equal(got, af * x[par_of] + bf * z)
    # Philox z: the stream philox_normal gives unit cand_id0 + child0 + i; a shard of children [2, 7)
    lo, hi, cand0, seed = 2, 7, 5 << 40, 42
    got = S.path_expand(x, parent, M, lo, hi - lo, a, b, seed=seed, cand_id0=cand0).view((hi - lo,) + shape)
    zp = S.philox_normal((hi - lo,) + shape, seed, cand0 + lo, S.TAG_FORWARD, dev)
    assert torch.equal(got, af * x[par_of[lo:hi]] + bf * zp)
    # parents straight from the top-k kernel, on the device
    idx, _ = S._topk_device(torch.tensor([0.1, 0.9, 0.3, 0.9, 0.5, 0.2], device=dev), 3)
    got = S.path_expand(x, idx, M, 0, 9, a, b, z=z.reshape(9, -1)).view((9,) + shape)
    assert torch.equal(got, af * x[torch.tensor([1, 3, 4], device=dev)[torch.arange(9, device=dev) // M]] + bf * z)


@pytest.mark.gpu
def test_segment_uncut_equals_the_sampler_and_replays_its_graph(cuda_dev):
    cfg = SOP_CASES["u_sop"]
    net, _ = build_shell(cfg, cuda_dev)
    smp = _sampler(cfg, net, cuda_dev)
    x_T = _randn(3, tuple(cfg["noise_shape"])).to(cuda_dev)
    whole = smp(x_T, seed=19, cand_id0=6)
    for x0 in (False, True):
        seg, p = smp.segment(x_T, t_start=cfg["T"] - 1, t_stop=0, seed=19, cand_id0=6, x0=x0)
        assert torch.equal(seg, whole)
        assert (p is not None) == x0
    # cut in two: the second call replays the captured graph with another step range
    mid, _ = smp.segment(x_T, t_start=cfg["T"] - 1, t_stop=4, seed=19, cand_id0=6, x0=True)
    end, _ = smp.segment(mid, t_start=3, t_stop=0, seed=19, cand_id0=6, x0=True)
    assert torch.equal(end, whole)
    assert smp.graph_captures == 2            # one graph per x0 mode: segment(x0=False) replays forward's


@pytest.mark.gpu
def test_search_captures_stage_0_and_round_graphs_once(cuda_dev):
    """One graph for stage 0 (N paths, steps 7 ... 5) and one for the rounds (N*M children); a second search
    replays both."""
    cfg = SOP_CASES["u_sop"]
    net, _ = build_shell(cfg, cuda_dev)
    smp = _sampler(cfg, net, cuda_dev)
    _, _, h, _ = _search(cfg, smp, cuda_dev, seed=4, start_step=4)
    assert len(h["rounds"]) > 1 and smp.graph_captures == 2
    _search(cfg, smp, cuda_dev, seed=4, start_step=4)
    assert smp.graph_captures == 2


@pytest.mark.gpu
def test_chunks_and_serial_calls_capture_the_step_graph_once(cuda_dev):
    """Chunks of a population and callable-mode candidates differ only in the candidate base: the step graph of
    their batch size is captured once, and the images equal one unchunked call bit for bit."""
    from its_b200.search import search_algorithm as S
    cfg = SOP_CASES["u_sop"]
    net, _ = build_shell(cfg, cuda_dev)
    smp = _sampler(cfg, net, cuda_dev)
    B = cfg["noise_shape"][0]
    cands = _randn(5, (4,) + tuple(cfg["noise_shape"])).to(cuda_dev)
    whole = S.make_denoise_fn(smp, max_images=4 * B, seed=11).denoise_candidates(cands, 0)
    assert smp.graph_captures == 1
    serial = S.make_denoise_fn(smp, max_images=B, seed=11)
    got = torch.stack([serial(c) for c in cands])
    assert torch.equal(got, whole) and smp.graph_captures == 2
    chunked = S.make_denoise_fn(smp, max_images=B, seed=11).denoise_candidates(cands, 0)
    assert torch.equal(chunked, whole) and smp.graph_captures == 2


def _compare_with_oracle(h, ref_h, N, tol, strict):
    for r, (got, ref) in enumerate(zip(h["scores"], ref_h["scores"])):
        got, ref = np.array(got), np.array(ref)
        print("round %d: scores %s vs oracle %s" % (r, got, ref))
        assert h["rounds"][r] == ref_h["rounds"][r]
        assert np.abs(got - ref).max() <= tol, r
        if h["survivors"][r] == ref_h["survivors"][r]:
            continue
        assert not strict, r
        # the survivors differ: only where the oracle's ranking near the cut is within the tolerance
        top = np.sort(ref)[::-1][: N + 1]
        assert np.diff(top).__abs__().min() <= 2 * tol, r
        far = np.abs(ref[:, None] - ref[None, :]) > 2 * tol
        assert np.array_equal((got[:, None] > got[None, :])[far], (ref[:, None] > ref[None, :])[far])
        return False                          # later rounds start from other states
    return True


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["16bit", "fp32"])
@pytest.mark.parametrize("name", ["u_sop", "c_sop"])
def test_search_over_paths_vs_oracle(cuda_dev, name, precision):
    cfg = SOP_CASES[name]
    net, sd = build_shell(cfg, cuda_dev)
    net.precision = precision
    smp = _sampler(cfg, net, cuda_dev)
    x_T, fwd, step_noise, labels = _sop_inputs(cfg)
    img, score, h, sop = _search(cfg, smp, cuda_dev, step_noise=step_noise, fwd=fwd, x_T=x_T, labels=labels)
    sched = O.schedule(cfg["beta_1"], cfg["beta_T"], cfg["T"])
    N, M = cfg["n_beams"], cfg["n_children"]
    with torch.no_grad():
        ref_img, ref_score, ref_h = search_over_paths(
            sd, sched, x_T, lambda t: step_noise[t], fwd, N, M, cfg["start_step"], cfg["delta_f"], cfg["delta_b"],
            O.VERIFIERS[cfg["verifier"]], labels, cfg.get("w", 0.0))
    strict = precision == "fp32"
    tol = 1e-4 if strict else SCORE_TOL
    if _compare_with_oracle(h, ref_h, N, tol, strict):
        last = np.sort(np.array(ref_h["scores"][-1]))[::-1]
        if strict or last[0] - last[1] > 2 * tol:
            assert h["lineage"] == ref_h["lineage"] and sop.last_index == ref_h["lineage"]["path"]
            assert abs(score - ref_score) <= tol
            assert (img.cpu() - ref_img).abs().max().item() <= (1e-3 if strict else 5e-2)
    steps = N * (cfg["T"] - 1 - cfg["start_step"]) + sum(N * M * (sp - e + 1) for _, sp, e in h["rounds"])
    assert sop.nfes == steps
    assert h["unet_image_steps"] == steps * cfg["noise_shape"][0] * (2 if cfg["kind"] == "cond" else 1)


@pytest.mark.gpu
def test_single_path_is_the_plain_sampler(cuda_dev):
    """N = M = 1, delta_f = 0 with injected step noise: the plain sampler's image, bit for bit."""
    cfg = SOP_CASES["u_sop"]
    net, _ = build_shell(cfg, cuda_dev)
    smp = _sampler(cfg, net, cuda_dev)
    step_noise = cases.search_noise(cfg).to(cuda_dev)
    x_T = _randn(12, (1,) + tuple(cfg["noise_shape"])).to(cuda_dev)
    img, score, h, _ = _search(cfg, smp, cuda_dev, step_noise=step_noise, x_T=x_T, n_beams=1, n_children=1,
                               delta_f=0, delta_b=2)
    ref = smp(x_T[0], noise=step_noise)
    assert torch.equal(img, ref)
    assert score == _verifier(cfg["verifier"]).score(ref)


@pytest.mark.gpu
def test_results_do_not_depend_on_chunking_and_follow_the_seed(cuda_dev):
    cfg = SOP_CASES["u_sop"]
    net, _ = build_shell(cfg, cuda_dev)
    smp = _sampler(cfg, net, cuda_dev)
    a = _search(cfg, smp, cuda_dev, seed=31, max_images=4)
    b = _search(cfg, smp, cuda_dev, seed=31, max_images=256)
    c = _search(cfg, smp, cuda_dev, seed=31, max_images=256)
    d = _search(cfg, smp, cuda_dev, seed=32, max_images=256)
    for other in (b, c):
        assert torch.equal(a[0], other[0]) and a[1] == other[1] and a[2] == other[2]
    assert not torch.equal(a[0], d[0]) and a[2]["scores"] != d[2]["scores"]
    assert a[3].last_seed == 31


@pytest.mark.gpu
def test_unrankable_scores_raise(cuda_dev):
    """The self-supervised score of a one-image candidate is NaN: no child can be ranked."""
    cfg = dict(SOP_CASES["u_sop"], noise_shape=[1, 3, 16, 16], verifier="self_supervised")
    net, _ = build_shell(cfg, cuda_dev)
    smp = _sampler(cfg, net, cuda_dev)
    with pytest.raises(ValueError, match="ranked"):
        _search(cfg, smp, cuda_dev)


@pytest.mark.gpu
def test_run_search_returns_the_search_images(cuda_dev):
    from its_b200 import inference as I
    from its_b200.search import search_algorithm as S
    cfg = SOP_CASES["u_sop"]
    net, _ = build_shell(cfg, cuda_dev)
    smp = _sampler(cfg, net, cuda_dev)
    B, H = cfg["noise_shape"][0], cfg["noise_shape"][2]
    conf = dict(img_size=H, batch_size=B, search=dict(algorithm="search_over_paths", verifier="oracle",
                                                      n_beams=2, n_children=3, start_step=6, delta_f=1, delta_b=3))
    best, score, images = I.run_search(smp, conf, cuda_dev, seed=8)
    img, ref_score, h, sop = _search(cfg, smp, cuda_dev, seed=8)
    assert torch.equal(images, img) and score == ref_score
    assert torch.equal(best, S.philox_normal((1, B, 3, H, H), 8, h["lineage"]["path"], S.TAG_X_T, cuda_dev)[0])
