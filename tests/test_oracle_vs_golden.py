"""CPU: the oracle restatement against fixtures produced by the reference itself
(tests/golden/make_golden.py), plus published known-answer vectors."""
import math

import numpy as np
import pytest
import torch

from oracle import ddpm_oracle as O
from oracle import philox
from tests import cases
from tests.util import build_shell, golden


@pytest.mark.parametrize("T,beta_T", [(1000, 0.02), (2000, 0.02), (3000, 0.028)])
def test_schedule_matches_reference_buffers(T, beta_T):
    g = golden("schedule")
    s = O.schedule(1e-4, beta_T, T)
    for k in ("betas", "coeff1", "coeff2", "posterior_var", "var"):
        assert np.array_equal(s[k].numpy(), g[f"T{T}_{k}"]), k


def test_schedule_survey_known_answers():
    """SURVEY.md §8a-a2 probes of the reference."""
    s = O.schedule(1e-4, 0.02, 1000)
    assert abs(s["coeff1"][0].item() - 1.0000500037) < 1e-9
    assert abs(s["coeff1"][999].item() - 1.0101525443) < 1e-9
    assert abs(s["coeff2"][0].item() - 0.0100004999) < 1e-9
    assert abs(s["coeff2"][999].item() - 0.0202034581) < 1e-9
    assert abs(s["var"][0].item() - 5.453188e-05) < 1e-10
    assert abs(s["var"][1].item() - 1.199199e-04) < 1e-9
    assert abs(s["var"][999].item() - 2e-2) < 1e-7
    assert abs(s["alphas_bar"][999].item() - 4.035831e-05) < 1e-10


def test_sampler_shell_buffers_match_reference():
    from its_b200.Diffusion import GaussianDiffusionSampler
    from its_b200.DiffusionFreeGuidence import GaussianDiffusionSampler as CondSampler
    g = golden("schedule")
    for cls, extra in ((GaussianDiffusionSampler, {}), (CondSampler, {"w": 1.8})):
        s = cls(torch.nn.Identity(), 1e-4, 0.02, 1000, **extra)
        for k in ("betas", "coeff1", "coeff2", "posterior_var"):
            assert np.array_equal(getattr(s, k).numpy(), g[f"T1000_{k}"]), k
        assert list(s.state_dict().keys())[:4] == ["betas", "coeff1", "coeff2", "posterior_var"]
        tab = s._coef_table(torch.device("cpu"))
        assert np.allclose(tab[:, 2].numpy(), np.sqrt(g["T1000_var"].astype(np.float32)), rtol=2e-7, atol=0)
        assert np.array_equal(tab[:, 0].numpy(), g["T1000_coeff1"].astype(np.float32))
        assert np.array_equal(tab[:, 1].numpy(), g["T1000_coeff2"].astype(np.float32))


@pytest.mark.parametrize("name", ["u_small", "u_3lvl", "c_small", "u_A", "c_C"])
def test_unet_forward_oracle_vs_reference(name):
    cfg = cases.FORWARD_CASES[name]
    _, sd = build_shell(cfg)       # also proves the shell's state-dict keys/shapes equal the reference's
    x, t, labels = cases.forward_inputs(cfg)
    with torch.no_grad():
        y = O.unet_forward(sd, x, t, labels)
    ref = torch.from_numpy(golden("fwd_" + name)["eps"])
    assert (y - ref).abs().max().item() <= 1e-5 * max(1.0, ref.abs().max().item())


def test_unet_forward_bf16_emulation_is_close():
    """The storage-rounding emulation the GPU tests compare against stays within
    bf16 noise of the fp32 reference (sizes the tolerance used on the GPU)."""
    cfg = cases.FORWARD_CASES["u_small"]
    _, sd = build_shell(cfg)
    x, t, labels = cases.forward_inputs(cfg)
    with torch.no_grad():
        y = O.unet_forward(sd, x, t, labels, quant="bf16")
    ref = torch.from_numpy(golden("fwd_u_small")["eps"])
    assert (y - ref).abs().max().item() < 0.05 * ref.abs().max().item()


@pytest.mark.parametrize("name", ["u_small_T20", "c_small_T20"])
def test_sampler_oracle_vs_reference(name):
    cfg = cases.SAMPLER_CASES[name]
    _, sd = build_shell(cfg)
    x_T, noise, labels = cases.sampler_inputs(cfg)
    sched = O.schedule(cfg["beta_1"], cfg["beta_T"], cfg["T"])
    with torch.no_grad():
        x0 = O.sample(sd, sched, x_T, lambda s: noise[s], labels, cfg.get("w", 0.0))
    g = golden("smp_" + name)
    assert (x0 - torch.from_numpy(g["x0"])).abs().max().item() <= 1e-4
    for k, f in O.VERIFIERS.items():
        assert abs(f(x0) - float(g["score_" + k])) <= 1e-3


def test_verifier_known_answers():
    g = golden("verifier")
    for i, im in enumerate(cases.verifier_images()):
        assert abs(O.oracle_verifier_score(im) - float(g[f"oracle_{i}"])) < 1e-6
        assert abs(O.aesthetic_score(im) - float(g[f"aesthetic_{i}"])) < 1e-6
        a, b = O.self_supervised_score(im), float(g[f"self_supervised_{i}"])
        assert (math.isnan(a) and math.isnan(b)) or abs(a - b) < 1e-6
    # identities probed on the reference (SURVEY.md §8c)
    im = cases.verifier_images()[0]
    assert abs(O.oracle_verifier_score(im) - 1 / (1 + im.flatten(1).var(1).mean().item())) < 1e-7
    assert abs(O.aesthetic_score(im) - 2 * ((im + 1) / 2).flatten(1).std(1).mean().item()) < 1e-6


def test_search_selection_rules_on_golden_scores():
    """The oracle's search loops reproduce the reference's selections from its scores."""
    for name, cfg in cases.SEARCH_CASES.items():
        g = golden("search_" + name)
        rs = list(g["rs_scores"])
        it = iter(rs)
        idx, best, scores = O.random_search([None] * len(rs), lambda z: z, lambda im: next(it))
        assert idx == int(g["rs_best_index"]) and best == float(g["rs_best_score"])
        # first maximum wins on ties, NaN never wins
        idx, best, _ = O.random_search([0, 1, 2, 3], lambda z: z, lambda z: [0.5, float("nan"), 0.7, 0.7][z])
        assert idx == 2 and best == 0.7


def test_philox_known_answers():
    """Random123 kat_vectors, philox4x32 with 10 rounds."""
    z = philox.philox4x32_10(np.zeros((1, 4), np.uint32), np.zeros(2, np.uint32))[0]
    assert [int(v) for v in z] == [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]
    f = philox.philox4x32_10(np.full((1, 4), 0xffffffff, np.uint32), np.full(2, 0xffffffff, np.uint32))[0]
    assert [int(v) for v in f] == [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]
    p = philox.philox4x32_10(np.array([[0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344]], np.uint32),
                             np.array([0xa4093822, 0x299f31d0], np.uint32))[0]
    assert [int(v) for v in p] == [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]
    x = philox.normal(7, 3, 11, 8, 4096)
    assert abs(float(x.mean())) < 0.02 and abs(float(x.std()) - 1.0) < 0.02


def test_gradient_based_search_matches_reference_on_differentiable_callables():
    """GradientBasedSearch (search_algorithm.py:343-438) is host-side torch over arbitrary differentiable
    callables: same Adam trajectory, scores, gradient norms and returned noise as the reference class.
    tests/golden/search_gradient.npz holds that trajectory as this class computed it when it was checked equal,
    value for value, to the reference class; the tolerance only absorbs last-bit differences of CPU kernels."""
    from its_b200.search import search_algorithm as S
    w = torch.linspace(-1, 1, 48).reshape(1, 3, 4, 4)

    def denoise(z, **kw):
        return torch.tanh(z * 0.7 + w)

    def verify(img, **kw):
        return -(img - 0.25).pow(2).mean()

    z0 = torch.sin(torch.arange(48.0)).reshape(1, 3, 4, 4)
    gs = S.GradientBasedSearch(n_iterations=7, lr=0.05)
    bn, bs, hist = gs.search(z0, denoise, verify, device="cpu")
    assert gs.nfes == 7 and len(hist["scores"]) == 7 and len(hist["grad_norms"]) == 7
    assert hist["scores"][-1] > hist["scores"][0] and bs == max(hist["scores"])
    g = golden("search_gradient")
    assert np.allclose(hist["scores"], g["scores"], rtol=1e-6, atol=0)
    assert np.allclose(hist["grad_norms"], g["grad_norms"], rtol=1e-6, atol=0)
    assert abs(bs - float(g["best_score"])) <= 1e-6 * abs(float(g["best_score"]))
    assert np.allclose(bn.numpy(), g["best_noise"], rtol=0, atol=1e-6)
    with pytest.raises(TypeError):
        gs.search(z0, S.SamplerDenoiser(None), verify)


def test_shell_constructor_reproduces_the_reference_init():
    """BASELINE north_star: "the same random-init weights".  torch.manual_seed(0) + the shell's constructor draws
    the parameters of the reference's constructor bit for bit (same modules created and re-initialised in the same
    order, including Model.py:199-204's re-initialisation of the attention projections inside ResBlock.initialize):
    checked against checksums of the reference's state dict stored by tests/golden/make_golden_long2.py."""
    cfg = cases.LONG_CASES["u_A_refinit"]
    g = golden("smp_u_A_refinit")
    from its_b200.Diffusion import UNet
    torch.manual_seed(cfg["init_seed"])
    m = UNet(T=cfg["T"], ch=cfg["ch"], ch_mult=cfg["ch_mult"], attn=cfg["attn"],
             num_res_blocks=cfg["num_res_blocks"], dropout=cfg["dropout"])
    sd = m.state_dict()
    assert len(sd) == len(g["sd_sums"]) == 333
    sums = np.array([float(v.double().sum()) for v in sd.values()])
    sq = np.array([float(v.double().pow(2).sum()) for v in sd.values()])
    # the checksums are fp64 sums of fp32 values: equal up to the summation order of the two runs
    assert np.abs(sums - g["sd_sums"]).max() < 1e-9
    assert (np.abs(sq - g["sd_sq"]) / np.maximum(g["sd_sq"], 1e-30)).max() < 1e-12
    # the quirk: attention output projections inside ResBlocks end with gain 1, block2's conv with gain 1e-5
    assert sd["downblocks.3.attn.proj.weight"].abs().max() > 1e-2 > sd["downblocks.3.block2.3.weight"].abs().max()
