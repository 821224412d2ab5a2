"""Cost of searching over the guidance weight (`guidance=`, its_ddpm_step_x0_w) on one GPU:
  (a) its_ddpm_step_x0_w against its_ddpm_step_x0 for 64 guided candidates of config C (3x32x32, x0 prediction on,
      Philox noise): device time per launch, CUDA events around --launches back-to-back launches, the two arms
      alternated --reps times;
  (b) RandomSearch(64) over config C's guided net (T = 1000, one image per candidate) with G = 4 weights against the
      same search at one scalar w, alternated --reps times after one warm-up each;
  (c) the workaround the feature replaces: 4 sequential RandomSearch(16) searches, one per weight (the sampler's w
      set before each, so each one captures its step graph anew, as a user's loop would), against one mixed
      RandomSearch(64).  x_T and the step noise are injected, so candidate i of the mixed search and its copy in
      search i mod 4 run the same trajectory: their scores must agree bit for bit (reported).
The weights are random (N(0, 1.5^2/fan_in)): the numbers are costs, not sample quality.  Prints one JSON line and
writes it to --out.

    python scripts/guidance_search_bench.py [--reps 3] [--out profiles/r07_guidance_search_bench.json]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
import torch

from its_b200 import _lib
from its_b200._sampler_base import guidance_pairs
from its_b200.search import search_algorithm as S
from its_b200.search import verifier as V
from denoising_verifier_bench import host_ms, make_sampler
from path_search_bench import gpu_identity

WEIGHTS = [0.0, 1.0, 1.8, 4.0]


def step_us(launches, reps, dev):
    """(scalar, per-image) µs per launch of the x0 step for 64 guided candidates of config C."""
    L = _lib.lib()
    n_img, n_per, T = 64, 3 * 32 * 32, 1000
    from its_b200.Diffusion import GaussianDiffusionSampler
    smp = GaussianDiffusionSampler(torch.nn.Identity(), 1e-4, 0.02, T).to(dev)    # the schedule tables only
    coef, x0tab = smp._coef_table(dev), smp._x0_table(dev)
    g = torch.Generator(device="cpu").manual_seed(3)
    x = torch.randn(n_img, n_per, generator=g).to(dev)
    e_c, e_u = torch.randn(n_img, n_per, generator=g).to(dev), torch.randn(n_img, n_per, generator=g).to(dev)
    x0 = torch.empty_like(x)
    t_dev = torch.tensor([500], dtype=torch.int32, device=dev)
    cand = torch.zeros(1, dtype=torch.int64, device=dev)
    flag = torch.zeros(1, dtype=torch.int32, device=dev)
    pairs = guidance_pairs([WEIGHTS[i % 4] for i in range(n_img)], n_img, dev)
    s = _lib.stream_ptr(dev)
    arms = {
        "its_ddpm_step_x0": lambda: L.its_ddpm_step_x0(x.data_ptr(), x0.data_ptr(), e_c.data_ptr(), e_u.data_ptr(),
                                                       None, 0, n_img, n_per, coef.data_ptr(), x0tab.data_ptr(),
                                                       t_dev.data_ptr(), 1.8, 7, cand.data_ptr(), flag.data_ptr(), 1,
                                                       s),
        "its_ddpm_step_x0_w": lambda: L.its_ddpm_step_x0_w(x.data_ptr(), x0.data_ptr(), e_c.data_ptr(),
                                                           e_u.data_ptr(), None, 0, n_img, n_per, coef.data_ptr(),
                                                           x0tab.data_ptr(), t_dev.data_ptr(), pairs.data_ptr(), 7,
                                                           cand.data_ptr(), flag.data_ptr(), 1, s),
    }
    out = {k: [] for k in arms}
    for _ in range(reps):
        for k, fn in arms.items():
            for _ in range(20):
                _lib.check(fn(), k)
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            t0.record()
            for _ in range(launches):
                fn()
            t1.record()
            torch.cuda.synchronize()
            out[k].append(round(t0.elapsed_time(t1) * 1e3 / launches, 2))
    out["bytes_per_launch"] = n_img * n_per * 4 * 5      # x in/out, eps_c, eps_u, x0 out (pairs: 512 B)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--T", type=int, default=1000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--launches", type=int, default=500)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07_guidance_search_bench.json"))
    a = ap.parse_args()
    _lib.require_cuda()
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    name, power = gpu_identity()
    res = {"gpu": name, "power_limit_and_max_sm_clock": power,
           "a_step_us_per_launch_64_candidates": step_us(a.launches, a.reps, dev)}

    T, n, G = a.T, 64, len(WEIGHTS)
    shape = (1, 3, 32, 32)
    _, smp = make_sampler(True, T, dev)
    w0 = smp.w
    labels = torch.tensor([3], dtype=torch.int64, device=dev)
    ver = V.OracleVerifier()
    grid = torch.tensor([WEIGHTS[i % G] for i in range(n)], dtype=torch.float64)

    # (b) one search of 64 at G weights against one at the scalar w
    den = S.make_denoise_fn(smp, labels, seed=11)
    arms = {"scalar_w": (S.RandomSearch(n_candidates=n), {}),
            "guidance_G4": (S.RandomSearch(n_candidates=n), {"guidance": grid})}
    times = {k: [] for k in arms}
    for k, (rs, kw) in arms.items():                       # warm-up: plans and step graphs
        rs.search(shape, den, ver.score, device=str(dev), verbose=False, seed=5, **kw)
    for _ in range(a.reps):
        for k, (rs, kw) in arms.items():
            _, ms = host_ms(lambda: rs.search(shape, den, ver.score, device=str(dev), verbose=False, seed=5, **kw))
            times[k].append(round(ms, 1))
    res["b_random_search_64_configC"] = {
        "T": T, "n_candidates": n, "images_per_candidate": 1, "weights": WEIGHTS,
        "scalar_w_ms": times["scalar_w"], "guidance_ms": times["guidance_G4"],
        "difference_of_minima_ms": round(min(times["guidance_G4"]) - min(times["scalar_w"]), 1),
        "chosen_weight": arms["guidance_G4"][0].last_guidance,
    }

    # (c) 4 sequential searches of 16, one per weight, against one mixed search of 64; everything injected
    g = torch.Generator(device="cpu").manual_seed(19)
    x_T = torch.randn((n,) + shape, generator=g).to(dev)
    step_noise = torch.randn((T,) + shape, generator=g).to(dev)
    den_c = S.make_denoise_fn(smp, labels, seed=13, step_noise=step_noise)

    def sequential():
        out = []
        for k, w in enumerate(WEIGHTS):
            smp.w = w
            rs = S.RandomSearch(n_candidates=n // G)
            rs.search(shape, den_c, ver.score, device=str(dev), verbose=False, seed=7, candidate_noise=x_T[k::G])
            out.append(rs.last_scores.clone())
        smp.w = w0
        return out

    def mixed():
        rs = S.RandomSearch(n_candidates=n)
        rs.search(shape, den_c, ver.score, device=str(dev), verbose=False, seed=7, candidate_noise=x_T, guidance=grid)
        return rs.last_scores.clone()

    seq_scores, mix_scores = sequential(), mixed()        # warm-up
    t_seq, t_mix = [], []
    for _ in range(a.reps):
        seq_scores, ms = host_ms(sequential)
        t_seq.append(round(ms, 1))
        mix_scores, ms = host_ms(mixed)
        t_mix.append(round(ms, 1))
    res["c_workaround_4x16_vs_mixed_64_configC"] = {
        "T": T, "weights": WEIGHTS, "sequential_4x16_ms": t_seq, "mixed_64_ms": t_mix,
        "speedup_of_minima": round(min(t_seq) / min(t_mix), 2),
        "scores_bit_identical": all(torch.equal(mix_scores[k::G], seq_scores[k]) for k in range(G)),
    }
    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
