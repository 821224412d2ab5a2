"""Cost of the rank-ensemble verifier (EnsembleVerifier, its_rank_ensemble) on one GPU:
  * its_rank_ensemble alone: device time per launch (CUDA events around --launches back-to-back launches, after a
    warm-up), for (n_seg, seg_len, V) = (1, 64, 2), (16, 64, 3), (1, 4096, 3) and (8, 1024, 8), on integer-valued
    scores (many ties);
  * one RandomSearch(64) over config A's net (T = 1000, 64 single-image candidates) with the ensemble
    [denoising, aesthetic] against the same search with the denoising verifier alone, the two arms alternated
    --reps times after one warm-up each; and the aesthetic verifier's score_candidates time on 64 images, so that the
    difference between the arms can be set against "aesthetic scoring plus one kernel launch".
The weights are random (N(0, 1.5^2/fan_in)): the numbers are costs, not sample quality.  Both arms score the same
candidates, and the ensemble's denoising column must equal the denoising-only scores bit for bit (reported).  Prints
one JSON line and writes it to --out.

    python scripts/ensemble_verifier_bench.py [--reps 3] [--out profiles/r06_ensemble_verifier_bench.json]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
import numpy as np
import torch

from its_b200 import _lib
from its_b200.search import search_algorithm as S
from its_b200.search import verifier as V
from denoising_verifier_bench import best_ms, host_ms, make_sampler
from path_search_bench import gpu_identity

KERNEL_SHAPES = [(1, 64, 2), (16, 64, 3), (1, 4096, 3), (8, 1024, 8)]


def kernel_us(n_seg, seg_len, n_members, launches, dev):
    g = torch.Generator(device="cpu").manual_seed(n_seg * 7919 + seg_len * 31 + n_members)
    scores = torch.randint(-50, 51, (n_seg * seg_len, n_members), generator=g).float().to(dev)
    w = torch.ones(n_members, dtype=torch.float32, device=dev)
    for _ in range(5):
        V.rank_ensemble(scores, w, n_seg)
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    t0.record()
    for _ in range(launches):
        V.rank_ensemble(scores, w, n_seg)
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) * 1e3 / launches


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--T", type=int, default=1000)
    ap.add_argument("--n", type=int, default=64)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--max-images", type=int, default=256)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_ensemble_verifier_bench.json"))
    a = ap.parse_args()
    _lib.require_cuda()
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    name, power = gpu_identity()
    res = {"gpu": name, "power_limit_and_max_sm_clock": power, "kernel_us_per_launch": {}}
    for n_seg, seg_len, nv in KERNEL_SHAPES:
        res["kernel_us_per_launch"][f"n_seg={n_seg},seg_len={seg_len},V={nv}"] = round(
            kernel_us(n_seg, seg_len, nv, a.launches, dev), 2)

    T, n = a.T, a.n
    shape = (1, 3, 32, 32)
    net, smp = make_sampler(False, T, dev)
    den = S.make_denoise_fn(smp, max_images=a.max_images, seed=11)
    alone = V.DenoisingVerifier(smp, "likelihood", n_levels=8, seed=0, max_images=a.max_images)
    ens = V.EnsembleVerifier([V.DenoisingVerifier(smp, "likelihood", n_levels=8, seed=0, max_images=a.max_images),
                              V.AestheticPredictor()])
    arms = {"denoising": (S.RandomSearch(n_candidates=n), alone), "ensemble_denoising_aesthetic":
            (S.RandomSearch(n_candidates=n), ens)}
    times = {k: [] for k in arms}
    for k, (rs, ver) in arms.items():                      # warm-up: step graphs, scoring graphs, plans
        rs.search(shape, den, ver.score, device=str(dev), verbose=False, seed=5)
    for _ in range(a.reps):
        for k, (rs, ver) in arms.items():
            _, ms = host_ms(lambda: rs.search(shape, den, ver.score, device=str(dev), verbose=False, seed=5))
            times[k].append(round(ms, 1))
    cands = S.philox_normal((n,) + shape, 5, 0, S.TAG_X_T, dev)
    with torch.no_grad():
        imgs = den.denoise_candidates(cands, 0, seed=5).reshape(n, *shape[1:])
    members = ens.score_candidates(imgs, 1)
    aest = V.AestheticPredictor()
    d_alone, d_ens = arms["denoising"][0].last_scores, arms["ensemble_denoising_aesthetic"][0].last_scores
    res["random_search_configA"] = {
        "T": T, "n_candidates": n, "images_per_candidate": 1, "score_levels": 8, "max_images": a.max_images,
        "denoising_only_ms": times["denoising"], "ensemble_ms": times["ensemble_denoising_aesthetic"],
        "difference_of_minima_ms": round(min(times["ensemble_denoising_aesthetic"]) - min(times["denoising"]), 2),
        "aesthetic_score_candidates_ms": round(best_ms(lambda: aest.score_candidates(imgs, 1), 10), 3),
        "rank_ensemble_launch_us_n_seg1_seg_len64_V2": res["kernel_us_per_launch"]["n_seg=1,seg_len=64,V=2"],
        "denoising_column_equals_denoising_only_scores": bool(torch.equal(members[:, 0], d_alone)),
        "winner_denoising_only": arms["denoising"][0].last_index,
        "winner_ensemble": arms["ensemble_denoising_aesthetic"][0].last_index,
        "ensemble_scores_finite": bool(torch.isfinite(d_ens).all()),
    }
    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
