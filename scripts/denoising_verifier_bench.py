"""Cost and 16-bit parity of the denoising verifier (DenoisingVerifier) on one GPU, at the sizes a user runs:
  * score_candidates for 64 single-image candidates of config A (likelihood) and config C (class), at S = 8 and 32
    levels: device time (warm-up first, then the best of --reps host-timed calls ending in a device synchronise),
    and the memory of the per-image-t plans at max_images;
  * that time as a share of one 64-candidate RandomSearch at T = 1000 with the oracle verifier;
  * one SearchOverPaths (N = M = 8, scripts/path_search_bench.py's schedule) with the denoising verifier against the
    same search with the oracle verifier;
  * 16-bit against fp32 scores of the same 64 images: maximum relative error and rank agreement (Spearman, and
    whether the top candidate is the same), i.e. whether the 16-bit plan resolves the differences between candidates.
The weights are random (N(0, 1.5^2/fan_in)) and the images are samples of that net: the numbers are costs and
parity, not sample quality.  Prints one JSON line and writes it to --out.

    python scripts/denoising_verifier_bench.py [--reps 3] [--out profiles/r05_denoising_verifier_bench.json]
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
import numpy as np
import torch

from its_b200 import _lib
from its_b200.search import search_algorithm as S
from its_b200.search import verifier as V
from path_search_bench import gpu_identity


def host_ms(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return out, (time.perf_counter() - t0) * 1e3


def best_ms(fn, reps):
    fn()                                                   # warm-up: plans, graphs, kernel attributes
    return min(host_ms(fn)[1] for _ in range(reps))


def make_sampler(cond: bool, T: int, dev):
    torch.manual_seed(0)
    if cond:
        from its_b200.DiffusionFreeGuidence import GaussianDiffusionSampler, UNet
        net = UNet(T=T, num_labels=10, ch=128, ch_mult=[1, 2, 3, 4], num_res_blocks=2, dropout=0.15)
    else:
        from its_b200.Diffusion import GaussianDiffusionSampler, UNet
        net = UNet(T=T, ch=128, ch_mult=[1, 2, 3, 4], attn=[1], num_res_blocks=2, dropout=0.15)
    net = net.to(dev).eval()
    with torch.no_grad():        # the reference's zero-gain initialisers would make every score equal
        for p in net.parameters():
            if p.dim() >= 2:
                p.copy_(torch.randn_like(p) * (1.5 / (p[0].numel() ** 0.5)))
    smp = (GaussianDiffusionSampler(net, 1e-4, 0.02, T, w=1.8) if cond else
           GaussianDiffusionSampler(net, 1e-4, 0.02, T)).to(dev)
    smp.print_steps = False
    return net, smp


def spearman(a, b):
    ra, rb = np.argsort(np.argsort(a)), np.argsort(np.argsort(b))
    return float(np.corrcoef(ra, rb)[0, 1])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--T", type=int, default=1000)
    ap.add_argument("--n", type=int, default=64)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--max-images", type=int, default=256)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_denoising_verifier_bench.json"))
    a = ap.parse_args()
    _lib.require_cuda()
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    name, power = gpu_identity()
    T, n = a.T, a.n
    shape = (1, 3, 32, 32)
    res = {"gpu": name, "power_limit_and_max_sm_clock": power, "T": T, "n_candidates": n,
           "max_images": a.max_images, "images_per_candidate": 1, "configs": {}}
    for cfg, cond, kind in (("A", False, "likelihood"), ("C", True, "class")):
        net, smp = make_sampler(cond, T, dev)
        labels = (1 + torch.arange(n, device=dev) % 10) if cond else None
        den = S.make_denoise_fn(smp, None if labels is None else labels[:1], max_images=a.max_images, seed=11)
        rs = S.RandomSearch(n_candidates=n)
        ora = V.OracleVerifier()
        rs_ms = best_ms(lambda: rs.search(shape, den, ora.score, device=str(dev), verbose=False, seed=5), 1)
        # the population the search scored: 64 finished samples of this net (every candidate with its label)
        cands = S.philox_normal((n,) + shape, 5, 0, S.TAG_X_T, dev)
        with torch.no_grad():
            imgs = den.denoise_candidates(cands, 0, seed=5, cand_labels=None if labels is None else labels.view(n, 1))
        imgs = imgs.reshape(n, *shape[1:])
        out = {"random_search_oracle_ms": round(rs_ms, 1), "kind": kind, "levels": {}}
        for S_lv in (8, 32):
            ver = V.DenoisingVerifier(smp, kind, n_levels=S_lv, seed=0, max_images=a.max_images)
            torch.cuda.synchronize()
            net.invalidate_plans()
            torch.cuda.empty_cache()
            m0 = torch.cuda.memory_allocated()
            ms = best_ms(lambda: ver.score_candidates(imgs, 1, labels), a.reps)
            plan_mb = (torch.cuda.memory_allocated() - m0) / 2 ** 20
            halves = 2 if kind == "class" else 1
            per_chunk = max(1, a.max_images // (halves * S_lv))
            entry = {"score_candidates_ms": round(ms, 2), "unet_image_evaluations": n * S_lv * halves,
                     "unet_images_per_pass": halves * S_lv * min(per_chunk, n),
                     "share_of_random_search": round(ms / rs_ms, 4),
                     "plans_and_graph_buffers_MiB": round(plan_mb, 1), "graph_captures": ver.graph_captures}
            if S_lv == 8:                      # 16-bit against fp32 for the same images
                s16 = ver.score_candidates(imgs, 1, labels).cpu().numpy()
                net.precision = "fp32"
                v32 = V.DenoisingVerifier(smp, kind, n_levels=S_lv, seed=0, max_images=a.max_images)
                s32 = v32.score_candidates(imgs, 1, labels).cpu().numpy()
                net.precision = "16bit"
                lik32 = s32 if kind == "likelihood" else V.DenoisingVerifier(
                    smp, "likelihood", n_levels=S_lv, seed=0, max_images=a.max_images).score_candidates(
                    imgs, 1, labels).cpu().numpy()
                gaps = np.diff(np.sort(s32))
                entry["fp16_vs_fp32"] = {
                    "max_rel_err_of_score": float(np.max(np.abs(s16 - s32) / np.abs(s32))),
                    "max_abs_err": float(np.max(np.abs(s16 - s32))),
                    "max_abs_err_over_mean_squared_error": float(np.max(np.abs(s16 - s32) / np.abs(lik32))),
                    "fp32_score_spread": float(s32.max() - s32.min()),
                    "fp32_median_gap_between_neighbours": float(np.median(gaps)),
                    "spearman": round(spearman(s16, s32), 4),
                    "same_top_candidate": bool(int(np.argmax(s16)) == int(np.argmax(s32))),
                    "top8_overlap": len(set(np.argsort(-s16)[:8].tolist()) & set(np.argsort(-s32)[:8].tolist())),
                }
            out["levels"][str(S_lv)] = entry
        res["configs"][cfg] = out
        if cfg == "A":
            # search over paths, N = M = 8 (path_search_bench.py's schedule), denoising verifier vs oracle verifier
            sop = S.SearchOverPaths(n_beams=8, n_children=8, start_step=900, delta_f=50, delta_b=100)
            den = S.make_denoise_fn(smp, max_images=a.max_images, seed=11)
            dv = V.DenoisingVerifier(smp, "likelihood", n_levels=8, seed=0, max_images=a.max_images)
            t_ora = best_ms(lambda: sop.search(shape, den, ora.score, device=str(dev), seed=5), 1)
            t_den = best_ms(lambda: sop.search(shape, den, dv.score, device=str(dev), seed=5), 1)
            rounds = S.path_rounds(T, 900, 50, 100)
            res["search_over_paths_N8_M8"] = {
                "rounds": len(rounds), "oracle_verifier_ms": round(t_ora, 1), "denoising_verifier_ms": round(t_den, 1),
                "scoring_unet_image_evaluations": len(rounds) * 64 * 8, "overhead": round(t_den / t_ora - 1, 4)}
        del net, smp, den
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
