"""Feynman-Kac steering on config A's net (ch 128, ch_mult [1,2,3,4], 32x32, T = 1000), N = 64 single-image
particles resampled every 50 steps from step 800 (16 resamplings), and a batch of K = 8 queries x N = 8: device time
of one search, the UNet share (captured single-pass time x passes), the time outside the UNet split into the x0 step,
x0 scoring, its_resample_systematic and the rest (gathers, index_select, host gaps), and a RandomSearch(64) at the
identical UNet budget.  Prints one JSON line (also written to --out when given).

    python scripts/fk_steering_bench.py [--reps 3] [--out path.json]

The weights are random (N(0, 1.5^2/fan_in)), so the scores and the resampling say nothing about sample quality.
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch

from its_b200 import _lib
from its_b200.Diffusion import GaussianDiffusionSampler, UNet
from its_b200.search import search_algorithm as S
from its_b200.search import verifier as V
from scripts.path_search_bench import gpu_identity, per_launch_ms, timed, unet_pass_ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--T", type=int, default=1000)
    ap.add_argument("--n-particles", type=int, default=64)
    ap.add_argument("--start-step", type=int, default=800)
    ap.add_argument("--interval", type=int, default=50)
    ap.add_argument("--lam", type=float, default=10.0)
    ap.add_argument("--queries", type=int, default=8)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    _lib.require_cuda()
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    name, power = gpu_identity()
    T, N, K = a.T, a.n_particles, a.queries
    torch.manual_seed(0)
    net = UNet(T=T, ch=128, ch_mult=[1, 2, 3, 4], attn=[1], num_res_blocks=2, dropout=0.15).to(dev).eval()
    with torch.no_grad():        # the reference's zero-gain initialisers would make every score equal
        for p in net.parameters():
            if p.dim() >= 2:
                p.copy_(torch.randn_like(p) * (1.5 / (p[0].numel() ** 0.5)))
    smp = GaussianDiffusionSampler(net, 1e-4, 0.02, T).to(dev)
    smp.print_steps = False
    shape = (1, 3, 32, 32)
    den = S.make_denoise_fn(smp, max_images=256, seed=11)
    ver = V.OracleVerifier()
    segments = S.fk_segments(T, a.start_step, a.interval)
    n_resample = len(segments) - 1

    def best_of(fn):
        fn()                                            # warm-up: plans, step graphs, kernel attributes
        return min((timed(fn) for _ in range(a.reps)), key=lambda r: r[1])

    fk = S.FKSteering(n_particles=N, start_step=a.start_step, resample_interval=a.interval, lam=a.lam)
    (_, best_score, hist), fk_ms, fk_host_ms = best_of(lambda: fk.search(shape, den, ver.score, device=str(dev),
                                                                         seed=5))
    t_unet = unet_pass_ms(net, N, dev)
    unet_ms = T * t_unet
    outside_ms = fk_ms - unet_ms

    # the kernels outside the UNet, each alone over repeated launches
    n_per = 3 * 32 * 32
    L = _lib.lib()
    stream = _lib.stream_ptr(dev)
    x, eps, x0 = torch.randn(N, n_per, device=dev), torch.randn(N, n_per, device=dev), torch.empty(N, n_per, device=dev)
    t_dev = torch.tensor([500], dtype=torch.int32, device=dev)
    cand = torch.zeros(1, dtype=torch.int64, device=dev)
    flag = torch.zeros(1, dtype=torch.int32, device=dev)
    coef, x0tab = smp._coef_table(dev), smp._x0_table(dev)
    t_step = per_launch_ms(lambda: _lib.check(L.its_ddpm_step_x0(
        x.data_ptr(), x0.data_ptr(), eps.data_ptr(), None, None, 0, N, n_per, coef.data_ptr(), x0tab.data_ptr(),
        t_dev.data_ptr(), 0.0, 5, cand.data_ptr(), flag.data_ptr(), 1, stream)))
    imgs = torch.rand(N, 3, 32, 32, device=dev) * 2 - 1
    t_score = per_launch_ms(lambda: ver.score_candidates(imgs, 1))
    rewards = torch.rand(N, device=dev)
    carried = torch.rand(N, device=dev)
    t_resample = per_launch_ms(lambda: S.resample_systematic(rewards, carried, a.lam, 1, 5, 3))
    rewards_kn = torch.rand(K * (N // K), device=dev)
    t_resample_kn = per_launch_ms(lambda: S.resample_systematic(rewards_kn, None, a.lam, K, 5, 3))
    components = {
        "ddpm_step_x0_ms": round(t_step * T, 3),
        "x0_scoring_ms": round(t_score * len(segments), 3),
        "resample_ms": round(t_resample * n_resample, 3),
    }
    components["gathers_host_gaps_and_rest_ms"] = round(outside_ms - sum(components.values()), 3)

    # K queries x N/K particles: the same population of N images per step
    fkb = S.FKSteering(n_particles=N // K, start_step=a.start_step, resample_interval=a.interval, lam=a.lam)
    (_, b_scores, b_hist), fkb_ms, _ = best_of(lambda: fkb.search_batch(shape, den, ver.score, K, seed=5,
                                                                        device=str(dev)))

    # RandomSearch at the identical UNet budget: N candidates of T steps
    rs = S.RandomSearch(n_candidates=N)
    (_, rs_score), rs_ms, _ = best_of(lambda: rs.search(shape, den, ver.score, device=str(dev), verbose=False, seed=5))

    image_steps = hist["unet_image_steps"]
    res = {
        "gpu": name, "power_limit_and_max_sm_clock": power,
        "workload": {"net": "config A (ch 128, ch_mult [1,2,3,4], 32x32, 1 image per particle), random weights",
                     "T": T, "n_particles": N, "start_step": a.start_step, "resample_interval": a.interval,
                     "lam": a.lam, "segments": len(segments), "resamplings": n_resample},
        "fk_steering": {
            "device_ms": round(fk_ms, 2), "host_ms": round(fk_host_ms, 2), "unet_image_steps": image_steps,
            "image_steps_per_s": round(image_steps / (fk_ms / 1e3), 1), "best_score": best_score,
            "mean_ess": round(sum(hist["ess"]) / max(1, len(hist["ess"])), 2),
            "unet_pass_ms": {"batch_%d" % N: round(t_unet, 4)}, "unet_ms": round(unet_ms, 2),
            "unet_share": round(unet_ms / fk_ms, 4), "outside_unet_ms": round(outside_ms, 2),
            "outside_unet_share": round(outside_ms / fk_ms, 4), "outside_components": components,
        },
        "fk_steering_batch": {
            "n_queries": K, "n_particles": N // K, "device_ms": round(fkb_ms, 2),
            "unet_image_steps": b_hist["unet_image_steps"],
            "outside_unet_share": round((fkb_ms - unet_ms) / fkb_ms, 4), "best_scores": b_scores,
        },
        "kernels": {
            "its_resample_systematic_us": {"1x%d" % N: round(t_resample * 1e3, 2),
                                           "%dx%d" % (K, N // K): round(t_resample_kn * 1e3, 2)},
            "its_ddpm_step_x0_us": round(t_step * 1e3, 2), "score_candidates_us": round(t_score * 1e3, 2),
        },
        "random_search_same_budget": {"n_candidates": N, "unet_image_steps": N * T, "device_ms": round(rs_ms, 2),
                                      "best_score": rs_score,
                                      "image_steps_per_s": round(N * T / (rs_ms / 1e3), 1)},
    }
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
