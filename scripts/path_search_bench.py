"""Search over paths on config A's net (ch 128, ch_mult [1,2,3,4], 32x32, T = 1000), N = M = 8 (64 children per
round): device time of one search, its UNet image-steps, the share of time spent outside the UNet segments
(expand, x0 step, top-k, scoring, gathers, host gaps), achieved GB/s of its_path_expand and its_ddpm_step_x0, and a
RandomSearch at the same UNet-step budget.  Prints one JSON line (also written to --out when given).

    python scripts/path_search_bench.py [--reps 3] [--out path.json]

Time outside the UNet = search time - (UNet steps at each batch size x time of one captured UNet pass at that
batch size).  The weights are random (N(0, 1.5^2/fan_in)), so the scores say nothing about sample quality.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch

from its_b200 import _lib
from its_b200.Diffusion import GaussianDiffusionSampler, UNet
from its_b200.search import search_algorithm as S
from its_b200.search import verifier as V


def gpu_identity():
    name = torch.cuda.get_device_name(0)
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        power = r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return name, power


def timed(fn):
    """(result, device ms, host ms) of fn() between two events on the current stream."""
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    out = fn()
    e1.record()
    e1.synchronize()
    return out, e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3


def per_launch_ms(fn, n=200):
    for _ in range(5):
        fn()
    _, ms, _ = timed(lambda: [fn() for _ in range(n)])
    return ms / n


def unet_pass_ms(net, n_img, dev, reps=20):
    """One UNet pass of n_img 32x32 images, replayed from a captured graph (the sampler's own plan)."""
    plan = net.plan(n_img, 32, 32, n_img_in=n_img, uniform_t=True, impl=getattr(net, "impl", None))
    plan.x_in.copy_(torch.randn(n_img, 3, 32, 32, device=dev))
    plan.t_dev.fill_(500)
    plan.run()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(reps):
            plan.run()
    g.replay()
    _, ms, _ = timed(lambda: [g.replay() for _ in range(3)])
    return ms / (3 * reps)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--T", type=int, default=1000)
    ap.add_argument("--n-beams", type=int, default=8)
    ap.add_argument("--n-children", type=int, default=8)
    ap.add_argument("--start-step", type=int, default=900)
    ap.add_argument("--delta-f", type=int, default=50)
    ap.add_argument("--delta-b", type=int, default=100)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    _lib.require_cuda()
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    name, power = gpu_identity()
    T, N, M = a.T, a.n_beams, a.n_children
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
    sop = S.SearchOverPaths(n_beams=N, n_children=M, start_step=a.start_step, delta_f=a.delta_f, delta_b=a.delta_b)
    rounds = S.path_rounds(T, a.start_step, a.delta_f, a.delta_b)

    def run_sop():
        return sop.search(shape, den, ver.score, device=str(dev), seed=5)

    run_sop()                                           # warm-up: plans, step graphs, kernel attributes
    times = [timed(run_sop) for _ in range(a.reps)]
    (_, best_score, hist), sop_ms, sop_host_ms = min(times, key=lambda r: r[1])
    image_steps = hist["unet_image_steps"]
    prefix_steps = T - 1 - a.start_step                 # UNet passes of N images (stage 0)
    round_steps = sum(sp - e + 1 for _, sp, e in rounds)   # UNet passes of N*M images
    t_unet_nm, t_unet_n = unet_pass_ms(net, N * M, dev), unet_pass_ms(net, N, dev)
    unet_ms = round_steps * t_unet_nm + prefix_steps * t_unet_n
    outside_ms = sop_ms - unet_ms

    # kernels of the search, each alone over repeated launches (algorithmic bytes / event time)
    n_c, n_per = N * M, 3 * 32 * 32
    L = _lib.lib()
    states = torch.randn(n_c, n_per, device=dev)
    out = torch.empty_like(states)
    par = torch.arange(N, dtype=torch.int32, device=dev)
    stream = _lib.stream_ptr(dev)
    expand = lambda: _lib.check(L.its_path_expand(out.data_ptr(), states.data_ptr(), par.data_ptr(), N, M, 0, n_c,
                                                   n_c, n_per, 0.9, 0.4, None, 5, 1 << 40, S.TAG_FORWARD, stream))
    t_expand = per_launch_ms(expand)
    expand_bytes = n_c * n_per * 4 * 2                  # read parent state + write child (Philox z in registers)
    x, eps, x0 = torch.randn(n_c, n_per, device=dev), torch.randn(n_c, n_per, device=dev), torch.empty(n_c, n_per, device=dev)
    t_dev = torch.tensor([500], dtype=torch.int32, device=dev)
    cand = torch.zeros(1, dtype=torch.int64, device=dev)
    flag = torch.zeros(1, dtype=torch.int32, device=dev)
    coef, x0tab = smp._coef_table(dev), smp._x0_table(dev)
    step = lambda: _lib.check(L.its_ddpm_step_x0(x.data_ptr(), x0.data_ptr(), eps.data_ptr(), None, None, 0, n_c,
                                                 n_per, coef.data_ptr(), x0tab.data_ptr(), t_dev.data_ptr(), 0.0, 5,
                                                 cand.data_ptr(), flag.data_ptr(), 1, stream))
    t_step = per_launch_ms(step)
    step_bytes = n_c * n_per * 4 * 4                    # read x, eps; write x, x0
    scores = torch.randn(n_c, device=dev)
    t_topk = per_launch_ms(lambda: S._topk_device(scores, N))
    imgs = torch.rand(n_c, 3, 32, 32, device=dev) * 2 - 1
    t_score = per_launch_ms(lambda: ver.score_candidates(imgs, 1))
    components = {
        "ddpm_step_x0_ms": round(t_step * round_steps, 3),
        "path_expand_ms": round(t_expand * len(rounds), 3),
        "topk_ms": round(t_topk * (len(rounds) - 1), 3),
        "scoring_ms": round(t_score * len(rounds), 3),
    }
    components["gathers_host_gaps_and_rest_ms"] = round(outside_ms - sum(components.values()), 3)

    # RandomSearch at the same UNet-step budget (T steps per single-image candidate)
    n_rand = max(1, round(image_steps / T))
    rs = S.RandomSearch(n_candidates=n_rand)
    run_rs = lambda: rs.search(shape, den, ver.score, device=str(dev), verbose=False, seed=5)
    run_rs()
    (_, rs_score), rs_ms, _ = min((timed(run_rs) for _ in range(a.reps)), key=lambda r: r[1])

    res = {
        "gpu": name, "power_limit_and_max_sm_clock": power,
        "workload": {"net": "config A (ch 128, ch_mult [1,2,3,4], 32x32, 1 image per candidate)", "T": T,
                     "n_beams": N, "n_children": M, "start_step": a.start_step, "delta_f": a.delta_f,
                     "delta_b": a.delta_b, "rounds": len(rounds)},
        "search_over_paths": {
            "device_ms": round(sop_ms, 2), "host_ms": round(sop_host_ms, 2), "unet_image_steps": image_steps,
            "image_steps_per_s": round(image_steps / (sop_ms / 1e3), 1), "best_score": best_score,
            "unet_pass_ms": {"batch_%d" % (N * M): round(t_unet_nm, 4), "batch_%d" % N: round(t_unet_n, 4)},
            "unet_ms": round(unet_ms, 2), "outside_unet_ms": round(outside_ms, 2),
            "outside_unet_share": round(outside_ms / sop_ms, 4), "outside_components": components,
        },
        "kernels": {
            "its_path_expand": {"us": round(t_expand * 1e3, 2), "bytes": expand_bytes,
                                "GB_per_s": round(expand_bytes / (t_expand * 1e-3) / 1e9, 1)},
            "its_ddpm_step_x0": {"us": round(t_step * 1e3, 2), "bytes": step_bytes,
                                 "GB_per_s": round(step_bytes / (t_step * 1e-3) / 1e9, 1)},
            "its_topk_first_us": round(t_topk * 1e3, 2), "score_candidates_us": round(t_score * 1e3, 2),
        },
        "random_search_same_budget": {"n_candidates": n_rand, "unet_image_steps": n_rand * T,
                                      "device_ms": round(rs_ms, 2), "best_score": rs_score,
                                      "image_steps_per_s": round(n_rand * T / (rs_ms / 1e3), 1)},
    }
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
