"""Batched searches against the same queries searched one after another, on config A's net (ch 128, ch_mult
[1,2,3,4], 32x32, random init N(0, 1.5^2/fan_in), T = 1000, one image per candidate):

  (a) K = 16 queries x N = 4 candidates: 16 RandomSearch.search calls against one RandomSearch.search_batch
  (b) search over paths, K = 8 queries, N = 2, M = 4, start step 900, delta_f 50, delta_b 100: 8
      SearchOverPaths.search calls against one SearchOverPaths.search_batch

x_T, step noise and re-noising draws are injected, so every query's winner (noise or images, score, index or lineage)
must be bit-identical between the two arms; the script asserts it.  Both arms are warmed up, then run alternately
--reps times; the minimum device time of each is reported with searched samples per second (one winner per query).
Prints one JSON line (also written to --out when given).

    python scripts/batched_search_bench.py [--reps 2] [--out path.json]
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
from its_b200.Diffusion import GaussianDiffusionSampler, UNet
from its_b200.search import search_algorithm as S
from its_b200.search import verifier as V
from path_search_bench import gpu_identity, timed


def compare(seq_fn, batch_fn, K, image_steps, reps):
    """Warm both arms, alternate them `reps` times; (report, sequential result, batched result)."""
    seq_fn()
    batch_fn()
    seq, bat = [], []
    for _ in range(reps):
        seq.append(timed(seq_fn))
        bat.append(timed(batch_fn))
    rep = {}
    for name, runs in (("sequential", seq), ("batched", bat)):
        _, ms, host_ms = min(runs, key=lambda r: r[1])
        rep[name] = {"device_ms": round(ms, 2), "host_ms": round(host_ms, 2),
                     "device_ms_all_reps": [round(r[1], 2) for r in runs],
                     "searched_samples_per_s": round(K / (ms / 1e3), 3),
                     "unet_image_steps_per_s": round(image_steps / (ms / 1e3), 1)}
    rep["speedup"] = round(rep["sequential"]["device_ms"] / rep["batched"]["device_ms"], 3)
    return rep, seq[-1][0], bat[-1][0]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    _lib.require_cuda()
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    name, power = gpu_identity()
    T = 1000
    torch.manual_seed(0)
    net = UNet(T=T, ch=128, ch_mult=[1, 2, 3, 4], attn=[1], num_res_blocks=2, dropout=0.15).to(dev).eval()
    with torch.no_grad():        # the reference's zero-gain initialisers would make every score equal
        for p in net.parameters():
            if p.dim() >= 2:
                p.copy_(torch.randn_like(p) * (1.5 / (p[0].numel() ** 0.5)))
    smp = GaussianDiffusionSampler(net, 1e-4, 0.02, T).to(dev)
    smp.print_steps = False
    shape = (1, 3, 32, 32)
    g = torch.Generator(device=dev).manual_seed(7)
    den = S.make_denoise_fn(smp, max_images=256, step_noise=torch.randn((T,) + shape, generator=g, device=dev))
    ver = V.OracleVerifier()
    res = {"gpu": name, "power_limit_and_max_sm_clock": power,
           "net": "config A (Model.UNet ch 128, ch_mult [1,2,3,4], attn [1], 32x32, random init), T = 1000, "
                  "1 image per candidate, OracleVerifier",
           "timing": "CUDA events around each arm; minimum over the alternated reps after one warm-up of each"}

    # (a) random search
    K, N = 16, 4
    x_T = torch.randn((K, N) + shape, generator=g, device=dev)
    rs = S.RandomSearch(n_candidates=N)

    def seq_rs():
        out = [rs.search(shape, den, ver.score, device=str(dev), verbose=False, candidate_noise=x_T[q], seed=1)
               for q in range(K)]
        return torch.stack([o[0] for o in out]), [o[1] for o in out]

    def batch_rs():
        return rs.search_batch(shape, den, ver.score, K, candidate_noise=x_T, seed=1, device=str(dev))

    rep, (s_best, s_scores), (b_best, b_scores) = compare(seq_rs, batch_rs, K, K * N * T, a.reps)
    same = torch.equal(s_best, b_best) and s_scores == b_scores
    assert same, "random search: batched winners differ from the sequential searches"
    res["random_search"] = dict(rep, queries=K, n_candidates=N, unet_image_steps=K * N * T,
                                winners_bit_identical=same)

    # (b) search over paths
    K, N, M = 8, 2, 4
    sop = S.SearchOverPaths(n_beams=N, n_children=M, start_step=900, delta_f=50, delta_b=100)
    rounds = S.path_rounds(T, 900, 50, 100)
    x_T = torch.randn((K, N) + shape, generator=g, device=dev)
    fwd = torch.randn((len(rounds), K, N * M) + shape, generator=g, device=dev)

    def seq_sop():
        out = [sop.search(shape, den, ver.score, device=str(dev), candidate_noise=x_T[q], forward_noise=fwd[:, q],
                          seed=1) for q in range(K)]
        return torch.stack([o[0] for o in out]), [o[1] for o in out], [o[2]["lineage"] for o in out]

    def batch_sop():
        img, scores, h = sop.search_batch(shape, den, ver.score, K, candidate_noise=x_T, forward_noise=fwd, seed=1,
                                          device=str(dev))
        return img, scores, h["lineage"]

    steps = K * (N * (T - 1 - 900) + sum(N * M * (sp - e + 1) for _, sp, e in rounds))
    rep, s_out, b_out = compare(seq_sop, batch_sop, K, steps, a.reps)
    same = torch.equal(s_out[0], b_out[0]) and s_out[1] == b_out[1] and s_out[2] == b_out[2]
    assert same, "search over paths: batched winners differ from the sequential searches"
    res["search_over_paths"] = dict(rep, queries=K, n_beams=N, n_children=M, start_step=900, delta_f=50, delta_b=100,
                                    rounds=len(rounds), unet_image_steps=steps, winners_bit_identical=same)
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
