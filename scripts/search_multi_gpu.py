"""Multi-GPU check of the searches (BASELINE.json configs[3]), single and batched: run under torchrun, one rank per GPU.
Every rank must end with the same selection, and that selection must be bit-identical to the one the
same rank computes alone over the whole population (candidate ids, Philox streams and summation orders
do not depend on the number of ranks).  The only collective per round is the score all_gather (search over
paths adds one all_gather of the candidates' states per round).

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29511 \
        scripts/search_multi_gpu.py
"""
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.distributed as dist

rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
if world > 1:
    dist.init_process_group("nccl", device_id=dev)

from its_b200.Diffusion import GaussianDiffusionSampler, UNet
from its_b200.search import search_algorithm as S
from its_b200.search import verifier as V

T = int(os.environ.get("ITS_CHECK_T", "40"))
torch.manual_seed(0)
net = UNet(T=T, ch=64, ch_mult=[1, 2, 2], attn=[1], num_res_blocks=1, dropout=0.0).to(dev).eval()
with torch.no_grad():            # the reference's zero-gain initialisers would make every score equal
    for p in net.parameters():
        if p.dim() >= 2:
            p.copy_(torch.randn_like(p) * (1.5 / (p[0].numel() ** 0.5)))
smp = GaussianDiffusionSampler(net, 1e-4, 0.02, T).to(dev)
smp.print_steps = False
shape = (2, 3, 32, 32)
den = S.make_denoise_fn(smp, max_images=64, seed=11)
ver = V.OracleVerifier()
dver = V.DenoisingVerifier(smp, "likelihood", n_levels=4, seed=3, max_images=64)
x0 = S.philox_normal((1,) + shape, 5, 0, S.TAG_X_T, dev)[0]


def run_all():
    out = {}
    rs = S.RandomSearch(n_candidates=13)            # ragged over 2/4/8 ranks
    bn, bs = rs.search(shape, den, ver.score, device=str(dev), verbose=False, seed=21)
    out["random"] = (bn.clone(), bs, rs.last_scores.clone())
    zo = S.ZeroOrderSearch(n_neighbors=6, lambda_radius=0.95, n_iterations=3)
    zn, zs, zh = zo.search(x0, den, ver.score, device=str(dev), seed=22)
    out["zero_order"] = (zn.clone(), zs, torch.tensor(zh["scores"]))
    for restart in (False, True):
        ps = S.PathSearch(n_paths=5, injection_step=T // 2, noise_scale=0.1)
        pn, pscore, ph = ps.search(x0, den, ver.score, timesteps=T, device=str(dev), seed=23, restart=restart)
        out["path_restart" if restart else "path"] = (pn.clone(), pscore, torch.tensor(ph["scores"]))
    sop = S.SearchOverPaths(n_beams=3, n_children=3, start_step=3 * T // 4, delta_f=T // 8, delta_b=T // 4)
    si, ss, sh = sop.search(shape, den, ver.score, device=str(dev), seed=24)   # 9 children: ragged over 2 ranks
    out["search_over_paths"] = (si.clone(), ss, torch.tensor(sh["scores"]))
    # batched: 3 queries x 5 candidates and 3 queries x 3 x 2 children, ragged over 2/4/8 ranks
    rb = S.RandomSearch(n_candidates=5)
    bn, bs = rb.search_batch(shape, den, ver.score, 3, seed=25, device=str(dev))
    out["random_batch"] = (bn.clone(), bs, rb.last_scores.clone())
    sb = S.SearchOverPaths(n_beams=3, n_children=2, start_step=3 * T // 4, delta_f=T // 8, delta_b=T // 4)
    si, ss, sh = sb.search_batch(shape, den, ver.score, 3, seed=26, device=str(dev))
    out["search_over_paths_batch"] = (si.clone(), ss, torch.tensor(sh["scores"]))
    # the denoising verifier: the model's own scores, with noise common to every candidate on every rank
    rd = S.RandomSearch(n_candidates=13)
    bn, bs = rd.search(shape, den, dver.score, device=str(dev), verbose=False, seed=27)
    out["random_denoising_verifier"] = (bn.clone(), bs, rd.last_scores.clone())
    return out


t0 = time.perf_counter()
sharded = run_all()
torch.cuda.synchronize()
t_sharded = time.perf_counter() - t0
# the same searches with the collective layer switched off: this rank evaluates every candidate
orig = S._dist
S._dist = lambda: (None, 0, 1)
alone = run_all()
S._dist = orig
ok = True
report = {}
for k in sharded:
    n_eq = torch.equal(sharded[k][0], alone[k][0])
    s_eq = torch.equal(sharded[k][2].cpu(), alone[k][2].cpu()) and sharded[k][1] == alone[k][1]
    ok = ok and n_eq and s_eq
    report[k] = {"best_score": sharded[k][1], "noise_bit_identical": n_eq, "scores_bit_identical": s_eq}
if world > 1:
    # every rank holds the same winner
    for k in sharded:
        t = sharded[k][0].clone()
        dist.broadcast(t, src=0)
        same = torch.equal(t, sharded[k][0])
        flag = torch.tensor([int(same)], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        report[k]["all_ranks_agree"] = bool(flag.item())
        ok = ok and bool(flag.item())
    okt = torch.tensor([int(ok)], device=dev)
    dist.all_reduce(okt, op=dist.ReduceOp.MIN)
    ok = bool(okt.item())
if rank == 0:
    print(json.dumps({"world": world, "ok": ok, "seconds_sharded": round(t_sharded, 3), "searches": report}))
if world > 1:
    dist.destroy_process_group()
sys.exit(0 if ok else 1)
