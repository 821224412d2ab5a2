#!/usr/bin/env python
"""Headline benchmark: candidate images / second of the inference-time-scaling
sampling path (BASELINE.json: "candidate images/sec (T=1000 NFE, verifier incl.)").

One "step" = one complete random search over the candidate population owned by a
GPU: every candidate runs the full T=1000 DDPM ancestral loop over the
unconditional CIFAR-10 UNet (config A/B of SURVEY.md §8), the finished samples are
scored by the verifier kernels and the best one is selected by the first-index
argmax (+ one all_gather of the scores when several GPUs take part).

    python bench.py --gpus 1 --steps K --warmup W                (our CUDA path)
    torchrun ... bench.py --gpus N --steps K --warmup W          (one rank per GPU, weak scaling)
    python bench.py --impl reference --steps K --warmup W        (the reference's CPU path)

Prints ONE JSON line (rank 0).  `value` is device-timed with the candidates
already resident in HBM; `e2e` goes through the public search API with the
candidate noise in pinned HOST memory (H2D inside the timed region) and the
scores + winning noise read back (D2H).  `roofline` is the tcgen05 tap-GEMM
family, timed launch by launch with CUDA events; `cpu_baseline` is the CPU port
of the reference path (oracle/) on this box's host cores.

`--dump-outputs DIR` writes what the last timed step returned (the winning noise, its score, every candidate's
score and the winner's index) as DIR/<name>.npy.  The weights, candidates and step noise are seeded, so two
builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import contextlib
import io
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the tree may be read-only: the benchmark writes nothing into it

import torch  # noqa: E402

METRIC = "candidate images/sec (T=1000 NFE, verifier incl.)"
UNIT = "images/s"
CFG_A = dict(T=1000, ch=128, ch_mult=[1, 2, 3, 4], attn=[1], num_res_blocks=2, dropout=0.15)
BETA_1, BETA_T = 1e-4, 0.02
# The default workload is BASELINE.json configs[1] (the configuration the metric is quoted on).  C and E
# are the other single-GPU shards of BASELINE.json (configs[2]: 256 guided candidates over 8 GPUs = 32 per
# GPU; configs[4]: 1024 candidates of the 64x64 net over 8 GPUs = 128 per GPU), run by hand / scripts.
WORKLOADS = {
    "A": dict(name="random_search_N64_uncond_cifar10_T1000 (BASELINE.json configs[1])", cond=False, img=32, T=1000,
              attn=[1], candidates=64, w=0.0,
              unet="Model.UNet ch=128 ch_mult=[1,2,3,4] attn=[1] num_res_blocks=2, random init"),
    "C": dict(name="random_search_cfg_w1.8_cond_cifar10_T1000 (BASELINE.json configs[2], 32 candidates per GPU)",
              cond=True, img=32, T=1000, attn=None, candidates=32, w=1.8,
              unet="ModelCondition.UNet num_labels=10 ch=128 ch_mult=[1,2,3,4] num_res_blocks=2, random init"),
    "E": dict(name="random_search_uncond_imagenet64_T2000 (BASELINE.json configs[4], 128 candidates per GPU)",
              cond=False, img=64, T=2000, attn=[2], candidates=128, w=0.0,
              unet="Model.UNet ch=128 ch_mult=[1,2,3,4] attn=[2] num_res_blocks=2 on 3x64x64, random init"),
}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(source="measured (MEASURED_PEAKS.json)", hbm=p["hbm_gbs"], burst=p["bf16_tflops"],
                    sustained=p.get("bf16_tflops_sustained", p["bf16_tflops"]))
    return dict(source="fallback (B200_PROFILING.md)", hbm=6650.0, burst=1590.0, sustained=1400.0)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        if self.proc is not None:
            self.proc.terminate()
            self.thread.join(timeout=2)

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------ CPU arm --
def _host_threads():
    """Threads the CPU arm may use: the cores this process is allowed on.  torchrun exports OMP_NUM_THREADS=1
    to its workers, which is what starved the round-1 reference arm at N > 1: set the count explicitly."""
    try:
        n = len(os.sched_getaffinity(0))
    except (AttributeError, OSError):
        n = os.cpu_count() or 1
    torch.set_num_threads(max(1, n))
    return torch.get_num_threads()


def _load_reference():
    """The reference's own modules (Diffusion/Diffusion.py, Diffusion/Model.py, search/verifier.py) loaded by file
    path when a checkout is reachable ($ITS_REF_DIR, then /root/reference — the build container only; the GPU
    box has none).  Returns None when absent: the oracle port (oracle/ddpm_oracle.py) is timed instead."""
    import importlib.util
    for root in (os.environ.get("ITS_REF_DIR"), "/root/reference"):
        if not root or not os.path.exists(os.path.join(root, "Diffusion", "Diffusion.py")):
            continue
        mods = {}
        try:
            for name, rel in (("diffusion", "Diffusion/Diffusion.py"), ("model", "Diffusion/Model.py"),
                              ("verifier", "search/verifier.py")):
                spec = importlib.util.spec_from_file_location("bench_ref_" + name, os.path.join(root, rel))
                mod = importlib.util.module_from_spec(spec)
                with contextlib.redirect_stdout(io.StringIO()):
                    spec.loader.exec_module(mod)
                mods[name] = mod
        except Exception:       # noqa: BLE001 — a broken checkout must not take the bench line down
            continue
        return mods
    return None


class CpuArm:
    """The reference's CPU path for workload A: `n_steps` of the T = 1000 ancestral loop over `batch` candidate
    images (Diffusion.py:84-102 through its public seam p_mean_variance) + OracleVerifier.score (verifier.py:62),
    fp32, every host thread.  The loop is step-homogeneous, so candidate images/s for the full trajectory is
    batch / (seconds * T / n_steps)."""

    def __init__(self, seed: int = 0):
        self.T = CFG_A["T"]
        self.threads = _host_threads()
        self.ref = _load_reference()
        torch.manual_seed(seed)
        if self.ref is not None:
            self.kind = "reference"
            net = self.ref["model"].UNet(**CFG_A).eval()
            self.smp = self.ref["diffusion"].GaussianDiffusionSampler(net, BETA_1, BETA_T, self.T)
            self.ver = self.ref["verifier"].OracleVerifier()
        else:
            from oracle import ddpm_oracle as O
            from its_b200.Diffusion import UNet
            self.kind = "port"
            self.O = O
            net = UNet(**CFG_A)                      # same constructor / initialisers as the reference
            self.sd = {k: v.detach().clone() for k, v in net.state_dict().items()}
            self.sched = O.schedule(BETA_1, BETA_T, self.T)

    def sample(self, batch: int, n_steps: int):
        """(seconds, extrapolated candidate images/s)."""
        T = self.T
        n_steps = max(1, min(n_steps, T))
        x = torch.randn(batch, 3, 32, 32)
        t0 = time.perf_counter()
        with torch.no_grad(), contextlib.redirect_stdout(io.StringIO()):
            for time_step in range(T - 1, T - 1 - n_steps, -1):
                t = torch.full((batch,), time_step, dtype=torch.long)
                if self.ref is not None:
                    mean, var = self.smp.p_mean_variance(x_t=x, t=t)
                else:
                    mean, var, _ = self.O.p_mean_variance(self.sd, self.sched, x, t)
                x = mean + torch.sqrt(var) * torch.randn_like(x)
            x0 = torch.clip(x, -1, 1)
            if self.ref is not None:
                self.ver.score(x0)
            else:
                self.O.oracle_verifier_score(x0)
        dt = time.perf_counter() - t0
        return dt, batch / (dt * T / n_steps)

    def describe(self, batch, n_steps, dt):
        what = ("the reference's own modules (Diffusion/Diffusion.py + Model.py + search/verifier.py, loaded by path)"
                if self.ref is not None else "oracle port of Diffusion.py:84-102 + verifier.py:62 (oracle/ddpm_oracle.py)")
        return (f"{what}, config A, {batch} candidate images per sample, {n_steps} of {self.T} denoising steps "
                f"({dt:.1f} s) + verifier, extrapolated x{self.T / n_steps:.1f} (the loop is step-homogeneous); "
                f"{self.threads} threads on {os.cpu_count()} logical CPUs")


def cpu_sample_for_budget(arm: CpuArm, batch: int, n_samples: int, budget_s: float, forced: int = 0):
    """(candidates per CPU sample, denoising steps per sample) so that `n_samples` samples fit `budget_s`.
    The population is the workload's own; it is only cut (never below 8 images) when one single denoising
    step of the whole population would already overrun the budget on this host."""
    if forced > 0:
        return batch, forced
    arm.sample(min(batch, 8), 1)                      # page-in / thread pool warm-up
    per = budget_s / max(n_samples, 1)
    while True:
        dt, _ = arm.sample(batch, 1)
        if dt <= per or batch <= 8:
            break
        batch = max(8, batch // 2)
    return batch, max(1, min(arm.T, int(per / max(dt, 1e-3))))


def run_reference(args):
    """`--impl reference`: the CPU arm on the same config / metric / unit as ours.  Under torchrun only rank 0
    works; every other rank exits 0 at once (no process group is created)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if args.workload != "A":
        print(json.dumps({"impl": "reference", "unavailable": "the CPU arm is defined for workload A (BASELINE.json configs[1])"}))
        return
    world = int(os.environ.get("WORLD_SIZE", "1"))
    arm = CpuArm()
    total = args.warmup + args.steps
    # the workload's own per-step population, T sampled
    batch, n_steps = cpu_sample_for_budget(arm, args.candidates, total, args.ref_budget, args.ref_steps)
    vals, secs = [], []
    for i in range(total):
        dt, v = arm.sample(batch, n_steps)
        if i >= args.warmup:
            vals.append(v); secs.append(dt)
    value = statistics.mean(vals)
    sample = arm.describe(batch, n_steps, statistics.mean(secs))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * statistics.mean(secs), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, world),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": arm.threads, "logical_cpus": os.cpu_count(),
                         "kind": arm.kind, "sample": sample},
        "reference_run": {"what": "GPU versus CPU: one host, all threads, no GPU", "candidates_per_sample": batch,
                          "denoising_steps_per_sample": n_steps, "of_T": arm.T, "extrapolation": arm.T / n_steps,
                          "threads": arm.threads, "logical_cpus": os.cpu_count(),
                          "omp_num_threads_env": os.environ.get("OMP_NUM_THREADS")},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def workload_config(args, world):
    wl = WORKLOADS[args.workload]
    cfg = {"workload": wl["name"], "unet": wl["unet"],
           "candidates_per_gpu": args.candidates, "noise_shape": [1, 3, wl["img"], wl["img"]], "T": wl["T"],
           "verifier": "OracleVerifier", "selection": "argmax_first", "global_candidates": args.candidates * world,
           "parallelism": f"candidate-sharded x{world}",
           "l2": "per-step working set (163 MB bf16 weights + >1 GB activations per UNet pass) exceeds the 126 MB L2"}
    if wl["cond"]:
        cfg["guidance_w"] = wl["w"]
        cfg["unet_evals_per_step"] = "2 (conditional + unconditional, one 2B-image pass)"
    return cfg


# ------------------------------------------------------------------ GPU arm --
def run_ours(args):
    import __graft_entry__ as ge
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    if not os.path.exists(ge.LIB_PATH):
        if rank == 0:
            ge.build()
        if world > 1:
            dist.barrier()
    from its_b200.search import search_algorithm as S
    from its_b200.search import verifier as V

    wl = WORKLOADS[args.workload]
    T, img = wl["T"], wl["img"]
    net, smp, labels = build_workload(args.workload, dev)
    n_local, n_total = args.candidates, args.candidates * world
    shape = (1, 3, img, img)
    den = S.make_denoise_fn(smp, labels, max_images=args.candidates, seed=1234)
    ver = V.OracleVerifier()
    rs = S.RandomSearch(n_candidates=n_total)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- value: candidates resident in HBM, device timed ----
    resident = S.philox_normal((n_total,) + shape, 1234, 0, S.TAG_X_T, dev)

    def step_resident():
        return rs.search(shape, den, ver.score, device=str(dev), verbose=False, candidate_noise=resident, seed=1234)

    for _ in range(args.warmup):
        step_resident()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clocks:
        e0.record()
        for _ in range(args.steps):
            best_noise, best_score = step_resident()
        e1.record()
        barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, best_noise=best_noise, best_score=best_score, scores=rs.last_scores,
                     best_index=rs.last_index)
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_per_step = ms.item() / args.steps
    value = n_total / (ms_per_step / 1e3)
    launches_per_traj = smp.last_launches_per_step * T
    gpu_launches = args.steps * (launches_per_traj + 4)   # + image_stats, candidate_scores, argmax, (philox)

    # ---- e2e: public API, candidates in pinned host memory, results read back ----
    host = resident.cpu().pin_memory()
    scores_host = torch.empty(n_total, dtype=torch.float32).pin_memory()

    def step_e2e():
        lo, hi = S._shard(n_total, rank, world)
        cand = torch.empty_like(resident)
        cand[lo:hi].copy_(host[lo:hi], non_blocking=True)            # H2D of this rank's candidates
        bn, bs = rs.search(shape, den, ver.score, device=str(dev), verbose=False, candidate_noise=cand, seed=1234)
        scores_host.copy_(rs.last_scores, non_blocking=True)         # D2H
        out = host[rs.last_index].clone()                            # winner is already on the host
        torch.cuda.synchronize()
        return out, bs

    step_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_e2e()
    barrier()
    dt = torch.tensor([time.perf_counter() - t0], device=dev)
    if world > 1:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    e2e_value = n_total * args.steps / dt.item()
    h2d = n_local * 3 * img * img * 4
    d2h = n_total * 4 + 8

    # ---- roofline of the dominant kernel family: every tap-GEMM launch timed with events ----
    pk = peaks()
    n_net = 2 * n_local if wl["cond"] else n_local
    plan = net.plan(n_net, img, img, n_img_in=n_local, uniform_t=True)
    roof = profile_tapgemm(plan, dev, pk)
    if roof["launches_per_unet_pass"] == 0:          # the fp32 parity path launches no tcgen05 kernel
        roof.update(achieved=0.0, frac=0.0, kernel="f32_conv2d_kernel (CUDA cores; --precision fp32 is the parity path)")
    roof["step_share"] = roof.pop("sum_ms") * T / ms_per_step if ms_per_step else None
    roof["model_flops_frac_of_sustained"] = (value / world) * plan.flops / n_local * T / (pk["sustained"] * 1e12)
    if args.workload == "A" and n_local == 64:
        roof.update(ncu_traffic("tapgemm"))
    hbm = profile_hbm_kernels(plan, smp, dev, pk, n_local, img, wl)
    # BASELINE.json configs[2] and configs[4] on the same record: one bounded search each (N = 1 default run only)
    extra = None
    if world == 1 and args.workload == "A" and not args.no_extra_workloads and PRECISION == "16bit":
        extra = {k: run_extra_workload(k, dev, pk) for k in ("C", "E")}

    line = None
    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu_baseline and args.workload == "A":
            arm = CpuArm()
            b_cpu, n_cpu = cpu_sample_for_budget(arm, n_local, 1, args.cpu_budget, args.ref_steps)
            dt_cpu, v_cpu = arm.sample(b_cpu, n_cpu)
            cpu = {"value": v_cpu, "unit": UNIT, "cores": arm.threads, "logical_cpus": os.cpu_count(), "kind": arm.kind,
                   "sample": arm.describe(b_cpu, n_cpu, dt_cpu)}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32" if PRECISION == "fp32" else "bf16/fp16 operands, fp32 accumulate", "data": "synthetic",
            "config": workload_config(args, world),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": gpu_launches, "roofline": roof, "roofline_hbm_kernels": hbm, "cpu_baseline": cpu,
            "clocks": clocks.summary(),
            "best_score": best_score,
        }
        if extra is not None:
            line["workloads"] = extra
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return line


PRECISION = "16bit"     # --precision: "16bit" (tensor-core path, the headline) or "fp32" (CUDA-core parity path)


def dump_outputs(out_dir, **values):
    """One .npy per value: tensors keep float32, Python scalars (score, index) are stored as float64."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, v in values.items():
        a = v.detach().cpu().numpy().astype(np.float32) if torch.is_tensor(v) else np.asarray(v, dtype=np.float64)
        np.save(os.path.join(out_dir, name + ".npy"), a)


def build_workload(key, dev):
    """(net, sampler, labels) of a workload with random-init weights of that architecture."""
    wl = WORKLOADS[key]
    T = wl["T"]
    torch.manual_seed(0)
    labels = None
    if wl["cond"]:
        from its_b200.DiffusionFreeGuidence import GaussianDiffusionSampler, UNet
        net = UNet(T=T, num_labels=10, ch=128, ch_mult=[1, 2, 3, 4], num_res_blocks=2, dropout=0.15).to(dev).eval()
        smp = GaussianDiffusionSampler(net, BETA_1, BETA_T, T, w=wl["w"]).to(dev)
        labels = torch.tensor([3], dtype=torch.int64, device=dev)     # one class per search (noise_shape batch = 1)
    else:
        from its_b200.Diffusion import GaussianDiffusionSampler, UNet
        net = UNet(**dict(CFG_A, T=T, attn=wl["attn"])).to(dev).eval()
        smp = GaussianDiffusionSampler(net, BETA_1, BETA_T, T).to(dev)
    smp.print_steps = False
    net.precision = PRECISION
    return net, smp, labels


def run_extra_workload(key, dev, pk):
    """One timed random search of another single-GPU shard of BASELINE.json (C: 32 guided candidates, configs[2];
    E: 128 candidates of the 64x64 net at T = 2000, configs[4]) so that those configurations are on the driver's
    record too.  Warm-up = the last steps of a trajectory (plan build, lazy kernel set-up, graph capture), then
    ONE complete search, device-timed, candidates resident in HBM; plus the tap-GEMM family's roofline."""
    from its_b200.search import search_algorithm as S
    from its_b200.search import verifier as V
    wl = WORKLOADS[key]
    T, img, n = wl["T"], wl["img"], wl["candidates"]
    net, smp, labels = build_workload(key, dev)
    shape = (1, 3, img, img)
    den = S.make_denoise_fn(smp, labels, max_images=n, seed=1234)
    ver = V.OracleVerifier()
    rs = S.RandomSearch(n_candidates=n)
    resident = S.philox_normal((n,) + shape, 1234, 0, S.TAG_X_T, dev)
    den.denoise_candidates(resident, 0, t_start=8)                  # warm-up: same plan, same step graph
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    _, best = rs.search(shape, den, ver.score, device=str(dev), verbose=False, candidate_noise=resident, seed=1234)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    value = n / (ms / 1e3)
    n_net = 2 * n if wl["cond"] else n
    plan = net.plan(n_net, img, img, n_img_in=n, uniform_t=True)
    roof = profile_tapgemm(plan, dev, pk)
    sum_ms = roof.pop("sum_ms")
    out = {"workload": wl["name"], "unet": wl["unet"], "candidates": n, "T": T, "value": value, "unit": UNIT,
           "ms_per_search": ms, "searches_timed": 1, "best_score": best,
           "launches_per_step": smp.last_launches_per_step,
           "model_flops_frac_of_sustained": value * plan.flops / n * T / (pk["sustained"] * 1e12),
           "roofline": {k: roof[k] for k in ("bound", "achieved", "peak", "unit", "frac", "launches_per_unet_pass",
                                             "flops_per_unet_pass")}}
    out["roofline"]["step_share"] = sum_ms * T / ms
    del net, smp, plan, den
    torch.cuda.empty_cache()
    return out


def ncu_traffic(family):
    """DRAM bytes (read + write) of one UNet pass of this kernel family, from the committed ncu capture of
    this workload (profiles/r02_traffic_configA_b64.json, written by scripts/summarize_launches.py)."""
    path = os.path.join(ROOT, "profiles", "r02_traffic_configA_b64.json")
    try:
        rec = json.load(open(path))
        fam = rec["families"][family]
        return {"traffic": fam["dram_bytes"], "traffic_unit": "bytes per UNet pass, all launches of the family (ncu dram__bytes_read.sum + dram__bytes_write.sum)",
                "traffic_source": os.path.relpath(path, ROOT)}
    except (OSError, KeyError, ValueError):
        return {"traffic": None}


def _graph_time_ms(fn, reps=20):
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(reps):
            fn()
    g.replay()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record(); g.replay(); e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / reps


def profile_hbm_kernels(plan, smp, dev, pk, n_local, img, wl):
    """The memory-bound kernels of a step against the measured HBM copy bandwidth: every GroupNorm-apply launch of
    one UNet pass (algorithmic bytes: one 16-bit read + one 16-bit write per element) and the fused
    guidance + posterior + Philox-noise + clip step (read x and eps, write x: 12 B per element, 16 guided)."""
    from its_b200 import _lib
    L = _lib.lib()
    gn_ms, gn_n = 0.0, 0
    for (fn, a), (kind, _, _) in zip(plan.ops, plan.op_info):
        if kind != "group_norm_apply":
            continue
        gn_ms += _graph_time_ms(lambda fn=fn, a=a: fn(*a, _lib.stream_ptr()))
        gn_n += 1
    gn_bytes = getattr(plan, "gn_bytes", 0)
    out = {"peak": pk["hbm"], "unit": "GB/s", "peak_source": pk["source"] + ", HBM copy"}
    if gn_ms > 0:
        ach = gn_bytes / (gn_ms * 1e-3) / 1e9
        out["group_norm_apply"] = {"launches_per_unet_pass": gn_n, "algorithmic_bytes_per_unet_pass": gn_bytes,
                                   "achieved": ach, "frac": ach / pk["hbm"],
                                   "note": "inputs were just written by the producing GEMM: largely served by the 126 MB L2"}
    n_per = 3 * img * img
    x = torch.randn(n_local, n_per, device=dev)
    eps = torch.randn(2 * n_local if wl["cond"] else n_local, n_per, device=dev)
    coef = smp._coef_table(dev)
    t_dev = torch.full((1,), 500, dtype=torch.int32, device=dev)
    nan = torch.zeros(1, dtype=torch.int32, device=dev)
    eps_u = eps[n_local:].data_ptr() if wl["cond"] else None
    ms = _graph_time_ms(lambda: L.its_ddpm_step(x.data_ptr(), eps.data_ptr(), eps_u, None, 0, n_local, n_per, coef.data_ptr(),
                                                t_dev.data_ptr(), float(wl["w"]), 1234, 0, nan.data_ptr(), 1,
                                                _lib.stream_ptr()))
    nbytes = n_local * n_per * (16 if wl["cond"] else 12)
    ach = nbytes / (ms * 1e-3) / 1e9
    out["ddpm_step"] = {"algorithmic_bytes": nbytes, "us": ms * 1e3, "achieved": ach, "frac": ach / pk["hbm"],
                        "note": "%d elements per launch: launch-latency bound at this population" % (n_local * n_per)}
    return out


def profile_tapgemm(plan, dev, pk):
    """CUDA-event time of every tcgen05 tap-GEMM launch of one UNet pass, each launch replayed 20x
    back to back inside its own CUDA graph (the regime of the sampler's step graph: device-side
    launch gaps, no Python between launches)."""
    from its_b200 import _lib
    for _ in range(2):
        plan.run()
    torch.cuda.synchronize()
    reps, tot_ms, tot_fl, n, persistent = 20, 0.0, 0, 0, 0
    for (fn, a), (kind, flops, _) in zip(plan.ops, plan.op_info):
        if kind != "tapgemm_sm100":
            continue
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for _ in range(reps):
                fn(*a, _lib.stream_ptr())
        g.replay()
        torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record(); g.replay(); e.record()
        torch.cuda.synchronize()
        tot_ms += s.elapsed_time(e) / reps
        tot_fl += flops
        n += 1
        persistent += int(a[0]._obj.schedule != 1 and a[0]._obj.stats_parts >= 0 and a[0]._obj.out_nchw == 0)
    achieved = tot_fl / (tot_ms * 1e-3) / 1e12 if tot_ms > 0 else 0.0
    return {"bound": "tensor",
            "kernel": "tapgemm_persist_kernel / tapgemm_sm100_kernel (tcgen05 implicit-GEMM conv, all launches of a UNet pass)",
            "achieved": achieved, "peak": pk["burst"], "unit": "TFLOP/s", "frac": achieved / pk["burst"],
            "peak_source": pk["source"] + ", bf16 burst (each launch timed in isolation, 20 graph replays)",
            "peak_sustained": pk["sustained"], "launches_per_unet_pass": n, "flops_per_unet_pass": tot_fl,
            "sum_ms": tot_ms, "traffic": None}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3, help="timed searches (at least 1)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="A", choices=sorted(WORKLOADS), help="A = BASELINE.json configs[1] (default)")
    ap.add_argument("--candidates", type=int, default=None, help="candidates per GPU (weak scaling); default per workload")
    ap.add_argument("--ref-steps", type=int, default=0,
                    help="denoising steps per CPU sample (of T=1000); 0 = sized from the time budget")
    ap.add_argument("--ref-budget", type=float, default=150.0, help="seconds for the whole --impl reference run")
    ap.add_argument("--cpu-budget", type=float, default=20.0, help="seconds for the cpu_baseline leg of our arm")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra-workloads", action="store_true",
                    help="skip the one-search measurements of workloads C and E appended to the default line")
    ap.add_argument("--precision", default="16bit", choices=["16bit", "fp32"],
                    help="16bit = tensor-core path (default, the headline number); fp32 = CUDA-core parity path")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed search's results as DIR/<name>.npy (our arm only)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    global PRECISION
    PRECISION = args.precision
    if args.candidates is None:
        args.candidates = WORKLOADS[args.workload]["candidates"]
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
