"""Fingerprint of the UNet execution plans: every launch of every plan in a matrix of nets, precisions and
plan settings, written as one JSON file per plan.  Pointers are replaced by (buffer ordinal by first use, byte
offset), so two builds that write byte-identical directories build the same launch lists; each file also holds
a sha256 of eps after one evaluation on seeded inputs.  Needs a GPU.
Usage: python scripts/plan_fingerprint.py OUT_DIR"""
import bisect
import ctypes as C
import hashlib
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from tests import cases
from tests.util import build_shell
from its_b200.engine import UNetPlan
from its_b200.engine_f32 import UNetPlanF32

# MainCondition.py's own shapes (scripts/stretch_maincondition.py): maps down to 1x1
MAINCOND = dict(kind="cond", T=3000, num_labels=10, ch=128, ch_mult=[1, 4, 8, 8, 4, 2], num_res_blocks=2,
                dropout=0.15, weight_seed=5, img=32, B=2)
NETS = dict(cases.FORWARD_CASES, maincond=MAINCOND)
# 16-bit plan settings: (environment, impl)
SETTINGS16 = {"gn0": ({"ITS_GN_FUSION": "0"}, None), "gnauto": ({"ITS_GN_FUSION": "auto"}, None),
              "gn1": ({"ITS_GN_FUSION": "1"}, None), "res16": ({"ITS_RESIDUAL_FP16": "1"}, None),
              "impl1": ({}, 1), "fork0": ({"ITS_FORK_TIME": "0"}, None)}
KNOBS = ("ITS_GN_FUSION", "ITS_RESIDUAL_FP16", "ITS_FORK_TIME")


class Pointers:
    """Device address -> ["buf", ordinal by first use, byte offset] over the buffers a plan owns."""

    def __init__(self, plan):
        bufs = list(plan.keep) + [getattr(plan, n) for n in ("x_in", "eps", "t_dev", "t_idx", "labels")]
        spans = sorted({(t.data_ptr(), t.data_ptr() + t.numel() * t.element_size()) for t in bufs if t is not None})
        self.spans, self.los, self.ids = spans, [lo for lo, _ in spans], {}

    def __call__(self, p):
        i = bisect.bisect_right(self.los, p) - 1
        hit = [self.spans[i]] if i >= 0 and p < self.spans[i][1] else [s for s in self.spans if s[0] <= p < s[1]]
        if not hit:
            return p if p < 2 ** 32 else "unresolved"
        lo = hit[0][0]
        return ["buf", self.ids.setdefault(lo, len(self.ids)), p - lo]


def plain(v, ptr):
    if hasattr(v, "_obj"):                      # C.byref(desc)
        v = v._obj
    if isinstance(v, C.Structure):
        return {f: plain(getattr(v, f), ptr) for f, _ in v._fields_}
    if isinstance(v, (C.Array, list)):
        return [plain(x, ptr) for x in v]
    if isinstance(v, int) and not isinstance(v, bool):
        return ptr(v)
    return v


def fingerprint(plan, cfg):
    ptr = Pointers(plan)
    rec = {"ops": [[fn.__name__, kind, n, fl, plain(list(a), ptr)]
                   for (fn, a), (kind, fl, n) in zip(plan.ops, plan.op_info)],
           "label_ops": [[fn.__name__, plain(list(a), ptr)] for fn, a in plan.label_ops]}
    fork = getattr(plan, "fork_time_chain", False)
    rec["fork"] = [plan._n_time_ops, plan._join_at] if fork else None
    for k in ("n_launches", "n_label_launches", "n_gn_fused", "gn_bytes", "flops"):
        rec[k] = getattr(plan, k, 0)          # the fp32 plan has no GroupNorm fusion counters
    g = torch.Generator().manual_seed(1234)
    with torch.no_grad():
        plan.x_in.copy_(torch.randn(plan.x_in.shape, generator=g))
        plan.t_idx.copy_(torch.randint(0, cfg["T"], (plan.n_img,), generator=g))
        plan.t_dev.fill_(cfg["T"] // 2)
        if plan.labels is not None:
            plan.labels.copy_(torch.randint(0, cfg["num_labels"] + 1, (plan.n_img,), generator=g))
    try:
        plan.run_label_ops()
        plan.run()
        torch.cuda.synchronize()
        rec["eps_sha256"] = hashlib.sha256(plan.eps.cpu().numpy().tobytes()).hexdigest()
    except RuntimeError as e:   # a launch the library refuses (MainCondition's 1536-channel GroupNorm with impl=1)
        torch.cuda.synchronize()
        rec["eps_sha256"] = f"refused: {e}"
    return rec


def main(out_dir):
    os.makedirs(out_dir, exist_ok=True)
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    for name, cfg in NETS.items():
        net, _ = build_shell(cfg, dev)
        B, S = cfg["B"], cfg["img"]
        guided = cfg["kind"] == "cond"
        for uniform in (True, False):
            shape = dict(n_img=2 * B if guided else B, n_img_in=B) if uniform else dict(n_img=B, n_img_in=B)
            runs = [("f32", UNetPlanF32, {}, None)] + [(s, UNetPlan, e, i) for s, (e, i) in SETTINGS16.items()]
            for tag, cls, env, impl in runs:
                for k in KNOBS:
                    os.environ.pop(k, None)
                os.environ.update(env)
                with torch.no_grad():
                    plan = cls(net, shape["n_img"], S, S, n_img_in=shape["n_img_in"], uniform_t=uniform, impl=impl)
                rec = fingerprint(plan, cfg)
                fn = os.path.join(out_dir, f"{name}_{'uniform' if uniform else 'per_image'}_t_{tag}.json")
                with open(fn, "w") as f:
                    json.dump(rec, f)
                print(fn, rec["n_launches"], rec["eps_sha256"][:12], flush=True)
                del plan
                torch.cuda.empty_cache()
        del net


if __name__ == "__main__":
    main(sys.argv[1])
