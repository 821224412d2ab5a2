"""Shared machinery of the two GaussianDiffusionSampler shells.

`forward` and `segment` keep the whole trajectory on the device: one CUDA graph
holds {UNet plan, fused DDPM step, step-counter decrement}; it is replayed once per
step with no host synchronisation (the reference syncs on a NaN assert every step,
Diffusion.py:100).  The NaN flag is OR-reduced on the device and checked once per
call, raising the same AssertionError("nan in tensor.").
"""
from __future__ import annotations

from typing import Dict, Optional, Tuple

import torch
import torch.nn.functional as F
from torch import nn

from . import _lib
from ._unet_base import PlannedUNet

X_T_TAG = 0x40000000  # Philox step tags >= this never collide with a time step


def guidance_pairs(guidance, n_img: int, device) -> torch.Tensor:
    """[n_img, 2] fp32 {w, 1 + w} per image from `guidance` (1-D tensor or sequence of n_img finite weights), formed
    in float64 and rounded to fp32 as its_ddpm_step_x0 forms its scalar pair from the Python float w."""
    g = torch.as_tensor(guidance, dtype=torch.float64).to(device)
    if g.dim() != 1 or g.shape[0] != n_img:
        raise ValueError(f"guidance must be 1-D with one weight per image ({n_img}), got shape {list(g.shape)}")
    if not bool(torch.isfinite(g).all()):
        raise ValueError("guidance weights must be finite")
    return torch.stack([g.float(), (1.0 + g).float()], dim=1)


def extract(v, t, x_shape):
    """Coefficients at the given timesteps as [B,1,1,...] fp32 (Diffusion.py:9-16)."""
    out = torch.gather(v, index=t, dim=0).float().to(t.device)
    return out.view([t.shape[0]] + [1] * (len(x_shape) - 1))


class _Trajectory:
    """Device state of one (plan, noise shape, x0, clip[, per-image weights]) and its captured step graph."""

    def __init__(self, plan, x: torch.Tensor, noise_buf: Optional[torch.Tensor], want_x0: bool,
                 per_image_w: bool = False):
        self.plan = plan      # the captured graph bakes pointers into this plan: holding it keeps them alive
        self.noise_buf = noise_buf       # [T, *x.shape] injected noise, shared with the plan's other graphs
        self.x0_buf = torch.empty_like(x, dtype=torch.float32) if want_x0 else None
        self.nan_flag = torch.zeros(1, dtype=torch.int32, device=x.device)
        self.cand_dev = torch.zeros(1, dtype=torch.int64, device=x.device)
        # [B, 2] fp32 {w, 1 + w} per image, written before every replay like cand_dev (its_ddpm_step_x0_w)
        self.w_img = torch.zeros(x.shape[0], 2, dtype=torch.float32, device=x.device) if per_image_w else None
        self.graph: Optional[torch.cuda.CUDAGraph] = None
        self.graph_key = None            # (seed or None, w) baked into the graph; w is None with per-image weights


class SamplerBase(nn.Module):
    guided = False

    def _init_schedule(self, model, beta_1, beta_T, T):
        self.model = model
        self.T = T
        # fp32 linspace upcast to double, then fp64 throughout (Diffusion.py:57-65)
        self.register_buffer('betas', torch.linspace(beta_1, beta_T, T).double())
        alphas = 1. - self.betas
        alphas_bar = torch.cumprod(alphas, dim=0)
        alphas_bar_prev = F.pad(alphas_bar, [1, 0], value=1)[:T]
        self.register_buffer('coeff1', torch.sqrt(1. / alphas))
        self.register_buffer('coeff2', self.coeff1 * (1. - alphas) / torch.sqrt(1. - alphas_bar))
        self.register_buffer('posterior_var', self.betas * (1. - alphas_bar_prev) / (1. - alphas_bar))
        self.print_steps = True    # the reference prints every time step (Diffusion.py:91)
        self.use_cuda_graph = True
        self._coef_cache: Dict = {}
        self._x0_cache: Dict = {}
        self._graphs: Dict = {}
        self.graph_captures = 0     # step graphs captured: per (plan, noise shape, x0, clip), again on a new seed or w

    # ----------------------------------------------------------- public seam --
    def predict_xt_prev_mean_from_eps(self, x_t, t, eps):
        assert x_t.shape == eps.shape
        return extract(self.coeff1, t, x_t.shape) * x_t - extract(self.coeff2, t, x_t.shape) * eps

    def _variance(self, x_t, t):
        var = torch.cat([self.posterior_var[1:2], self.betas[1:]])   # "fixed large", Diffusion.py:76
        return extract(var, t, x_t.shape)

    # -------------------------------------------------------------- internals --
    def _unet(self) -> PlannedUNet:
        m = self.model
        m = getattr(m, "module", m)            # tolerate a DataParallel-style wrapper
        if not isinstance(m, PlannedUNet):
            raise TypeError("its_b200 samplers drive an its_b200 UNet (kernel plan); got %r" % type(m).__name__)
        return m

    def _coef_table(self, dev) -> torch.Tensor:
        """[T][4] fp32 {c1, c2, sigma, 0}: the per-step scalars exactly as the
        reference forms them (fp64 gather -> .float(); sigma = sqrt of the fp32
        variance, Diffusion.py:13-15,76-77,99)."""
        key = (str(dev), self.T, self.betas.data_ptr())
        tab = self._coef_cache.get(key)
        if tab is None:
            var = torch.cat([self.posterior_var[1:2], self.betas[1:]]).float().to(dev)
            # sqrt on the target device, where the reference would evaluate torch.sqrt(var)
            tab = torch.stack([self.coeff1.float().to(dev), self.coeff2.float().to(dev), torch.sqrt(var),
                               torch.zeros_like(var)], dim=1).contiguous()
            self._coef_cache = {key: tab}
        return tab

    def _x0_table(self, dev) -> torch.Tensor:
        """[T][2] fp32 {sqrt(1/abar), sqrt(1/abar - 1)}, formed in fp64 from abar = cumprod(1 - betas)."""
        key = (str(dev), self.T, self.betas.data_ptr())
        tab = self._x0_cache.get(key)
        if tab is None:
            abar = torch.cumprod(1. - self.betas.cpu(), dim=0)     # sequential fp64 product, as _init_schedule
            tab = torch.stack([torch.sqrt(1. / abar), torch.sqrt(1. / abar - 1.)], dim=1).float().to(dev).contiguous()
            self._x0_cache = {key: tab}
        return tab

    def _run(self, x: torch.Tensor, labels: Optional[torch.Tensor], *, t_start: Optional[int], t_stop: int,
             seed: Optional[int], cand_id0: int, noise: Optional[torch.Tensor], clip: bool, want_x0: bool,
             check_nan: bool, guidance=None) -> Tuple[torch.Tensor, Optional[torch.Tensor]]:
        """Steps time_step = t_start (default T-1) ... t_stop of the ancestral loop from state `x` (the x_t that step
        t_start takes) on the device.  Returns (state after step t_stop, clipped when `clip` if t_stop == 0;
        x0 prediction of step t_stop if `want_x0`, else None).  Per-step noise is keyed by (seed, candidate,
        time_step), so a trajectory cut into segments equals the uncut one.  The candidate base `cand_id0` is
        written to device memory, so one captured step graph per (plan, noise shape, x0, clip) is replayed by every
        call with the same seed and guidance weight.  `guidance` (guided sampler): one weight per image instead of
        `self.w`, on a trajectory of its own whose graph does not bake the weights in (its_ddpm_step_x0_w), so one
        capture serves every weight vector."""
        first = self.T - 1 if t_start is None else int(t_start)
        if not (0 <= first < self.T):
            raise ValueError(f"t_start={t_start} outside [0, {self.T})")
        t_stop = int(t_stop)
        if not (0 <= t_stop <= first):
            raise ValueError(f"t_stop={t_stop} outside [0, t_start={first}]")
        if guidance is not None and not self.guided:
            raise ValueError("guidance weights need the guided sampler (DiffusionFreeGuidence); this one has no "
                             "unconditional branch to mix")
        _lib.require_cuda()
        L = _lib.lib()
        if x.device.type != "cuda":
            raise RuntimeError("its_b200 samplers run on CUDA only (no CPU fallback)")
        net = self._unet()
        if net.head.weight.device != x.device:
            raise RuntimeError(f"x lives on {x.device} but the UNet on {net.head.weight.device}")
        if self.guided:
            if getattr(net, "is_conditional", False) and self.T > net.time_embedding.timembedding[0].num_embeddings:
                raise IndexError("index out of range in self")     # the net's time table is shorter than the schedule
            net.check_indices(None, labels)
        n_shape = None if noise is None else tuple(noise.shape)
        if noise is not None and n_shape != (self.T, *x.shape):
            raise ValueError("injected noise must be [T, *x.shape]; entry t is used at time_step t")
        if seed is None:
            seed = int(torch.randint(0, 2 ** 62, (1,)).item())   # follows torch.manual_seed
        B, Cc, H, W = x.shape
        per_image_w = guidance is not None
        w_pairs = guidance_pairs(guidance, B, x.device) if per_image_w else None
        with torch.cuda.device(x.device):   # every launch below goes to this device's current stream
            plan = net.plan(2 * B if self.guided else B, H, W, n_img_in=B, uniform_t=True,
                            impl=getattr(net, "impl", None))
            key = (plan, n_shape, want_x0, clip) + (("w_img",) if per_image_w else ())
            tr = self._graphs.get(key)
            if tr is None:
                live = list(net._plans.values())   # drop the graphs of plans the net has since rebuilt
                self._graphs = {k: v for k, v in self._graphs.items() if any(k[0] is p for p in live)}
                noise_buf = next((v.noise_buf for k, v in self._graphs.items() if k[:2] == (plan, n_shape)), None)
                if noise is not None and noise_buf is None:
                    noise_buf = torch.empty(n_shape, dtype=torch.float32, device=x.device)
                tr = self._graphs[key] = _Trajectory(plan, x, noise_buf, want_x0, per_image_w)
            with torch.no_grad():
                plan.x_in.copy_(x)
                plan.t_dev.fill_(first)
                tr.cand_dev.fill_(cand_id0)
                if per_image_w:
                    tr.w_img.copy_(w_pairs)
                tr.nan_flag.zero_()
                if self.guided:
                    lab = labels.reshape(-1).to(device=x.device, dtype=torch.int64)
                    plan.labels.copy_(torch.cat([lab, torch.zeros_like(lab)]))
                    plan.run_label_ops()      # label embedding -> cond_proj vectors: once per call
                if noise is not None:
                    tr.noise_buf.copy_(noise)
            coef = self._coef_table(x.device)
            x0tab = self._x0_table(x.device).data_ptr() if want_x0 else None
            x0_ptr = tr.x0_buf.data_ptr() if want_x0 else None
            eps_u = plan.eps[B:].data_ptr() if self.guided else None
            noise_ptr, stride = (tr.noise_buf.data_ptr(), B * Cc * H * W) if noise is not None else (None, 0)
            w = None if per_image_w else float(getattr(self, "w", 0.0))

            def step():
                plan.run()
                s = _lib.stream_ptr()
                if per_image_w:
                    _lib.check(L.its_ddpm_step_x0_w(plan.x_in.data_ptr(), x0_ptr, plan.eps.data_ptr(), eps_u,
                                                    noise_ptr, stride, B, Cc * H * W, coef.data_ptr(), x0tab,
                                                    plan.t_dev.data_ptr(), tr.w_img.data_ptr(), seed,
                                                    tr.cand_dev.data_ptr(), tr.nan_flag.data_ptr(), int(clip), s),
                               "its_ddpm_step_x0_w")
                else:
                    _lib.check(L.its_ddpm_step_x0(plan.x_in.data_ptr(), x0_ptr, plan.eps.data_ptr(), eps_u, noise_ptr,
                                                  stride, B, Cc * H * W, coef.data_ptr(), x0tab, plan.t_dev.data_ptr(),
                                                  w, seed, tr.cand_dev.data_ptr(), tr.nan_flag.data_ptr(), int(clip),
                                                  s), "its_ddpm_step_x0")
                _lib.check(L.its_step_advance(plan.t_dev.data_ptr(), -1, s), "its_step_advance")

            t_cur = first
            # with injected noise the Philox key is never read: keep it out of the graph key
            graph_key = (None, w) if noise is not None else (seed, w)
            if self.use_cuda_graph and tr.graph_key != graph_key and first > t_stop:
                # (re)capture: the seed and guidance weight are baked into the graph.  One eager step first: it is a
                # real step and it performs the lazy one-time kernel attribute setup outside of stream capture.
                if self.print_steps:
                    print(t_cur)
                step()
                t_cur -= 1
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    step()
                tr.graph, tr.graph_key = g, graph_key
                self.graph_captures += 1
            replay = self.use_cuda_graph and tr.graph_key == graph_key
            while t_cur >= t_stop:
                if self.print_steps:
                    print(t_cur)
                if replay:
                    tr.graph.replay()
                else:
                    step()
                t_cur -= 1
            if check_nan and int(tr.nan_flag.item()) != 0:
                raise AssertionError("nan in tensor.")
            self.last_launches_per_step = plan.n_launches + 2
            return plan.x_in.clone(), (tr.x0_buf.clone() if want_x0 else None)

    def segment(self, x: torch.Tensor, labels: Optional[torch.Tensor] = None, *, t_start: int, t_stop: int,
                seed: int, cand_id0: int = 0, noise: Optional[torch.Tensor] = None, x0: bool = False,
                check_nan: bool = True, guidance=None) -> Tuple[torch.Tensor, Optional[torch.Tensor]]:
        """Steps time_step = t_start ... t_stop of the ancestral loop from state `x` (the x_t that step t_start
        takes), as `forward(x, t_start=..., t_stop=...)` computes them, bit for bit; the state after step 0 is
        clipped.  Returns (state after step t_stop, x0 prediction of step t_stop or None).  With `x0` the last
        step also yields clip(sqrt(1/abar)*x_t - sqrt(1/abar - 1)*eps, -1, 1) from that step's (guidance-mixed)
        eps: no extra UNet evaluation.  `forward` and `segment` share the sampler's step graphs (`_run`).
        `guidance` (guided sampler only, else ValueError): a 1-D tensor or sequence of B finite weights, image i
        mixed at guidance[i] instead of `self.w`; None keeps the scalar path."""
        if not (0 <= int(t_stop) <= int(t_start) < self.T):
            raise ValueError(f"segment needs 0 <= t_stop <= t_start < T={self.T}; got t_start={t_start} t_stop={t_stop}")
        return self._run(x, labels, t_start=int(t_start), t_stop=int(t_stop), seed=int(seed), cand_id0=int(cand_id0),
                         noise=noise, clip=True, want_x0=bool(x0), check_nan=check_nan, guidance=guidance)
