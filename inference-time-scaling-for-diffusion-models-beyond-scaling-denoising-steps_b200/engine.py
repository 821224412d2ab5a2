"""Execution plans: the UNet forward as a fixed list of libits_b200 kernel launches.

A plan is built once per (model, batch, resolution).  It owns
  * packed weights rebuilt from the nn.Parameters of the shell modules (which keep
    the reference's state-dict layout),
  * every activation buffer (nothing is recycled inside a step, so that a step is a
    pure function of (x, t, labels); HBM is 180 GB),
  * the launch list.  All launches go to the caller's current stream, never
    synchronise or allocate, so a whole sampler step is captured into one CUDA
    graph and replayed T times with the step index living on the device.

`PlanBase` walks the network once for every plan: input buffers, time-embedding
chain, label chain, the down / middle / up path with its skip stack, the tail
GroupNorm; it also owns the launch lists and run().  A subclass supplies the
layers: `UNetPlan` here (16-bit operands on the tcgen05 tap-GEMM, NHWC bf16 / fp16
activations, weights packed K-major [Cout][taps*Cin] with shortcut / dual-conv /
sub-pixel phases concatenated along K), `engine_f32.UNetPlanF32` (fp32 CUDA-core
kernels, the parity path).

torch is used here for device memory and streams only; all arithmetic on the hot
path is in the .so.
"""
from __future__ import annotations

import contextlib
import ctypes as C
import math
from typing import List, Optional, Sequence, Tuple

import torch

from . import _lib
from ._lib import ConvDesc

BF16 = torch.bfloat16
FP16 = torch.float16
# Operand formats.  Both operands of an MMA share one 16-bit format.  GroupNorm(+Swish) outputs are
# bounded, so they are stored as IEEE fp16 and the weight columns multiplying them are packed as
# fp16 too (3 more mantissa bits than bf16: weight rounding was the largest single error term of
# the bf16 path); raw feature maps (residual stream, skips, q/k/v) keep bf16's range, and so do the
# weight columns of the taps that read them.  ITS_FP16_GN=0 restores all-bf16 (triage).
import os as _os
FP16_GN = _os.environ.get("ITS_FP16_GN", "1") != "0"


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def pack_conv_weight(w: torch.Tensor) -> torch.Tensor:
    """OIHW -> [Cout][kh*kw*Cin], tap-major then channel (the tap-GEMM's K order)."""
    return w.detach().float().permute(0, 2, 3, 1).reshape(w.shape[0], -1)


def taps_square(k: int, src: int = 0) -> List[Tuple[int, int, int]]:
    p = k // 2
    return [(src, ky - p, kx - p) for ky in range(k) for kx in range(k)]


class PlanBase:
    """Launch plan of one UNet evaluation for n_img images of H x W: what every precision shares.

    The constructor walks the network once (_build): input buffers, time-embedding chain, label chain, the
    down / middle / up path with its skip stack, the tail GroupNorm.  The subclass emits the layers through
    conv / group_norm / head_conv / _res_block / _attn_block / _down / _up / _tail_conv and sets its knobs in
    _configure."""

    ACT_DTYPE = BF16        # activation dtype of _new

    def __init__(self, model, n_img: int, H: int, W: int, *, n_img_in: Optional[int] = None,
                 uniform_t: bool = False, impl: Optional[int] = None, device=None):
        _lib.require_cuda()
        self.L = _lib.lib()
        self.model = model
        self.cond = bool(getattr(model, "is_conditional", False))
        self.n_img, self.H, self.W = int(n_img), int(H), int(W)
        self.n_img_in = int(n_img_in or n_img)
        self.uniform_t = uniform_t
        self.dev = torch.device(device) if model is None else model.head.weight.device
        if self.dev.type != "cuda":
            raise RuntimeError("its_b200 UNet must live on a CUDA device (no CPU fallback); call .cuda()")
        self.impl_forced = impl
        self.keep: List[torch.Tensor] = []      # everything the launches point into
        self.ops: List[Tuple] = []
        self.label_ops: List[Tuple] = []         # label embedding -> cond_proj of every ResBlock
        self.op_info: List[Tuple[str, int, int]] = []   # (kind, algorithmic flops, launches) per op
        self.n_launches = self.n_label_launches = 0
        self.flops = 0                           # algorithmic 2*MAC of the GEMMs, convolutions and linears
        self.gn_bytes = 0                        # algorithmic bytes of the stand-alone 16-bit GroupNorm launches
        self._to_label_ops = False
        self.x_in = self.eps = self.t_dev = self.t_idx = self.labels = None
        self.tproj = self.cproj = None           # every ResBlock's projected time / label embedding
        # run() may run ops[:_n_time_ops] (the time chain) on a side stream, joined before ops[_join_at]
        self.fork_time_chain = False
        self._n_time_ops, self._join_at = 0, None
        self._side = self._ev_fork = self._ev_join = None
        self._configure()
        if model is not None:
            with torch.no_grad():
                self._build()

    def _configure(self) -> None:
        """Knobs and state of the subclass's layers."""

    # ------------------------------------------------------------ buffers --
    def _new(self, shape: Sequence[int], dtype=None) -> torch.Tensor:
        t = torch.empty(tuple(int(s) for s in shape), dtype=dtype or self.ACT_DTYPE, device=self.dev)
        self.keep.append(t)
        return t

    def _hold(self, t: torch.Tensor, dtype=torch.float32) -> torch.Tensor:
        t = t.detach().to(device=self.dev, dtype=dtype).contiguous()
        self.keep.append(t)
        return t

    def _op(self, fn, *args, launches: int = 1, flops: int = 0, kind: str = "other"):
        if self._to_label_ops:
            self.label_ops.append((fn, args))
            self.n_label_launches += launches
            return
        self.ops.append((fn, args))
        self.op_info.append((kind, flops, launches))
        self.n_launches += launches
        self.flops += flops

    @contextlib.contextmanager
    def _label_ops(self):
        """Launches appended inside depend on the labels only (constant over a trajectory): they go to
        label_ops, which run_label_ops() enqueues."""
        self._to_label_ops = True
        try:
            yield
        finally:
            self._to_label_ops = False

    def linear(self, x: torch.Tensor, W: torch.Tensor, b: Optional[torch.Tensor], *, silu_in=False,
               silu_out=False) -> torch.Tensor:
        rows, K = x.shape
        N = W.shape[0]
        y = self._new((rows, N), torch.float32)
        self._op(self.L.its_linear, y.data_ptr(), x.data_ptr(), W.data_ptr(), _ptr(b), rows, K, N,
                 int(silu_in), int(silu_out), 0, flops=2 * rows * K * N, kind="linear")
        return y

    def _linear_of(self, x: torch.Tensor, lin, **kw) -> torch.Tensor:
        return self.linear(x, self._hold(lin.weight), self._hold(lin.bias), **kw)

    # -------------------------------------------------------------- build --
    def _build(self):
        m, L = self.model, self.L
        B, H, W = self.n_img, self.H, self.W
        ch = m.head.out_channels
        self.x_in = self._new((self.n_img_in, 3, H, W), torch.float32)
        self.t_dev = torch.zeros(1, dtype=torch.int32, device=self.dev)
        self.t_idx = torch.zeros(B, dtype=torch.int64, device=self.dev)
        self.labels = torch.zeros(B, dtype=torch.int64, device=self.dev) if self.cond else None
        rows = 1 if self.uniform_t else B
        t_idx_ptr = None if self.uniform_t else self.t_idx.data_ptr()
        te = m.time_embedding
        emb = self._new((rows, ch), torch.float32)
        if self.cond:
            table = self._hold(te.timembedding[0].weight)
            self._op(L.its_embed_rows, emb.data_ptr(), table.data_ptr(), t_idx_ptr, self.t_dev.data_ptr(), rows,
                     ch, table.shape[0])
            lin1, lin2 = te.timembedding[1], te.timembedding[3]
        else:
            freq = self._hold(te.freq_coeffs)
            self._op(L.its_time_embed, emb.data_ptr(), t_idx_ptr, self.t_dev.data_ptr(), freq.data_ptr(), rows, ch)
            lin1, lin2 = te.timembedding[0], te.timembedding[2]
        temb = self._linear_of(self._linear_of(emb, lin1, silu_out=True), lin2)
        # every ResBlock's temb_proj (and cond_proj) as ONE linear over concatenated weights (Model.py:181-184)
        blocks = [b for b in list(m.downblocks) + list(m.middleblocks) + list(m.upblocks) if hasattr(b, "temb_proj")]
        offs, o = {}, 0
        for rb in blocks:
            offs[id(rb)] = o
            o += rb.temb_proj[1].out_features

        def proj(x, name):
            w = torch.cat([getattr(rb, name)[1].weight.detach().float() for rb in blocks], 0)
            b = torch.cat([getattr(rb, name)[1].bias.detach().float() for rb in blocks], 0)
            return self.linear(x, self._hold(w), self._hold(b), silu_in=True)
        self.tproj = proj(temb, "temb_proj")
        # The time-embedding chain (embedding -> two linears -> every temb_proj) depends on t only; the head
        # (patch gather, head GEMM, first GroupNorm) depends on x only.  run() may fork the chain onto a side
        # stream and join before the first launch that adds the projected embedding (_join_at, set by conv).
        self._n_time_ops = len(self.ops)
        if self.cond:
            # Everything from the label embedding to the per-ResBlock cond_proj vectors is a function of
            # the labels alone (ModelCondition.py:216,131-135,154).  The labels of a trajectory never
            # change, so the sampler runs these launches once per forward() instead of once per step;
            # UNet.forward() runs them on every call.
            with self._label_ops():
                ce = m.cond_embedding.condEmbedding
                ctab = self._hold(ce[0].weight)
                cemb0 = self._new((B, ch), torch.float32)
                self._op(L.its_embed_rows, cemb0.data_ptr(), ctab.data_ptr(), self.labels.data_ptr(), None, B, ch,
                         ctab.shape[0])
                cemb = self._linear_of(self._linear_of(cemb0, ce[1], silu_out=True), ce[3])
                self.cproj = proj(cemb, "cond_proj")
        # The GroupNorm -> Swish that the NEXT layer opens with, when that layer reads this layer's output alone
        # (down path, middle, tail): the producing launch may apply it in its epilogue.  Up-path ResBlocks
        # normalise the concatenation [h, skip] (their groups mix both tensors) and resampling convs read
        # the raw tensor: nothing is passed there.
        seq = list(m.downblocks) + list(m.middleblocks)

        def opens_with(layer):
            return (layer.block1[0], True) if hasattr(layer, "temb_proj") else None

        next_gn = [opens_with(layer) for layer in seq[1:]] + [None]
        h = self.head_conv(m.head.weight, m.head.bias, self.x_in, B, H, W, next_gn=opens_with(seq[0]))
        hs = [h]
        for i, layer in enumerate(seq):
            if hasattr(layer, "temb_proj"):
                h = self._res_block(layer, [h], offs[id(layer)], next_gn[i])
            else:
                h = self._down(layer, h, next_gn[i])
            if i < len(m.downblocks):
                hs.append(h)
        ups = list(m.upblocks)
        for i, layer in enumerate(ups):
            if hasattr(layer, "temb_proj"):      # torch.cat([h, hs.pop()], 1)
                tail_gn = (m.tail[0], True) if i == len(ups) - 1 else None
                h = self._res_block(layer, [h, hs.pop()], offs[id(layer)], tail_gn)
            else:
                h = self._up(layer, h)
        assert len(hs) == 0
        a = self.group_norm([h], m.tail[0], silu=True)
        self.eps = self._new((B, 3, H, W), torch.float32)
        self._tail_conv(m.tail[2], a)

    # ---------------------------------------------------------------- run --
    @staticmethod
    def _launch(ops, stream: int) -> None:
        for fn, args in ops:
            rc = fn(*args, stream)
            if rc != 0:
                _lib.check(rc, fn.__name__)

    def run_label_ops(self) -> None:
        """Enqueue the launches that depend on `self.labels` only (conditional net; no-op otherwise).
        Must run after every change of the labels and before run()."""
        self._launch(self.label_ops, _lib.stream_ptr(self.dev))

    def run(self) -> None:
        """Enqueue every launch on the current stream of the plan's device (graph-capturable).  With
        fork_time_chain, the time-embedding chain runs on a side stream next to the head of the network
        (fork / join by events, so the pair is two parallel branches of the captured step graph)."""
        s = _lib.stream_ptr(self.dev)
        n_time, join_at = self._n_time_ops, self._join_at
        if not (self.fork_time_chain and n_time > 0 and join_at is not None and join_at > n_time):
            self._launch(self.ops, s)
            return
        if self._side is None:
            self._side = torch.cuda.Stream(device=self.dev)
            self._ev_fork, self._ev_join = torch.cuda.Event(), torch.cuda.Event()
        main = torch.cuda.current_stream()
        self._ev_fork.record(main)
        self._side.wait_event(self._ev_fork)
        self._launch(self.ops[:n_time], self._side.cuda_stream)
        self._ev_join.record(self._side)
        self._launch(self.ops[n_time:join_at], s)
        main.wait_event(self._ev_join)
        self._launch(self.ops[join_at:], s)


class UNetPlan(PlanBase):
    """16-bit plan: tcgen05 tap-GEMMs (CUDA-core twins where a shape or `impl` asks for them)."""

    @classmethod
    def scratch(cls, device, n_img: int, impl: Optional[int] = None) -> "UNetPlan":
        """A plan without a model: lets tests and micro-benchmarks append single
        launches (conv / group_norm / linear) through the same descriptor builder."""
        return cls(None, n_img, 0, 0, impl=impl, device=device)

    def _configure(self) -> None:
        """Every knob of a 16-bit plan.  A scratch plan (no model) differs from a model plan on purpose:
          * gn_fusion: ITS_GN_FUSION defaults to 1 ("all": tests fuse wherever the tiling allows) and a forced
            impl keeps it; a model plan defaults to "auto" and turns it "off" whenever impl is forced;
          * schedule, fused_attention, head_on_tensor_cores, fork_time_chain: the defaults (0 / True / True /
            False), whatever ITS_SCHEDULE, ITS_FUSED_ATTENTION, ITS_HEAD_TC and ITS_FORK_TIME say;
          * res_dtype, gn_dtype: a model plan also needs a head width that is a multiple of 64, and for fp16
            residuals also FP16_GN; its model's `residual_fp16` asks for them like ITS_RESIDUAL_FP16=1."""
        m, impl, env = self.model, self.impl_forced, _os.environ.get
        scratch = m is None
        self.descs: List[ConvDesc] = []
        self.gn_partials = self.ws = self.ws_persist = None     # workspaces, grown as layers need them
        self.stats_of = {}          # raw tensor -> GroupNorm statistics its producing tap-GEMM left behind
        self.prefused, self.n_gn_fused = {}, 0      # (tensor, GroupNorm) -> normalised tensor of a fused epilogue
        self.split_k, self.fold_residual, self.sm_count = True, True, 148
        self.attn_v_mn = env("ITS_ATTN_VT", "0") != "1"
        # GroupNorm(+Swish) applied by the epilogue of the convolution that produces its input.  ITS_GN_FUSION:
        # auto = where it was measured to pay (_fusion_pays), 1 = wherever the tiling allows it, 0 = never
        # (every GroupNorm as its own its_group_norm_apply launch, the round-1 plan)
        self.gn_fusion = {"0": "off", "1": "all"}.get(env("ITS_GN_FUSION", "1" if scratch else "auto"), "auto")
        if impl is not None and not scratch:
            self.gn_fusion = "off"
        if scratch:
            self.schedule, self.fused_attention, self.head_on_tensor_cores = 0, True, True
        else:       # debugging switches (tests/parity triage): fall back to the simpler schedule of a stage
            self.schedule = int(env("ITS_SCHEDULE", "0"))
            self.fused_attention = env("ITS_FUSED_ATTENTION", "1") != "0"
            self.head_on_tensor_cores = env("ITS_HEAD_TC", "1") != "0"
            self.fork_time_chain = env("ITS_FORK_TIME", "1") != "0"
        ch64 = scratch or m.head.out_channels % 64 == 0
        # Opt-in: raw feature maps (residual stream, conv1 outputs) in IEEE fp16 instead of bf16 — 5x smaller
        # error per evaluation (DESIGN.md section 5), but the residual stream follows |x_t|: only for trained
        # checkpoints / schedules whose state stays far below fp16's 65504 (an overflow surfaces as the
        # sampler's "nan in tensor." assertion).  Model attribute `residual_fp16` or ITS_RESIDUAL_FP16=1.
        want16 = bool(getattr(m, "residual_fp16", False)) or env("ITS_RESIDUAL_FP16", "0") == "1"
        self.res_dtype = FP16 if (want16 and impl is None and (scratch or (ch64 and FP16_GN))) else BF16
        self.gn_dtype = FP16 if (FP16_GN and impl != 1 and ch64) else BF16

    # --------------------------------------------------------- primitives --
    def _impl_for(self, chans: Sequence[int], cout: int, out_nchw: bool = False) -> int:
        if self.impl_forced is not None:
            return self.impl_forced
        ok = all(c % 64 == 0 for c in chans) and (out_nchw or (cout % 8 == 0 and cout >= 16))
        return 0 if ok else 1

    @staticmethod
    def _tiles(B: int, Hm: int, Wm: int, cout: int, per_image_w: bool) -> Tuple[int, int]:
        """(M tiles, N tile width) exactly as the library tiles a tap-GEMM (csrc/conv_direct.cu)."""
        bw = min(Wm, 128)
        bh = min(Hm, 128 // bw)
        bb = 128 // (bw * bh)
        if per_image_w and bb > 1:
            bh, bb = 128 // bw, 1
        tiles_m = -(-Wm // bw) * -(-Hm // bh) * -(-B // bb)
        bn = 256 if cout % 256 == 0 else 192 if cout % 192 == 0 else 128 if cout % 128 == 0 else 64 if cout > 32 else 32
        return tiles_m, bn

    # The split-K factor changes the fp32 summation order, so it must not depend on the actual
    # batch: it is derived from the layer shape at this nominal per-GPU population.  A candidate's
    # numbers are then bit-identical whatever batch / rank evaluates it.
    DESIGN_BATCH = 64

    def _splits_for(self, B, Hm, Wm, cout, nphases, nkb_min, per_image_w) -> int:
        """Split K when a layer has too few output tiles to fill the 148 SMs (4x4 / 8x8 maps)."""
        tiles_m, bn = self._tiles(self.DESIGN_BATCH, Hm, Wm, cout, per_image_w)
        ctas = tiles_m * -(-cout // bn) * nphases
        if ctas >= 96:
            return 1
        s = min(148 // ctas, nkb_min // 4, 16)
        return max(1, s)

    @staticmethod
    def _box(Hm: int, Wm: int) -> Tuple[int, int, int]:
        bw = min(Wm, 128)
        bh = min(Hm, 128 // bw)
        return bw, bh, 128 // (bw * bh)

    def _tiles_at(self, B: int, Hm: int, Wm: int) -> int:
        bw, bh, bb = self._box(Hm, Wm)
        return -(-Wm // bw) * -(-Hm // bh) * -(-B // bb)

    # Measured cost (ns) of one 64-deep k-block of a 128-row box on the persistent schedule
    # (scripts/split_probe.py, scripts/tma_box_probe.py): the TMA unit delivers ~0.6 128-byte rows
    # per clock, so narrow N tiles are operand-rate-bound, only the 256-wide one is tensor-bound.
    _T_KB = {256: 290.0, 192: 250.0, 128: 215.0, 64: 175.0}
    _T_SPLIT2 = 5000.0      # publish + re-read of the fp32 partial through L2, flag round trip

    def _fusion_pays(self, Hm, Wm, cout, nkb) -> bool:
        """Whether applying the consumer's GroupNorm in this layer's own epilogue beats the separate
        its_group_norm_apply launch — from the layer shape only (never the batch: the two plans differ in
        rounding, and a candidate's numbers must not depend on what it is batched with).  Measured on B200
        (profiles/r02_gn_fusion_per_layer.txt): the second epilogue pass and the peer rendezvous cost 6-17 us
        per launch unless a long K loop hides them behind the next tile's MMAs, so it pays only for 32x32 / 64x64
        layers in transposed-accumulator mode (Cout = 128) with K >= 2304 (-2 .. -11 us per layer on configs A, C
        and E); never on 16x16 maps (one round of 256-wide tiles: the chain is fully exposed), on 8x8 maps only
        at 128 images per pass (a loss at 64, and the rule may not depend on the batch), break-even on 4x4."""
        bw, bh, bb = self._box(Hm, Wm)
        return bb == 1 and cout == 128 and Hm * Wm >= 1024 and nkb >= 36

    # N tiles that may split K inside the launch (ITS_SPLIT_BNS overrides, for measurements)
    _SPLIT_BNS = tuple(int(x) for x in _os.environ.get("ITS_SPLIT_BNS", "64").split(","))

    def _persist_plan(self, Hm, Wm, cout, nphases, nkb, group_width: int = 0) -> Tuple[int, int]:
        """(N tile, split-K factor) of a layer on the persistent schedule, from the layer shape at the
        design batch only (so that the fp32 summation order never depends on the actual batch).
        group_width > 0: the layer's own GroupNorm is to be fused into its epilogue, so a group must lie
        inside one N tile (its_conv_gn_sync_words); (0, 0) when no N tile allows that."""
        bw, bh, bb = self._box(Hm, Wm)
        tiles_y = -(-Hm // bh)
        tiles_m = self._tiles_at(self.DESIGN_BATCH, Hm, Wm)
        best = None
        for bn in (256, 192, 128, 64):
            if cout % bn or (group_width and bn % group_width):
                continue
            tiles = tiles_m * (cout // bn) * nphases
            two_rows = bn <= 128 and bb == 1 and tiles_y % 2 == 0
            for S in (1, 2):
                if S > 1 and (bn not in self._SPLIT_BNS or nkb < 16 or tiles * S > self.sm_count or two_rows):
                    break
                if two_rows:                # two row boxes share each weight tile (measured ~410 ns per pair)
                    rounds = -(-(tiles // 2) // self.sm_count)
                    t = rounds * nkb * 410.0
                else:
                    rounds = -(-(tiles * S) // self.sm_count)
                    t = rounds * -(-nkb // S) * self._T_KB[bn]
                if S > 1:
                    t += self._T_SPLIT2
                if best is None or t < best[0] - 1e-9:
                    best = (t, bn, S)
        if best is None:
            return 0, 0
        return best[1], best[2]

    def conv(self, srcs, phases, Hm, Wm, w, cout, *, out=None, out_scale=1, bias=None, vec=None,
             vec_off=0, vec2=None, vec2_off=0, res=None, alpha=1.0, out_fp32=False, w_batch_stride=0,
             w_pitch=None, B=None, out_shape=None, out_nchw=False, want_stats=True, out_dtype=None,
             fuse_gn=None, gn_only=False) -> torch.Tensor:
        """Append one tap-GEMM launch.  srcs: list of (tensor NHWC, C_used, c_off, stride, bcast);
        phases: list of (taps[(src,dy,dx)], w_k0, py, px).
        fuse_gn = (GroupNorm module, silu): the GroupNorm(+Swish) that the consumer of this tensor opens with is
        applied by this launch's own epilogue when the tiling allows it (its_conv_gn_sync_words); group_norm()
        then finds the normalised tensor instead of launching.  gn_only: nobody reads the raw tensor (a
        ResBlock's conv1 output feeds block2's GroupNorm only) — it is then not stored at all and the
        normalised tensor is returned in its place."""
        B = self.n_img if B is None else B
        d = ConvDesc()
        d.nsrc = len(srcs)
        for i, (t, c_used, c_off, stride, bcast) in enumerate(srcs):
            s = d.src[i]
            s.ptr, s.c_pitch, s.c_off, s.C = t.data_ptr(), t.shape[-1], c_off, c_used
            s.H, s.W, s.stride, s.bcast = t.shape[1], t.shape[2], stride, int(bcast)
            s.fp16 = int(t.dtype == FP16)
        d.nphases = len(phases)
        flops = 0
        for i, (taps, w_k0, py, px) in enumerate(phases):
            ph = d.phase[i]
            ph.ntaps, ph.w_k0, ph.py, ph.px = len(taps), w_k0, py, px
            for j, (si, dy, dx) in enumerate(taps):
                ph.src[j], ph.dy[j], ph.dx[j] = si, dy, dx
            flops += 2 * B * Hm * Wm * cout * sum(srcs[si][1] for si, _, _ in taps)
        d.B, d.Hm, d.Wm = B, Hm, Wm
        d.w, d.w_pitch, d.w_batch_stride, d.Cout = w.data_ptr(), (w_pitch or w.shape[-1]), w_batch_stride, cout
        Hout, Wout = Hm * out_scale, Wm * out_scale
        if out is None:
            out = self._new(out_shape or (B, Hout, Wout, cout), torch.float32 if out_fp32 else (out_dtype or BF16))
        d.out, d.out_fp32 = out.data_ptr(), int(out_fp32)
        d.out_fp16 = int(out.dtype == FP16) | (int(res is not None and res.dtype == FP16) << 1)
        d.Hout, d.Wout, d.out_scale, d.out_c_pitch, d.out_c_off = Hout, Wout, out_scale, out.shape[-1], 0
        d.bias = _ptr(bias)
        if vec is not None and vec is self.tproj and self._join_at is None:
            self._join_at = len(self.ops)       # first consumer of the projected time embedding
        if vec is not None:
            d.vec, d.vec_stride, d.vec_off = vec.data_ptr(), (0 if vec.shape[0] == 1 else vec.shape[1]), vec_off
        if vec2 is not None:
            d.vec2, d.vec2_stride, d.vec2_off = vec2.data_ptr(), (0 if vec2.shape[0] == 1 else vec2.shape[1]), vec2_off
        if res is not None:
            d.res, d.res_c_pitch, d.res_c_off = res.data_ptr(), res.shape[-1], 0
        d.alpha, d.bn, d.out_nchw = alpha, 0, int(out_nchw)
        d.schedule = self.schedule
        impl = self._impl_for([s[1] for s in srcs], cout, out_nchw)
        launches = 1
        nkb_min = min(sum(srcs[si][1] for si, _, _ in taps) // 64 for taps, _, _, _ in phases)
        can_fold = (res is not None and impl == 0 and self.fold_residual and self.schedule != 1
                    and len(phases) == 1 and alpha == 1.0 and not out_fp32 and not out_nchw and not w_batch_stride
                    and len(srcs) < _lib.MAX_SRC and cout % 64 == 0 and res.shape[-1] == cout
                    and (w_pitch or w.shape[-1]) == w.shape[-1] and w.dim() == 2 and w.dtype == torch.float32)
        if can_fold:
            d.res = None
        persistent = impl == 0 and self.L.its_conv_stats_parts(C.byref(d)) > 0
        bn, splits = 0, 1
        want_fuse = (fuse_gn is not None and persistent and self.gn_fusion != "off" and want_stats
                     and self.gn_dtype == FP16 and len(phases) == 1 and out_scale == 1
                     and cout % fuse_gn[0].num_groups == 0
                     and (self.gn_fusion == "all" or self._fusion_pays(Hm, Wm, cout, nkb_min)))
        if persistent and self.split_k:
            nkb_plan = nkb_min + (cout // 64 if can_fold else 0)
            bn, splits = 0, 0
            if want_fuse:
                bn, splits = self._persist_plan(Hm, Wm, cout, len(phases), nkb_plan, cout // fuse_gn[0].num_groups)
            if bn == 0:
                want_fuse = False
                bn, splits = self._persist_plan(Hm, Wm, cout, len(phases), nkb_plan)
        if persistent:
            if can_fold:
                # identity shortcut as one more K block with identity weights (exact: 1.0 * bf16 value
                # in the fp32 accumulator): the persistent schedule has no residual read in its epilogue
                k_used = sum(srcs[si][1] for si, _, _ in phases[0][0])
                w = torch.cat([w[:, :k_used].float(), torch.eye(cout, device=w.device)], 1)
                i = d.nsrc
                sN = d.src[i]
                sN.ptr, sN.c_pitch, sN.c_off, sN.C = res.data_ptr(), res.shape[-1], 0, cout
                sN.H, sN.W, sN.stride, sN.bcast = res.shape[1], res.shape[2], 1, 0
                sN.fp16 = int(res.dtype == FP16)
                d.nsrc = i + 1
                ph = d.phase[0]
                ph.src[ph.ntaps], ph.dy[ph.ntaps], ph.dx[ph.ntaps] = i, 0, 0
                ph.ntaps += 1
                d.w_pitch = w.shape[-1]
            d.bn = bn
            if splits > 1:
                tiles = self._tiles_at(B, Hm, Wm) * (cout // bn) * len(phases)
                nflag = -(-(tiles * (splits - 1)) // 64) * 64
                need = nflag + tiles * (splits - 1) * 128 * bn
                if self.ws_persist is None or self.ws_persist.numel() < need:
                    # flags at the head must start out zero; the kernel leaves them zero again
                    self.ws_persist = torch.zeros(need, dtype=torch.float32, device=self.dev)
                    self.keep.append(self.ws_persist)
                d.splits, d.ws, d.ws_elems = splits, self.ws_persist.data_ptr(), self.ws_persist.numel()
            if want_stats:
                parts = self.L.its_conv_stats_parts(C.byref(d))
                st = self._new((B, parts, cout // 4, 2), torch.float32)
                d.stats, d.stats_parts = st.data_ptr(), parts
                self.stats_of[out.data_ptr()] = (st, parts)
            if want_fuse:
                gnm, gn_silu = fuse_gn
                d.gn_groups = gnm.num_groups
                words = self.L.its_conv_gn_sync_words(C.byref(d))
                if words < 0:
                    d.gn_groups = 0
                else:
                    gn_out = self._new((B, Hout, Wout, cout), FP16)
                    gamma, beta = self._hold(gnm.weight, torch.float32), self._hold(gnm.bias, torch.float32)
                    d.gn_out, d.gn_c_pitch = gn_out.data_ptr(), cout
                    d.gn_gamma, d.gn_beta, d.gn_eps = gamma.data_ptr(), beta.data_ptr(), float(gnm.eps)
                    d.gn_silu, d.gn_only = int(gn_silu), int(bool(gn_only))
                    if words > 0:
                        # arrival counters of the tiles an image spans (monotonic: zeroed once, here)
                        sync = torch.zeros(words, dtype=torch.int32, device=self.dev)
                        self.keep.append(sync)
                        d.gn_sync = sync.data_ptr()
                    self.n_gn_fused += 1
                    if gn_only:
                        # the raw tensor is never stored: drop its buffer, the map is encoded over gn_out
                        self.keep = [t for t in self.keep if t is not out]
                        self.stats_of.pop(out.data_ptr(), None)
                        d.out, d.out_c_pitch = gn_out.data_ptr(), cout
                        d.out_fp16 = (d.out_fp16 & ~1) | 1
                        out = gn_out
                    self.prefused[(out.data_ptr(), id(gnm))] = (gn_out, bool(gn_silu))
        else:
            if res is not None:
                d.res = res.data_ptr()
            d.schedule = 1 if impl == 0 else d.schedule
            if impl == 0 and not out_nchw and self.split_k:
                splits = splits if splits > 1 else self._splits_for(B, Hm, Wm, cout, len(phases), nkb_min, bool(w_batch_stride))
                if splits > 1:
                    need = len(phases) * splits * B * Hm * Wm * cout
                    if self.ws is None or self.ws.numel() < need:
                        self.ws = self._new((need,), torch.float32)
                    d.splits, d.ws, d.ws_elems = splits, self.ws.data_ptr(), self.ws.numel()
                    launches = 2
        if w.dtype == torch.float32:
            # real weights: pack every tap's columns in the 16-bit format of the source it multiplies
            w16 = torch.empty(w.shape, dtype=torch.int16, device=self.dev)
            wf = w.to(self.dev)
            for f in range(d.nphases):
                k = d.phase[f].w_k0
                for t in range(d.phase[f].ntaps):
                    sc = d.src[d.phase[f].src[t]]
                    fmt = FP16 if sc.fp16 else BF16
                    w16[..., k:k + sc.C] = wf[..., k:k + sc.C].to(fmt).view(torch.int16)
                    k += sc.C
            self.keep.append(w16)
            d.w = w16.data_ptr()
        elif persistent and can_fold:
            raise RuntimeError("residual folding needs fp32 weights")
        self.descs.append(d)
        self._op(self.L.its_conv_igemm, C.byref(d), impl, flops=flops, launches=launches,
                 kind="tapgemm_sm100" if impl == 0 else "tapgemm_cudacore")
        return out

    def group_norm(self, srcs: Sequence[torch.Tensor], gn, silu: bool) -> torch.Tensor:
        if len(srcs) == 1:
            pre = self.prefused.get((srcs[0].data_ptr(), id(gn)))
            if pre is not None:       # already applied by the epilogue of the launch that produced srcs[0]
                if pre[1] != bool(silu):
                    raise RuntimeError("fused GroupNorm was built with a different activation")
                return pre[0]
        x0 = srcs[0]
        x1 = srcs[1] if len(srcs) > 1 else None
        B, H, W, C0 = x0.shape
        C1 = x1.shape[-1] if x1 is not None else 0
        Ct = C0 + C1
        out = self._new((B, H, W, Ct), self.gn_dtype)
        f16 = int(self.gn_dtype == FP16)
        HW = H * W
        st = [self.stats_of.get(t.data_ptr()) for t in srcs]
        if all(x is not None for x in st) and (Ct // gn.num_groups) % 4 == 0:
            # statistics were left behind by the producing tap-GEMMs: one streaming apply pass
            gamma, beta = self._hold(gn.weight, torch.float32), self._hold(gn.bias, torch.float32)
            s0, p0 = st[0]
            s1, p1 = st[1] if x1 is not None else (None, 0)
            fmt = f16 | (int(x0.dtype == FP16) << 1) | (int(x1 is not None and x1.dtype == FP16) << 2)
            self._op(self.L.its_group_norm_apply, out.data_ptr(), x0.data_ptr(), C0, s0.data_ptr(), p0, _ptr(x1), C1,
                     _ptr(s1), p1, gamma.data_ptr(), beta.data_ptr(), B, HW, gn.num_groups, float(gn.eps),
                     int(silu), fmt, launches=1, kind="group_norm_apply")
            self.gn_bytes += B * HW * Ct * 2 * 2
            return out
        prow = max(1, 256 // (Ct // 8))
        # the split depends on (HW, C) only, never on the batch: a candidate's numbers are then
        # bit-identical whatever batch / rank it is evaluated in (fixed summation order)
        chunks = max(1, min(HW // prow, 8))
        chunks = 1 << (chunks.bit_length() - 1)      # cluster of 1/2/4/8 CTAs per image
        need = B * chunks * 32 * 2
        if self.gn_partials is None or self.gn_partials.numel() < need:
            self.gn_partials = self._new((need,), torch.float32)
        gamma, beta = self._hold(gn.weight, torch.float32), self._hold(gn.bias, torch.float32)
        self._op(self.L.its_group_norm, out.data_ptr(), x0.data_ptr(), C0, _ptr(x1), C1, gamma.data_ptr(),
                 beta.data_ptr(), B, HW, gn.num_groups, float(gn.eps), int(silu),
                 self.gn_partials.data_ptr(), chunks,
                 f16 | (int(x0.dtype == FP16) << 1) | (int(x1 is not None and x1.dtype == FP16) << 2),
                 launches=1, kind="group_norm")
        self.gn_bytes += B * HW * Ct * 2 * 2     # one read + one write, 16-bit
        return out

    # ------------------------------------------------------------- blocks --
    def _res_block(self, rb, xs: List[torch.Tensor], proj_off: int, next_gn=None) -> torch.Tensor:
        B, H, W = xs[0].shape[:3]
        cin = sum(t.shape[-1] for t in xs)
        cout = rb.block1[2].out_channels
        a1 = self.group_norm(xs, rb.block1[0], silu=True)
        w1 = self._hold(pack_conv_weight(rb.block1[2].weight), torch.float32)
        b1 = self._hold(rb.block1[2].bias, torch.float32)
        h1 = self.conv([(a1, cin, 0, 1, False)], [(taps_square(3), 0, 0, 0)], H, W, w1, cout, bias=b1,
                       vec=self.tproj, vec_off=proj_off, vec2=self.cproj, vec2_off=proj_off, out_dtype=self.res_dtype,
                       fuse_gn=(rb.block2[0], True), gn_only=True)
        a2 = self.group_norm([h1], rb.block2[0], silu=True)
        has_attn = not isinstance(rb.attn, torch.nn.Identity)
        gn_after = (rb.attn.group_norm, False) if has_attn else next_gn   # what reads this block's conv2 output
        conv2 = rb.block2[3]
        w2 = pack_conv_weight(conv2.weight)
        b2 = conv2.bias.detach().float()
        has_sc = not isinstance(rb.shortcut, torch.nn.Identity)
        if has_sc:
            ws = rb.shortcut.weight.detach().float()[:, :, 0, 0]
            w2 = self._hold(torch.cat([w2, ws], dim=1), torch.float32)
            b2 = self._hold(b2 + rb.shortcut.bias.detach().float(), torch.float32)
            srcs = [(a2, cout, 0, 1, False)] + [(t, t.shape[-1], 0, 1, False) for t in xs]
            taps = taps_square(3) + [(1 + i, 0, 0) for i in range(len(xs))]
            h2 = self.conv(srcs, [(taps, 0, 0, 0)], H, W, w2, cout, bias=b2, out_dtype=self.res_dtype,
                           fuse_gn=gn_after)
        else:
            if len(xs) != 1:
                raise RuntimeError("identity shortcut over a concatenated input is not supported")
            w2 = self._hold(w2, torch.float32)
            b2 = self._hold(b2, torch.float32)
            h2 = self.conv([(a2, cout, 0, 1, False)], [(taps_square(3), 0, 0, 0)], H, W, w2, cout, bias=b2,
                           res=xs[0], out_dtype=self.res_dtype, fuse_gn=gn_after)
        if has_attn:
            h2 = self._attn_block(rb.attn, h2, next_gn)
        return h2

    def _attn_block(self, at, x: torch.Tensor, next_gn=None) -> torch.Tensor:
        B, H, W, Cc = x.shape
        N = H * W
        scale = float(int(Cc) ** (-0.5))
        a = self.group_norm([x], at.group_norm, silu=False)
        wq, wk, wv = (m.weight.detach().float()[:, :, 0, 0] for m in (at.proj_q, at.proj_k, at.proj_v))
        bq, bk, bv = (m.bias.detach().float() for m in (at.proj_q, at.proj_k, at.proj_v))
        one = [(0, 0, 0)]
        on_tc = self._impl_for([Cc], Cc) == 0 and self.fused_attention
        flops = 4 * B * N * N * Cc

        def project(w, b, cout):    # 1x1 projection(s) of the normalised input
            return self.conv([(a, Cc, 0, 1, False)], [(one, 0, 0, 0)], H, W, self._hold(w), cout, bias=self._hold(b),
                             want_stats=False)
        if N > 64:      # batched-GEMM formulation (tcgen05, or its CUDA-core twin when forced)
            core = (("attention_fused", self.L.its_attention_fused) if N == 256 and Cc % 64 == 0 and Cc <= 384 else
                    ("attention_flash", self.L.its_attention_flash) if N % 128 == 0 and N > 256 and Cc in (64, 128)
                    else None)
            fused = core is not None and on_tc
            if fused and self.attn_v_mn:
                # one projection launch for q|k|v; the attention core reads V as an MN-major B operand
                # straight from that tensor (no V^T projection launch)
                qk = project(torch.cat([wq, wk, wv]), torch.cat([bq, bk, torch.zeros_like(bv)]), 3 * Cc)
                vT = None
            else:
                qk = project(torch.cat([wq, wk]), torch.cat([bq, bk]), 2 * Cc)
                # V^T[b] = Wv . a[b]^T : weights are the A operand, the image is the B operand
                wv_img = self._hold(wv.reshape(1, 1, Cc, Cc), a.dtype)
                vT = self.conv([(wv_img, Cc, 0, 1, True)], [(one, 0, 0, 0)], 1, Cc, a.view(B, N, Cc), N,
                               w_batch_stride=N * Cc, out_shape=(B, 1, Cc, N), want_stats=False)
            if fused:
                # scores in TMEM, probabilities in shared memory: one launch for QK^T, softmax and PV; V's bias is
                # added after the product (the rows of softmax(S) sum to one)
                o = self._new((B, H, W, Cc))
                bvh = self._hold(bv)
                self._op(core[1], o.data_ptr(), qk.data_ptr(), _ptr(vT), bvh.data_ptr(), B, N, Cc, scale,
                         flops=flops, kind=core[0])
            else:
                # S = scale * Q K^T (fp32), per image
                k_view = qk.view(B, N, 2 * Cc)[:, :, Cc:]
                S = self.conv([(qk, Cc, 0, 1, False)], [(one, 0, 0, 0)], H, W, k_view, N, alpha=scale,
                              out_fp32=True, w_batch_stride=N * 2 * Cc, w_pitch=2 * Cc)
                P = self._new((B, H, W, N))
                self._op(self.L.its_softmax_rows, P.data_ptr(), S.data_ptr(), B * N, N, kind="softmax")
                bvh = self._hold(bv)
                o = self.conv([(P, N, 0, 1, False)], [(one, 0, 0, 0)], H, W, vT.view(B, Cc, N), Cc, bias=bvh,
                              w_batch_stride=Cc * N, want_stats=False)
        elif N in (32, 64) and Cc % 64 == 0 and Cc <= 512 and (Cc <= 256 or Cc % 128 == 0) and on_tc:
            # small maps on the tensor cores: 128 / N images per tile, block-diagonal softmax mask.  (4x4 maps
            # stay on the CUDA-core kernel: at the design batch they are only 8 tiles, a latency-bound chain
            # of 13.6 us against 8.7 us for one CTA per query; the choice depends on the shape only, never on
            # the batch, so a candidate's numbers do not depend on what it is batched with.)
            qkv = project(torch.cat([wq, wk, wv]), torch.cat([bq, bk, torch.zeros_like(bv)]), 3 * Cc)
            o = self._new((B, H, W, Cc))
            bvh = self._hold(bv)
            self._op(self.L.its_attention_group, o.data_ptr(), qkv.data_ptr(), bvh.data_ptr(), B, N, Cc, scale,
                     flops=flops, kind="attention_group")
        else:
            qkv = project(torch.cat([wq, wk, wv]), torch.cat([bq, bk, bv]), 3 * Cc)
            o = self._new((B, H, W, Cc))
            self._op(self.L.its_attention_small, o.data_ptr(), qkv.data_ptr(), B, N, Cc, scale,
                     flops=flops, kind="attention_small")
        wp, bp = self._hold(at.proj.weight.detach().float()[:, :, 0, 0]), self._hold(at.proj.bias)
        return self.conv([(o, Cc, 0, 1, False)], [(one, 0, 0, 0)], H, W, wp, Cc, bias=bp, res=x,
                         out_dtype=self.res_dtype, fuse_gn=next_gn)

    def _down(self, ds, x: torch.Tensor, next_gn=None) -> torch.Tensor:
        B, H, W, Cc = x.shape
        if hasattr(ds, "main"):       # Model.py:96-108
            w = self._hold(pack_conv_weight(ds.main.weight), torch.float32)
            b = self._hold(ds.main.bias, torch.float32)
            taps = taps_square(3)
        else:                          # ModelCondition.py:65-73: 3x3 s2 + 5x5 s2, one accumulator
            w = self._hold(torch.cat([pack_conv_weight(ds.c1.weight), pack_conv_weight(ds.c2.weight)], 1), torch.float32)
            b = self._hold(ds.c1.bias.detach().float() + ds.c2.bias.detach().float(), torch.float32)
            taps = taps_square(3) + taps_square(5)
        return self.conv([(x, Cc, 0, 2, False)], [(taps, 0, 0, 0)], H // 2, W // 2, w, Cc, bias=b, out_dtype=self.res_dtype,
                         fuse_gn=next_gn)

    def _up(self, us, x: torch.Tensor) -> torch.Tensor:
        B, H, W, Cc = x.shape
        if hasattr(us, "main"):
            # nearest x2 + 3x3 (Model.py:122-125) folded into four 2x2 sub-pixel phases
            w = us.main.weight.detach().float()
            groups = {0: [(-1, [0]), (0, [1, 2])], 1: [(0, [0, 1]), (1, [2])]}
            mats, phases, k0 = [], [], 0
            for py in (0, 1):
                for px in (0, 1):
                    taps = []
                    for dy, kys in groups[py]:
                        for dx, kxs in groups[px]:
                            mats.append(sum(w[:, :, ky, kx] for ky in kys for kx in kxs))
                            taps.append((0, dy, dx))
                    phases.append((taps, k0, py, px))
                    k0 += len(taps) * Cc
            wp = self._hold(torch.cat(mats, 1), torch.float32)
            b = self._hold(us.main.bias, torch.float32)
            return self.conv([(x, Cc, 0, 1, False)], phases, H, W, wp, Cc, out_scale=2, bias=b, out_dtype=self.res_dtype)
        # ConvTranspose2d(5, 2, 2, 1) as four phases (ModelCondition.py:80), then 3x3
        wt = us.t.weight.detach().float()  # [Cin, Cout, 5, 5]
        mats, phases, k0 = [], [], 0
        for py in (0, 1):
            kys = [0, 2, 4] if py == 0 else [1, 3]
            for px in (0, 1):
                kxs = [0, 2, 4] if px == 0 else [1, 3]
                taps = []
                for ky in kys:
                    for kx in kxs:
                        mats.append(wt[:, :, ky, kx].t())
                        taps.append((0, (py + 2 - ky) // 2, (px + 2 - kx) // 2))
                phases.append((taps, k0, py, px))
                k0 += len(taps) * Cc
        wp = self._hold(torch.cat(mats, 1), torch.float32)
        bt = self._hold(us.t.bias, torch.float32)
        y = self.conv([(x, Cc, 0, 1, False)], phases, H, W, wp, Cc, out_scale=2, bias=bt, out_dtype=self.res_dtype)
        wc = self._hold(pack_conv_weight(us.c.weight), torch.float32)
        bc = self._hold(us.c.bias, torch.float32)
        return self.conv([(y, Cc, 0, 1, False)], [(taps_square(3), 0, 0, 0)], 2 * H, 2 * W, wc, Cc, bias=bc,
                         out_dtype=self.res_dtype)

    def head_conv(self, weight, bias, x_in: torch.Tensor, B: int, H: int, W: int, next_gn=None) -> torch.Tensor:
        """Model.py:269: conv3x3(3 -> ch) of the NCHW fp32 sampler state into NHWC bf16."""
        L = self.L
        ch = weight.shape[0]
        n_img_in = x_in.shape[0]
        hb = self._hold(bias, torch.float32)
        if self._impl_for([128], ch) == 0 and self.head_on_tensor_cores:
            # patches [x_hi | x_lo | x_hi | 0] x weights [w_hi | w_hi | w_lo | 0]: fp32-grade head on
            # the persistent tap-GEMM, which also leaves the GroupNorm statistics of h behind
            patches = self._new((B, H, W, 128))
            self._op(L.its_head_patches, patches.data_ptr(), x_in.data_ptr(), B, n_img_in, H, W, 3,
                     kind="head_patches")
            w32 = weight.detach().float().reshape(ch, 27)
            w_hi = w32.to(BF16).float()
            wpk = torch.zeros(ch, 128, device=w32.device)
            wpk[:, 0:27], wpk[:, 27:54], wpk[:, 54:81] = w_hi, w_hi, w32 - w_hi
            h = self.conv([(patches, 128, 0, 1, False)], [([(0, 0, 0)], 0, 0, 0)], H, W, self._hold(wpk, BF16), ch,
                          bias=hb, B=B, out_dtype=self.res_dtype, fuse_gn=next_gn)
            self.flops -= 2 * B * H * W * ch * (128 - 27)     # algorithmic work is the 27-tap convolution
            return h
        h = self._new((B, H, W, ch))
        hw = self._hold(weight, torch.float32)
        self._op(L.its_conv_head, h.data_ptr(), x_in.data_ptr(), hw.data_ptr(), hb.data_ptr(), B,
                 n_img_in, H, W, 3, ch, flops=2 * B * H * W * ch * 27, kind="conv_head")
        return h

    def _tail_conv(self, conv, a: torch.Tensor) -> None:
        """Model.py:257-262: conv3x3(ch -> 3) of the tail GroupNorm's output into eps (NCHW fp32)."""
        B, H, W, ct = a.shape
        if self._impl_for([ct], 3, True) == 0:
            # 3-channel tail on the tensor cores: N tile of 32 (rows 3..31 of the weight box are
            # TMA zero fill), epilogue writes NCHW fp32 directly (coalesced over pixels)
            tw, tb = self._hold(pack_conv_weight(conv.weight)), self._hold(conv.bias)
            self.conv([(a, ct, 0, 1, False)], [(taps_square(3), 0, 0, 0)], H, W, tw, 3, bias=tb, out=self.eps,
                      out_fp32=True, out_nchw=True)
        else:
            tw, tb = self._hold(conv.weight), self._hold(conv.bias)
            self._op(self.L.its_conv_tail, self.eps.data_ptr(), a.data_ptr(), tw.data_ptr(), tb.data_ptr(), B, H, W,
                     ct, 3, flops=2 * B * H * W * 3 * 9 * ct, kind="conv_tail")
