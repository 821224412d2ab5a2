"""fp32-grade execution plan (`model.precision = "fp32"`).

The reference is fp32 end to end (Diffusion/Diffusion.py:74-99 over Model.py / ModelCondition.py) and north_star
states 1e-4 on the samples for an fp32 mode.  This plan evaluates the UNet with the `its_f32_*` kernels of
libits_b200 (csrc/fp32_path.cu): NHWC fp32 activations, fp32 weights, one launch per reference operation, in the
reference's own order.  It is an `engine.PlanBase`, so the network walk, the time / label chains, the buffers
(x_in / t_dev / t_idx / labels / eps) and run() / run_label_ops() are the ones of the 16-bit plan; only the layers
differ.  The samplers, the searches and the drivers use it unchanged.  It is the parity instrument and an
independent on-device cross-check of the tcgen05 plan — CUDA-core arithmetic, roughly two orders of magnitude
slower than the 16-bit plan.
"""
from __future__ import annotations

from typing import List

import torch

from .engine import PlanBase, _ptr

F32 = torch.float32


class UNetPlanF32(PlanBase):
    """Launch plan of one fp32 UNet evaluation for n_img images of H x W (`impl` is ignored)."""

    ACT_DTYPE = F32

    def _pack(self, w: torch.Tensor, transposed: bool = False) -> torch.Tensor:
        """OIHW (or ConvTranspose2d's [Cin][Cout][k][k]) -> [k*k][Cin][CoutP] fp32, CoutP = Cout rounded up to 4."""
        w = w.detach().float()
        w = w.permute(2, 3, 0, 1) if transposed else w.permute(2, 3, 1, 0)     # [ky][kx][Cin][Cout]
        k, _, cin, cout = w.shape
        coutp = (cout + 3) // 4 * 4
        out = torch.zeros(k * k, cin, coutp, dtype=F32, device=w.device)
        out[:, :, :cout] = w.reshape(k * k, cin, cout)
        return self._hold(out)

    def conv(self, xs: List[torch.Tensor], weight, bias, *, stride=1, mode=0, vec=None, vec_off=0, vec2=None,
             vec2_off=0, res=None, out=None, out_nchw=False, transposed=False) -> torch.Tensor:
        """nn.Conv2d / up-sampled conv / ConvTranspose2d over the channel concatenation of xs (one or two tensors)."""
        x0 = xs[0]
        x1 = xs[1] if len(xs) > 1 else None
        B, Hin, Win, C0 = x0.shape
        C1 = x1.shape[-1] if x1 is not None else 0
        k = weight.shape[-1]
        cout = weight.shape[1] if transposed else weight.shape[0]
        Hout, Wout = (Hin // stride, Win // stride) if mode == 0 else (2 * Hin, 2 * Win)
        if out is None:
            out = self._new((B, Hout, Wout, cout))
        wt = self._pack(weight, transposed)
        b = self._hold(bias) if bias is not None else None

        def vptr(v, off):
            if v is None:
                return None, 0
            return v.data_ptr() + 4 * off, (0 if v.shape[0] == 1 else v.shape[1])
        vp, vs = vptr(vec, vec_off)
        vp2, vs2 = vptr(vec2, vec2_off)
        self._op(self.L.its_f32_conv2d, out.data_ptr(), x0.data_ptr(), C0, _ptr(x1), C1, wt.data_ptr(), _ptr(b),
                 vp, vs, vp2, vs2, _ptr(res), B, Hin, Win, cout, k, stride, mode, int(out_nchw),
                 flops=2 * B * Hout * Wout * cout * (C0 + C1) * k * k // (4 if mode == 2 else 1), kind="f32_conv2d")
        return out

    def group_norm(self, xs: List[torch.Tensor], gn, silu: bool) -> torch.Tensor:
        x0 = xs[0]
        x1 = xs[1] if len(xs) > 1 else None
        B, H, W, C0 = x0.shape
        C1 = x1.shape[-1] if x1 is not None else 0
        out = self._new((B, H, W, C0 + C1))
        self._op(self.L.its_f32_group_norm, out.data_ptr(), x0.data_ptr(), C0, _ptr(x1), C1,
                 self._hold(gn.weight).data_ptr(), self._hold(gn.bias).data_ptr(), B, H * W, gn.num_groups,
                 float(gn.eps), int(silu), kind="f32_group_norm")
        return out

    # ----------------------------------------------------------------- blocks --
    def _res_block(self, rb, xs: List[torch.Tensor], off: int, next_gn=None) -> torch.Tensor:
        """Model.py:167-209 / ModelCondition.py:121-161."""
        a1 = self.group_norm(xs, rb.block1[0], True)
        h = self.conv([a1], rb.block1[2].weight, rb.block1[2].bias, vec=self.tproj, vec_off=off, vec2=self.cproj,
                      vec2_off=off)
        a2 = self.group_norm([h], rb.block2[0], True)
        conv2 = rb.block2[3]
        if isinstance(rb.shortcut, torch.nn.Identity):
            if len(xs) != 1:
                raise RuntimeError("identity shortcut over a concatenated input is not supported")
            h = self.conv([a2], conv2.weight, conv2.bias, res=xs[0])
        else:
            h = self.conv([a2], conv2.weight, conv2.bias)
            h = self.conv(xs, rb.shortcut.weight, rb.shortcut.bias, res=h)          # h + shortcut(x)
        if not isinstance(rb.attn, torch.nn.Identity):
            h = self._attn_block(rb.attn, h)
        return h

    def _attn_block(self, at, x: torch.Tensor) -> torch.Tensor:
        """Model.py:129-164."""
        B, H, W, Cc = x.shape
        a = self.group_norm([x], at.group_norm, False)
        wqkv = torch.cat([at.proj_q.weight, at.proj_k.weight, at.proj_v.weight], 0)
        bqkv = torch.cat([at.proj_q.bias, at.proj_k.bias, at.proj_v.bias], 0)
        qkv = self.conv([a], wqkv, bqkv)
        o = self._new((B, H, W, Cc))
        self._op(self.L.its_f32_attention, o.data_ptr(), qkv.data_ptr(), B, H * W, Cc, float(int(Cc) ** (-0.5)),
                 flops=4 * B * H * W * H * W * Cc, kind="f32_attention")
        return self.conv([o], at.proj.weight, at.proj.bias, res=x)

    def _down(self, ds, x: torch.Tensor, next_gn=None) -> torch.Tensor:
        if hasattr(ds, "main"):                                       # Model.py:96-108
            return self.conv([x], ds.main.weight, ds.main.bias, stride=2)
        t = self.conv([x], ds.c1.weight, ds.c1.bias, stride=2)       # ModelCondition.py:65-73: c1(x) + c2(x)
        return self.conv([x], ds.c2.weight, ds.c2.bias, stride=2, res=t)

    def _up(self, us, x: torch.Tensor) -> torch.Tensor:
        if hasattr(us, "main"):                                       # Model.py:111-126
            return self.conv([x], us.main.weight, us.main.bias, mode=1)
        t = self.conv([x], us.t.weight, us.t.bias, stride=2, mode=2, transposed=True)   # ModelCondition.py:76-86
        return self.conv([t], us.c.weight, us.c.bias)

    def head_conv(self, weight, bias, x_in: torch.Tensor, B: int, H: int, W: int, next_gn=None) -> torch.Tensor:
        """Model.py:269 on the NCHW fp32 sampler state (broadcast over n_img / n_img_in)."""
        x = self._new((B, H, W, 3))
        self._op(self.L.its_f32_nchw_to_nhwc, x.data_ptr(), x_in.data_ptr(), B, x_in.shape[0], 3, H, W, kind="layout")
        return self.conv([x], weight, bias)

    def _tail_conv(self, conv, a: torch.Tensor) -> None:
        self.conv([a], conv.weight, conv.bias, out=self.eps, out_nchw=True)     # Model.py:257-262
