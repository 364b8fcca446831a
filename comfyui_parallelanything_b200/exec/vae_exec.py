"""SD-style VAE decoder on hand-written sm_100a kernels (SURVEY §2.6 "VAE decode conv").

Every conv is the tcgen05 implicit GEMM (NHWC), GroupNorm(+SiLU) the fused kernel, 2x nearest upsample a
vector-copy kernel.  The single 512-wide attention of the mid block is evaluated on the tensor cores as
``S = Q K^T`` (GEMM) -> row softmax -> ``O = P V`` (GEMM against V^T, which is produced directly by a GEMM
with swapped operands, so no transpose kernel exists); V's bias is folded into the output projection.
Decode is batch-parallel: the engine splits the latent batch across GPUs exactly like a denoise step and the
final kernel stores RGB NCHW rows straight into the lead GPU's buffer.
"""
from __future__ import annotations

from typing import Optional

import torch
import torch.nn as nn

from .. import ops
from ..models import vae as vae_model
from . import bf16 as _bf
from .unet_exec import _Conv, _GN


class _VRes:
    def __init__(self, m: "vae_model.VaeResBlock", d):
        self.gn1, self.c1, self.gn2, self.c2 = _GN(m.norm1, d), _Conv(m.conv1, d), _GN(m.norm2, d), _Conv(m.conv2, d)
        self.skip = _Conv(m.nin_shortcut, d) if m.nin_shortcut is not None else None

    def __call__(self, x3, hw):
        b, (h, w) = x3.shape[0], hw
        t = self.c1(self.gn1(x3, True).view(b, h, w, -1))
        t = self.gn2(t, True)
        skip = x3 if self.skip is None else self.skip(x3.view(b, h, w, -1))
        return self.c2(t.view(b, h, w, -1), "res", residual=skip)


class _VAttn:
    def __init__(self, m: "vae_model.VaeAttnBlock", d):
        c = m.q.in_channels
        self.c = c
        self.gn = _GN(m.norm, d)
        w = lambda conv: _bf(conv.weight.reshape(conv.out_channels, conv.in_channels), d)  # noqa: E731
        self.wq, self.bq, self.wk, self.bk = w(m.q), _bf(m.q.bias, d), w(m.k), _bf(m.k.bias, d)
        self.wv = w(m.v)
        self.wp = w(m.proj_out)
        # softmax rows sum to one => P (V + 1 b_v^T) = P V + b_v, and proj(O + b_v) = proj(O) + W_p b_v + b_p
        self.bp = (m.proj_out.weight.detach().reshape(c, c).float().to(d) @ m.v.bias.detach().float().to(d)
                   + m.proj_out.bias.detach().float().to(d)).to(torch.bfloat16)

    def __call__(self, x3):
        b, l, c = x3.shape
        C = ops.require()
        e = lambda *s: torch.empty(*s, dtype=torch.bfloat16, device=x3.device)  # noqa: E731
        n = self.gn(x3, False)
        q, k = e(b, l, c), e(b, l, c)
        ops.gemm(n, self.wq, "bias", out=q, bias=self.bq)
        ops.gemm(n, self.wk, "bias", out=k, bias=self.bk)
        o = e(b, l, c)
        if l % 32:
            raise ValueError("VAE attention needs H*W to be a multiple of 32")
        for i in range(b):                                    # per-sample key/value operands
            s = e(l, l)
            ops.gemm(q[i], k[i], "bias", out=s)               # S = Q K^T
            C.softmax_rows(s, float(c) ** -0.5)
            vt = e(c, l)
            ops.gemm(self.wv, n[i], "bias", out=vt)           # V^T = W_v n^T  (bias folded into proj)
            ops.gemm(s, vt, "bias", out=o[i])                 # O = P V
        out = e(b, l, c)
        ops.gemm(o, self.wp, "res", out=out, bias=self.bp, residual=x3)
        return out


class VAEDecoderExecutor(nn.Module):
    pa_family = "vae"
    pa_native = True

    def __init__(self, model: "vae_model.VAEDecoder", device, cuda_graphs: bool = False, fp8: bool = False):
        super().__init__()
        ops.require()
        d = self.device = torch.device(device)
        self.zc = model.conv_in.in_channels
        self.zpad = (self.zc + 7) // 8 * 8
        self.conv_in = _Conv(model.conv_in, d)
        self.conv_in.w = (self.conv_in.w.float() / model.scaling_factor).to(torch.bfloat16)   # z / scaling_factor
        self.mid = [_VRes(model.mid.block_1, d), _VAttn(model.mid.attn_1, d), _VRes(model.mid.block_2, d)]
        self.up = []
        for lvl in model.up:
            self.up.append(([_VRes(b, d) for b in lvl.block], _Conv(lvl.upsample.conv, d) if lvl.upsample else None))
        self.gn_out, self.conv_out = _GN(model.norm_out, d), _Conv(model.conv_out, d)
        self.out_ch = model.conv_out.out_channels

    def parameters(self, recurse: bool = True):  # type: ignore[override]
        return iter(())

    def release(self) -> None:
        self.mid, self.up = [], []

    @torch.no_grad()
    def decode(self, z: torch.Tensor, out: Optional[torch.Tensor] = None, out_ptr: Optional[int] = None,
               out_sample_off: int = 0, z_src_ptr: Optional[int] = None) -> torch.Tensor:
        C = ops.require()
        with torch.cuda.device(self.device):
            z = z.to(device=self.device, dtype=torch.bfloat16).contiguous()
            B, _, H, W = z.shape
            zh = torch.empty(B, H, W, self.zpad, dtype=torch.bfloat16, device=self.device)
            C.nchw_to_nhwc_pad(z_src_ptr if z_src_ptr is not None else z.data_ptr(), zh, B, self.zc, H * W)
            h, hw = self.conv_in(zh), (H, W)
            h = self.mid[0](h, hw)
            h = self.mid[1](h)
            h = self.mid[2](h, hw)
            for blocks, upconv in self.up:
                for blk in blocks:
                    h = blk(h, hw)
                if upconv is not None:
                    up = torch.empty(B, 2 * hw[0], 2 * hw[1], h.shape[-1], dtype=torch.bfloat16, device=self.device)
                    C.upsample2x(h.view(B, hw[0], hw[1], -1), up)
                    hw = (2 * hw[0], 2 * hw[1])
                    h = upconv(up)
            h = self.conv_out(self.gn_out(h, True).view(B, hw[0], hw[1], -1))
            if out is None and out_ptr is None:
                out = torch.empty(B, self.out_ch, hw[0], hw[1], dtype=torch.bfloat16, device=self.device)
            C.unet_out_gather(h, None, out_ptr if out_ptr is not None else out.data_ptr(), None, B, self.out_ch, False,
                              1.0, 0, out_sample_off)
            return out

    def forward(self, z, timesteps=None, context=None, **kwargs):
        return self.decode(z)


def build_vae_executor(model: nn.Module, device, **kw) -> VAEDecoderExecutor:
    return VAEDecoderExecutor(model, device, **kw)
