"""FLUX.1-style MM-DiT in plain PyTorch (random-init architecture definition).

ComfyUI / diffusers are not installed in this image and there is no network for
checkpoints, so the architecture of the public FLUX.1 model is defined here with
ComfyUI-compatible attribute names (``params``, ``double_blocks``,
``single_blocks``, ``img_in`` ...) so that (a) the *reference's* cloning and
pipeline logic (/root/reference/any_device_parallel.py:284-350, 1156) works on it
unmodified, (b) it is the fp32/bf16 numerics oracle for the hand-written sm_100a
executor in ``exec/flux_exec.py``, and (c) the bench's reference arm has a stock
torch model to wrap.  Only stock torch ops are used here (``nn.Linear``,
``F.scaled_dot_product_attention``, ``F.layer_norm``).

Forward contract (what ComfyUI's sampler calls):
``model(x[B,16,H,W], timesteps[B], context=ctx[B,L,4096], y=vec[B,768], guidance=g[B])``
returns the velocity prediction ``[B,16,H,W]``.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import List, Optional

import torch
import torch.nn as nn
import torch.nn.functional as F


@dataclass
class FluxParams:
    in_channels: int = 64
    out_channels: int = 64
    vec_in_dim: int = 768
    context_in_dim: int = 4096
    hidden_size: int = 3072
    mlp_ratio: float = 4.0
    num_heads: int = 24
    depth: int = 19
    depth_single_blocks: int = 38
    axes_dim: List[int] = field(default_factory=lambda: [16, 56, 56])
    theta: int = 10_000
    patch_size: int = 2
    qkv_bias: bool = True
    guidance_embed: bool = True


def flux_dev_params() -> FluxParams:
    return FluxParams()


def flux_tiny_params(hidden: int = 256, heads: int = 2, depth: int = 2, depth_single: int = 2) -> FluxParams:
    """head_dim stays 128 (what the sm_100a kernels are specialised for)."""
    return FluxParams(in_channels=64, out_channels=64, vec_in_dim=64, context_in_dim=128, hidden_size=hidden,
                      mlp_ratio=4.0, num_heads=heads, depth=depth, depth_single_blocks=depth_single,
                      axes_dim=[16, 56, 56], theta=10_000, patch_size=2, qkv_bias=True, guidance_embed=True)


# ------------------------------------------------------------------------- pieces

def timestep_embedding(t: torch.Tensor, dim: int, max_period: int = 10000, time_factor: float = 1000.0):
    t = time_factor * t.float()
    half = dim // 2
    freqs = torch.exp(-math.log(max_period) * torch.arange(half, dtype=torch.float32, device=t.device) / half)
    args = t[:, None] * freqs[None]
    emb = torch.cat([torch.cos(args), torch.sin(args)], dim=-1)
    if dim % 2:
        emb = torch.cat([emb, torch.zeros_like(emb[:, :1])], dim=-1)
    return emb


def rope(pos: torch.Tensor, dim: int, theta: int) -> torch.Tensor:
    scale = torch.arange(0, dim, 2, dtype=torch.float64, device=pos.device) / dim
    omega = 1.0 / (theta ** scale)
    out = pos.to(torch.float64)[..., None] * omega
    out = torch.stack([torch.cos(out), -torch.sin(out), torch.sin(out), torch.cos(out)], dim=-1)
    return out.reshape(*out.shape[:-1], 2, 2).float()


def apply_rope(xq: torch.Tensor, xk: torch.Tensor, freqs_cis: torch.Tensor):
    xq_ = xq.float().reshape(*xq.shape[:-1], -1, 1, 2)
    xk_ = xk.float().reshape(*xk.shape[:-1], -1, 1, 2)
    xq_out = freqs_cis[..., 0] * xq_[..., 0] + freqs_cis[..., 1] * xq_[..., 1]
    xk_out = freqs_cis[..., 0] * xk_[..., 0] + freqs_cis[..., 1] * xk_[..., 1]
    return xq_out.reshape(*xq.shape).type_as(xq), xk_out.reshape(*xk.shape).type_as(xk)


def attention(q, k, v, pe):
    q, k = apply_rope(q, k, pe)
    x = F.scaled_dot_product_attention(q, k, v)
    b, h, l, d = x.shape
    return x.transpose(1, 2).reshape(b, l, h * d)


class EmbedND(nn.Module):
    def __init__(self, dim: int, theta: int, axes_dim: List[int]):
        super().__init__()
        self.dim, self.theta, self.axes_dim = dim, theta, list(axes_dim)

    def forward(self, ids: torch.Tensor) -> torch.Tensor:
        emb = torch.cat([rope(ids[..., i], self.axes_dim[i], self.theta) for i in range(ids.shape[-1])], dim=-3)
        return emb.unsqueeze(1)


def position_ids(b: int, hh: int, ww: int, txt_len: int, device) -> torch.Tensor:
    """[b, txt_len + hh*ww, 3] RoPE positions: text tokens at (0, 0, 0), image token (r, c) at (0, r, c)."""
    img_ids = torch.zeros(hh, ww, 3, device=device, dtype=torch.float32)
    img_ids[..., 1] = torch.arange(hh, device=device, dtype=torch.float32)[:, None]
    img_ids[..., 2] = torch.arange(ww, device=device, dtype=torch.float32)[None, :]
    img_ids = img_ids.reshape(1, hh * ww, 3).expand(b, -1, -1)
    txt_ids = torch.zeros(b, txt_len, 3, device=device, dtype=torch.float32)
    return torch.cat((txt_ids, img_ids), dim=1)


class MLPEmbedder(nn.Module):
    def __init__(self, in_dim: int, hidden_dim: int):
        super().__init__()
        self.in_layer = nn.Linear(in_dim, hidden_dim)
        self.silu = nn.SiLU()
        self.out_layer = nn.Linear(hidden_dim, hidden_dim)

    def forward(self, x):
        return self.out_layer(self.silu(self.in_layer(x)))


class RMSNorm(nn.Module):
    def __init__(self, dim: int):
        super().__init__()
        self.scale = nn.Parameter(torch.ones(dim))

    def forward(self, x):
        dt = x.dtype
        x = x.float()
        rrms = torch.rsqrt(torch.mean(x * x, dim=-1, keepdim=True) + 1e-6)
        return (x * rrms).to(dt) * self.scale.to(dt)


class QKNorm(nn.Module):
    def __init__(self, dim: int):
        super().__init__()
        self.query_norm = RMSNorm(dim)
        self.key_norm = RMSNorm(dim)

    def forward(self, q, k, v):
        return self.query_norm(q).to(v), self.key_norm(k).to(v)


class SelfAttention(nn.Module):
    def __init__(self, dim: int, num_heads: int, qkv_bias: bool):
        super().__init__()
        self.num_heads = num_heads
        self.qkv = nn.Linear(dim, dim * 3, bias=qkv_bias)
        self.norm = QKNorm(dim // num_heads)
        self.proj = nn.Linear(dim, dim)


class Modulation(nn.Module):
    def __init__(self, dim: int, double: bool):
        super().__init__()
        self.is_double = double
        self.multiplier = 6 if double else 3
        self.lin = nn.Linear(dim, self.multiplier * dim)

    def forward(self, vec):
        out = self.lin(F.silu(vec))[:, None, :].chunk(self.multiplier, dim=-1)
        return out[:3], (out[3:] if self.is_double else None)


def _split_heads(qkv: torch.Tensor, heads: int):
    b, l, _ = qkv.shape
    qkv = qkv.view(b, l, 3, heads, -1).permute(2, 0, 3, 1, 4)
    return qkv[0], qkv[1], qkv[2]


class DoubleStreamBlock(nn.Module):
    def __init__(self, hidden_size: int, num_heads: int, mlp_ratio: float, qkv_bias: bool):
        super().__init__()
        mlp_hidden = int(hidden_size * mlp_ratio)
        self.num_heads, self.hidden_size = num_heads, hidden_size
        self.img_mod = Modulation(hidden_size, True)
        self.img_norm1 = nn.LayerNorm(hidden_size, elementwise_affine=False, eps=1e-6)
        self.img_attn = SelfAttention(hidden_size, num_heads, qkv_bias)
        self.img_norm2 = nn.LayerNorm(hidden_size, elementwise_affine=False, eps=1e-6)
        self.img_mlp = nn.Sequential(nn.Linear(hidden_size, mlp_hidden), nn.GELU(approximate="tanh"),
                                     nn.Linear(mlp_hidden, hidden_size))
        self.txt_mod = Modulation(hidden_size, True)
        self.txt_norm1 = nn.LayerNorm(hidden_size, elementwise_affine=False, eps=1e-6)
        self.txt_attn = SelfAttention(hidden_size, num_heads, qkv_bias)
        self.txt_norm2 = nn.LayerNorm(hidden_size, elementwise_affine=False, eps=1e-6)
        self.txt_mlp = nn.Sequential(nn.Linear(hidden_size, mlp_hidden), nn.GELU(approximate="tanh"),
                                     nn.Linear(mlp_hidden, hidden_size))

    def forward(self, img, txt, vec, pe):
        (i_sh1, i_sc1, i_g1), (i_sh2, i_sc2, i_g2) = self.img_mod(vec)
        (t_sh1, t_sc1, t_g1), (t_sh2, t_sc2, t_g2) = self.txt_mod(vec)
        im = (1 + i_sc1) * self.img_norm1(img) + i_sh1
        iq, ik, iv = _split_heads(self.img_attn.qkv(im), self.num_heads)
        iq, ik = self.img_attn.norm(iq, ik, iv)
        tm = (1 + t_sc1) * self.txt_norm1(txt) + t_sh1
        tq, tk, tv = _split_heads(self.txt_attn.qkv(tm), self.num_heads)
        tq, tk = self.txt_attn.norm(tq, tk, tv)
        attn = attention(torch.cat((tq, iq), 2), torch.cat((tk, ik), 2), torch.cat((tv, iv), 2), pe)
        t_attn, i_attn = attn[:, :txt.shape[1]], attn[:, txt.shape[1]:]
        img = img + i_g1 * self.img_attn.proj(i_attn)
        img = img + i_g2 * self.img_mlp((1 + i_sc2) * self.img_norm2(img) + i_sh2)
        txt = txt + t_g1 * self.txt_attn.proj(t_attn)
        txt = txt + t_g2 * self.txt_mlp((1 + t_sc2) * self.txt_norm2(txt) + t_sh2)
        return img, txt


class SingleStreamBlock(nn.Module):
    def __init__(self, hidden_size: int, num_heads: int, mlp_ratio: float = 4.0):
        super().__init__()
        self.hidden_size, self.num_heads = hidden_size, num_heads
        self.mlp_hidden_dim = int(hidden_size * mlp_ratio)
        self.linear1 = nn.Linear(hidden_size, hidden_size * 3 + self.mlp_hidden_dim)
        self.linear2 = nn.Linear(hidden_size + self.mlp_hidden_dim, hidden_size)
        self.norm = QKNorm(hidden_size // num_heads)
        self.pre_norm = nn.LayerNorm(hidden_size, elementwise_affine=False, eps=1e-6)
        self.mlp_act = nn.GELU(approximate="tanh")
        self.modulation = Modulation(hidden_size, False)

    def forward(self, x, vec, pe):
        (shift, scale, gate), _ = self.modulation(vec)
        xm = (1 + scale) * self.pre_norm(x) + shift
        qkv, mlp = torch.split(self.linear1(xm), [3 * self.hidden_size, self.mlp_hidden_dim], dim=-1)
        q, k, v = _split_heads(qkv, self.num_heads)
        q, k = self.norm(q, k, v)
        attn = attention(q, k, v, pe)
        out = self.linear2(torch.cat((attn, self.mlp_act(mlp)), 2))
        return x + gate * out


class LastLayer(nn.Module):
    def __init__(self, hidden_size: int, patch_size: int, out_channels: int):
        super().__init__()
        self.norm_final = nn.LayerNorm(hidden_size, elementwise_affine=False, eps=1e-6)
        self.linear = nn.Linear(hidden_size, patch_size * patch_size * out_channels)
        self.adaLN_modulation = nn.Sequential(nn.SiLU(), nn.Linear(hidden_size, 2 * hidden_size))

    def forward(self, x, vec):
        shift, scale = self.adaLN_modulation(vec).chunk(2, dim=1)
        x = (1 + scale[:, None, :]) * self.norm_final(x) + shift[:, None, :]
        return self.linear(x)


class Flux(nn.Module):
    """Takes either a ``FluxParams`` or the same fields as keyword arguments (the
    reference's rebuild-from-config path calls ``cls(**config)``, ADP:613-634)."""

    pa_family = "flux"

    def __init__(self, params: Optional[FluxParams] = None, dtype: Optional[torch.dtype] = None, device=None,
                 **kw):
        super().__init__()
        if params is None:
            params = FluxParams(**{k: v for k, v in kw.items() if k in FluxParams.__dataclass_fields__})
        self.params = params
        self.dtype = dtype
        p = params
        self.patch_size = p.patch_size
        self.in_channels = p.in_channels
        self.out_channels = p.out_channels
        self.hidden_size, self.num_heads = p.hidden_size, p.num_heads
        pe_dim = p.hidden_size // p.num_heads
        if sum(p.axes_dim) != pe_dim:
            raise ValueError(f"axes_dim {p.axes_dim} must sum to head_dim {pe_dim}")
        self.pe_embedder = EmbedND(pe_dim, p.theta, p.axes_dim)
        lat_ch = p.in_channels  # already patchified: C*ph*pw
        self.img_in = nn.Linear(lat_ch, p.hidden_size)
        self.time_in = MLPEmbedder(256, p.hidden_size)
        self.vector_in = MLPEmbedder(p.vec_in_dim, p.hidden_size)
        self.guidance_in = MLPEmbedder(256, p.hidden_size) if p.guidance_embed else nn.Identity()
        self.txt_in = nn.Linear(p.context_in_dim, p.hidden_size)
        self.double_blocks = nn.ModuleList(
            [DoubleStreamBlock(p.hidden_size, p.num_heads, p.mlp_ratio, p.qkv_bias) for _ in range(p.depth)])
        self.single_blocks = nn.ModuleList(
            [SingleStreamBlock(p.hidden_size, p.num_heads, p.mlp_ratio) for _ in range(p.depth_single_blocks)])
        self.final_layer = LastLayer(p.hidden_size, 1, p.out_channels)
        if dtype is not None or device is not None:
            self.to(device=device, dtype=dtype)

    # -- helpers shared with the native executor
    def patchify(self, x: torch.Tensor) -> torch.Tensor:
        b, c, h, w = x.shape
        ps = self.patch_size
        x = x.view(b, c, h // ps, ps, w // ps, ps).permute(0, 2, 4, 1, 3, 5)
        return x.reshape(b, (h // ps) * (w // ps), c * ps * ps)

    def unpatchify(self, t: torch.Tensor, h: int, w: int) -> torch.Tensor:
        b = t.shape[0]
        ps = self.patch_size
        c = t.shape[-1] // (ps * ps)
        t = t.view(b, h // ps, w // ps, c, ps, ps).permute(0, 3, 1, 4, 2, 5)
        return t.reshape(b, c, h, w)

    def make_ids(self, b: int, h: int, w: int, txt_len: int, device) -> torch.Tensor:
        return position_ids(b, h // self.patch_size, w // self.patch_size, txt_len, device)

    def forward_orig(self, img, ids, txt, timesteps, y, guidance=None):
        img = self.img_in(img)
        vec = self.time_in(timestep_embedding(timesteps, 256).to(img.dtype))
        if self.params.guidance_embed:
            if guidance is None:
                raise ValueError("guidance-distilled model needs a guidance strength")
            vec = vec + self.guidance_in(timestep_embedding(guidance, 256).to(img.dtype))
        vec = vec + self.vector_in(y[:, :self.params.vec_in_dim])
        txt = self.txt_in(txt)
        pe = self.pe_embedder(ids)
        for blk in self.double_blocks:
            img, txt = blk(img=img, txt=txt, vec=vec, pe=pe)
        x = torch.cat((txt, img), 1)
        for blk in self.single_blocks:
            x = blk(x, vec=vec, pe=pe)
        img = x[:, txt.shape[1]:]
        return self.final_layer(img, vec)

    def forward(self, x, timesteps, context=None, y=None, guidance=None, control=None,
                transformer_options=None, **kwargs):
        b, c, h, w = x.shape
        img = self.patchify(x)
        ids = self.make_ids(b, h, w, context.shape[1], x.device)
        if y is None:
            y = torch.zeros(b, self.params.vec_in_dim, device=x.device, dtype=x.dtype)
        out = self.forward_orig(img, ids, context, timesteps, y, guidance)
        return self.unpatchify(out, h, w)


def example_inputs(params: FluxParams, batch: int, height: int = 1024, width: int = 1024, txt_len: int = 512,
                   device="cpu", dtype=torch.bfloat16, seed: int = 0):
    """Synthetic latents / conditioning of the named shape (1024x1024 -> 16x128x128)."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    c = params.in_channels // (params.patch_size ** 2)
    x = torch.randn(batch, c, height // 8, width // 8, generator=g).to(device=device, dtype=dtype)
    t = torch.rand(batch, generator=g).to(device=device, dtype=dtype)
    ctx = torch.randn(batch, txt_len, params.context_in_dim, generator=g).to(device=device, dtype=dtype)
    y = torch.randn(batch, params.vec_in_dim, generator=g).to(device=device, dtype=dtype)
    guidance = torch.full((batch,), 3.5).to(device=device, dtype=dtype)
    return dict(x=x, timesteps=t, context=ctx, y=y, guidance=guidance)
