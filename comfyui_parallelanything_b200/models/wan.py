"""WAN2.x-style video DiT in plain PyTorch, random init (stock torch ops only).

Shape of the public WAN 2.1/2.2 T2V transformer as ComfyUI instantiates it:
``patch_embedding`` Conv3d(1,2,2), text/time embedders, ``blocks`` of
(self-attn with full-width RMS q/k norm + 3-D RoPE, cross-attn to the text,
GELU-tanh FFN) modulated by a 6-way time projection, and a modulated head.
WAN2.2-A14B uses dim 5120 / ffn 13824 / 40 heads / 40 layers per expert.  WAN2.2-TI2V-5B (48 latent channels in and
out, WAN2.2 VAE) also takes one timestep per latent frame: ``timesteps`` [B, T_lat] modulate each frame's tokens with
that frame's vectors.

Note the block list is called ``blocks`` — the reference's pipeline planner only
looks at ``double_blocks/single_blocks/transformer_blocks/layers``
(/root/reference/any_device_parallel.py:1156), so its batch==1 mode is a no-op for
WAN; ours includes ``blocks`` (parallel/pipeline.py).
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Optional, Tuple

import torch
import torch.nn as nn
import torch.nn.functional as F

from .flux import EmbedND, apply_rope, timestep_embedding


@dataclass
class WanParams:
    in_dim: int = 16
    out_dim: int = 16
    dim: int = 5120
    ffn_dim: int = 13824
    num_heads: int = 40
    num_layers: int = 40
    text_dim: int = 4096
    text_len: int = 512
    freq_dim: int = 256
    patch_size: Tuple[int, int, int] = (1, 2, 2)
    eps: float = 1e-6
    clip_dim: int = 0               # CLIP image feature width (1280) of WAN2.1 I2V / FLF2V / Fun-InP; 0 = no image branch
    clip_pos_tokens: int = 0        # FLF2V: learned position embedding over 2 x 257 CLIP tokens (514)


def wan22_a14b_params() -> WanParams:
    return WanParams()


def wan22_i2v_a14b_params() -> WanParams:
    """WAN2.2-I2V-A14B: the T2V layer stack with a 36-channel input ([noise 16 | mask 4 | image latent 16], concatenated
    by the sampler before every call) and the 16 noise channels as output."""
    return WanParams(in_dim=36)


def wan21_i2v_14b_params() -> WanParams:
    """WAN2.1-I2V-14B (480p and 720p): the A14B layer stack, 36-channel input and a CLIP image cross-attention in every
    block (257 image tokens of width 1280)."""
    return WanParams(in_dim=36, clip_dim=1280)


def wan21_flf2v_14b_params() -> WanParams:
    """WAN2.1-FLF2V-14B (first and last frame): as I2V, with 2 x 257 CLIP tokens and their position embedding."""
    return WanParams(in_dim=36, clip_dim=1280, clip_pos_tokens=514)


def wan22_ti2v_5b_params() -> WanParams:
    """WAN2.2-TI2V-5B: 48 latent channels in and out (WAN2.2 VAE, 16x spatial and 4x temporal compression), dim 3072,
    30 layers.  In image-to-video mode it takes per-frame timesteps (``ti2v_inputs``)."""
    return WanParams(in_dim=48, out_dim=48, dim=3072, ffn_dim=14336, num_heads=24, num_layers=30, text_dim=4096,
                     freq_dim=256)


def wan_tiny_params() -> WanParams:
    return WanParams(in_dim=16, out_dim=16, dim=256, ffn_dim=512, num_heads=2, num_layers=2, text_dim=64,
                     text_len=16)


class WanRMSNorm(nn.Module):
    def __init__(self, dim: int, eps: float = 1e-6):
        super().__init__()
        self.eps = eps
        self.weight = nn.Parameter(torch.ones(dim))

    def forward(self, x):
        xf = x.float()
        return (xf * torch.rsqrt(xf.pow(2).mean(-1, keepdim=True) + self.eps)).type_as(x) * self.weight


class WanSelfAttention(nn.Module):
    def __init__(self, dim: int, num_heads: int, eps: float):
        super().__init__()
        self.dim, self.num_heads, self.head_dim = dim, num_heads, dim // num_heads
        self.q, self.k, self.v, self.o = (nn.Linear(dim, dim) for _ in range(4))
        self.norm_q, self.norm_k = WanRMSNorm(dim, eps), WanRMSNorm(dim, eps)

    def forward(self, x, freqs):
        b, s, _ = x.shape
        n, d = self.num_heads, self.head_dim
        q = self.norm_q(self.q(x)).view(b, s, n, d).transpose(1, 2)
        k = self.norm_k(self.k(x)).view(b, s, n, d).transpose(1, 2)
        v = self.v(x).view(b, s, n, d).transpose(1, 2)
        q, k = apply_rope(q, k, freqs)
        o = F.scaled_dot_product_attention(q, k, v)
        return self.o(o.transpose(1, 2).reshape(b, s, n * d))


class WanCrossAttention(WanSelfAttention):
    def forward(self, x, context):  # type: ignore[override]
        b, s, _ = x.shape
        n, d = self.num_heads, self.head_dim
        q = self.norm_q(self.q(x)).view(b, s, n, d).transpose(1, 2)
        k = self.norm_k(self.k(context)).view(b, -1, n, d).transpose(1, 2)
        v = self.v(context).view(b, -1, n, d).transpose(1, 2)
        o = F.scaled_dot_product_attention(q, k, v)
        return self.o(o.transpose(1, 2).reshape(b, s, n * d))


class WanI2VCrossAttention(WanCrossAttention):
    """Text plus CLIP image cross-attention of WAN2.1 I2V / FLF2V (ComfyUI ``comfy/ldm/wan/model.py``,
    ``WanI2VCrossAttention``): ``o(attn(q, norm_k(k(txt)), v(txt)) + attn(q, norm_k_img(k_img(img)), v_img(img)))`` with
    ``img = context[:, :context_img_len]`` and ``txt = context[:, context_img_len:]``.  ``context_img_len = None`` makes
    both slices the whole context, so the image branch then attends over the text tokens too."""

    def __init__(self, dim: int, num_heads: int, eps: float):
        super().__init__(dim, num_heads, eps)
        self.k_img, self.v_img = nn.Linear(dim, dim), nn.Linear(dim, dim)
        self.norm_k_img = WanRMSNorm(dim, eps)

    def forward(self, x, context, context_img_len=None):  # type: ignore[override]
        img = context[:, :context_img_len]
        txt = context[:, context_img_len:]
        b, s, _ = x.shape
        n, d = self.num_heads, self.head_dim
        q = self.norm_q(self.q(x)).view(b, s, n, d).transpose(1, 2)

        def attend(k, v):
            return F.scaled_dot_product_attention(q, k.view(b, -1, n, d).transpose(1, 2), v.view(b, -1, n, d).transpose(1, 2))

        o = attend(self.norm_k(self.k(txt)), self.v(txt)) + attend(self.norm_k_img(self.k_img(img)), self.v_img(img))
        return self.o(o.transpose(1, 2).reshape(b, s, n * d))


def frame_rows(v: torch.Tensor, tokens: int) -> torch.Tensor:
    """Per-frame vectors [B, T, dim] -> per-token [B, tokens, dim]: frame f's vector on each of its tokens/T tokens."""
    return v.repeat_interleave(tokens // v.shape[1], dim=1)


class WanImageProjection(nn.Module):
    """ComfyUI's ``MLPProj``: CLIP vision features [B, Li, 1280] -> [B, Li, dim] image context tokens.
    ``proj = LayerNorm, Linear, GELU (exact erf), Linear, LayerNorm`` (both norms affine); FLF2V adds ``emb_pos``
    [1, 514, 1280], applied as ``clip_fea[:, :P] + emb_pos[:, :Li]`` with ``P = emb_pos.shape[1]``."""

    def __init__(self, clip_dim: int, dim: int, pos_tokens: int = 0):
        super().__init__()
        self.proj = nn.Sequential(nn.LayerNorm(clip_dim), nn.Linear(clip_dim, clip_dim), nn.GELU(),
                                  nn.Linear(clip_dim, dim), nn.LayerNorm(dim))
        self.emb_pos = nn.Parameter(torch.randn(1, pos_tokens, clip_dim) * 0.02) if pos_tokens else None

    def forward(self, clip_fea):
        if self.emb_pos is not None:
            clip_fea = clip_fea[:, :self.emb_pos.shape[1]] + self.emb_pos[:, :clip_fea.shape[1]].to(clip_fea.dtype)
        return self.proj(clip_fea)


class WanAttentionBlock(nn.Module):
    def __init__(self, dim: int, ffn_dim: int, num_heads: int, eps: float):
        super().__init__()
        self.norm1 = nn.LayerNorm(dim, eps, elementwise_affine=False)
        self.self_attn = WanSelfAttention(dim, num_heads, eps)
        self.norm3 = nn.LayerNorm(dim, eps, elementwise_affine=True)
        self.cross_attn = WanCrossAttention(dim, num_heads, eps)
        self.norm2 = nn.LayerNorm(dim, eps, elementwise_affine=False)
        self.ffn = nn.Sequential(nn.Linear(dim, ffn_dim), nn.GELU(approximate="tanh"), nn.Linear(ffn_dim, dim))
        self.modulation = nn.Parameter(torch.randn(1, 6, dim) / dim ** 0.5)

    def forward(self, x, e, freqs, context, context_img_len=None):
        if e.dim() == 4:            # per-frame timesteps: e [B, T, 6, dim]
            e = [frame_rows(v, x.shape[1]) for v in (self.modulation.to(e.dtype).unsqueeze(0) + e).unbind(2)]
        else:
            e = (self.modulation.to(e.dtype) + e).chunk(6, dim=1)
        y = self.self_attn(self.norm1(x) * (1 + e[1]) + e[0], freqs)
        x = x + y * e[2]
        if isinstance(self.cross_attn, WanI2VCrossAttention):
            x = x + self.cross_attn(self.norm3(x), context, context_img_len)
        else:
            x = x + self.cross_attn(self.norm3(x), context)
        y = self.ffn(self.norm2(x) * (1 + e[4]) + e[3])
        return x + y * e[5]


class Head(nn.Module):
    def __init__(self, dim: int, out_dim: int, patch_size, eps: float):
        super().__init__()
        self.norm = nn.LayerNorm(dim, eps, elementwise_affine=False)
        self.head = nn.Linear(dim, out_dim * patch_size[0] * patch_size[1] * patch_size[2])
        self.modulation = nn.Parameter(torch.randn(1, 2, dim) / dim ** 0.5)

    def forward(self, x, e):
        if e.dim() == 3:            # per-frame timesteps: e [B, T, dim]
            e = (self.modulation.to(e.dtype).unsqueeze(0) + e.unsqueeze(2)).unbind(2)
            e = [frame_rows(v, x.shape[1]) for v in e]
        else:
            e = (self.modulation.to(e.dtype) + e.unsqueeze(1)).chunk(2, dim=1)
        return self.head(self.norm(x) * (1 + e[1]) + e[0])


class WanModel(nn.Module):
    pa_family = "wan"

    def __init__(self, params: Optional[WanParams] = None, dtype=None, device=None, **kw):
        super().__init__()
        if params is None:
            params = WanParams(**{k: v for k, v in kw.items() if k in WanParams.__dataclass_fields__})
        self.params = p = params
        self.dim, self.num_heads, self.patch_size = p.dim, p.num_heads, tuple(p.patch_size)
        self.freq_dim = p.freq_dim
        self.dtype = dtype
        self.patch_embedding = nn.Conv3d(p.in_dim, p.dim, kernel_size=self.patch_size, stride=self.patch_size)
        self.text_embedding = nn.Sequential(nn.Linear(p.text_dim, p.dim), nn.GELU(approximate="tanh"),
                                            nn.Linear(p.dim, p.dim))
        self.time_embedding = nn.Sequential(nn.Linear(p.freq_dim, p.dim), nn.SiLU(), nn.Linear(p.dim, p.dim))
        self.time_projection = nn.Sequential(nn.SiLU(), nn.Linear(p.dim, p.dim * 6))
        self.blocks = nn.ModuleList([WanAttentionBlock(p.dim, p.ffn_dim, p.num_heads, p.eps)
                                     for _ in range(p.num_layers)])
        self.head = Head(p.dim, p.out_dim, self.patch_size, p.eps)
        d = p.dim // p.num_heads
        self.rope_embedder = EmbedND(dim=d, theta=10000, axes_dim=[d - 4 * (d // 6), 2 * (d // 6), 2 * (d // 6)])
        self.img_emb = None
        if p.clip_dim:
            # created after every other module, so models without the image branch draw the same random numbers
            self.img_emb = WanImageProjection(p.clip_dim, p.dim, p.clip_pos_tokens)
            for blk in self.blocks:
                ca = WanI2VCrossAttention(p.dim, p.num_heads, p.eps)
                ca.load_state_dict(blk.cross_attn.state_dict(), strict=False)
                blk.cross_attn = ca
        if dtype is not None or device is not None:
            self.to(device=device, dtype=dtype)

    @staticmethod
    def make_ids(b: int, t: int, h: int, w: int, device) -> torch.Tensor:
        ids = torch.zeros(t, h, w, 3, device=device, dtype=torch.float32)
        ids[..., 0] = torch.arange(t, device=device, dtype=torch.float32)[:, None, None]
        ids[..., 1] = torch.arange(h, device=device, dtype=torch.float32)[None, :, None]
        ids[..., 2] = torch.arange(w, device=device, dtype=torch.float32)[None, None, :]
        return ids.reshape(1, t * h * w, 3).expand(b, -1, -1)

    def unpatchify(self, x: torch.Tensor, grid) -> torch.Tensor:
        b = x.shape[0]
        c = self.params.out_dim
        pt, ph, pw = self.patch_size
        t, h, w = grid
        u = x.view(b, t, h, w, pt, ph, pw, c).permute(0, 7, 1, 4, 2, 5, 3, 6)
        return u.reshape(b, c, t * pt, h * ph, w * pw)

    def forward(self, x, timesteps, context=None, clip_fea=None, transformer_options=None, **kwargs):
        # x: [B, C, T, H, W]; timesteps: [B], [B, 1] or one per latent frame [B, T] (WAN2.2 TI2V)
        x = self.patch_embedding(x)
        grid = x.shape[2:]
        x = x.flatten(2).transpose(1, 2)
        if timesteps.dim() == 2 and timesteps.shape[1] == 1:
            timesteps = timesteps[:, 0]
        if timesteps.dim() == 2:
            if timesteps.shape[1] != grid[0]:
                raise ValueError(f"per-frame timesteps {tuple(timesteps.shape)} do not match {grid[0]} latent frames")
            e = self.time_embedding(timestep_embedding(timesteps.flatten(), self.freq_dim, time_factor=1.0).to(x.dtype))
            e = e.unflatten(0, tuple(timesteps.shape))                          # [B, T, dim]
            e0 = self.time_projection(e).unflatten(2, (6, self.dim))           # [B, T, 6, dim]
        else:
            e = self.time_embedding(timestep_embedding(timesteps, self.freq_dim, time_factor=1.0).to(x.dtype))
            e0 = self.time_projection(e).unflatten(1, (6, self.dim))
        ctx = self.text_embedding(context)
        context_img_len = None
        if clip_fea is not None and self.img_emb is not None:
            ctx = torch.cat([self.img_emb(clip_fea), ctx], 1)
            context_img_len = clip_fea.shape[-2]
        freqs = self.rope_embedder(self.make_ids(x.shape[0], *grid, x.device))
        for blk in self.blocks:
            x = blk(x, e0, freqs, ctx, context_img_len)
        x = self.head(x, e)
        return self.unpatchify(x, grid)


def example_inputs(params: WanParams, batch: int, frames: int = 16, height: int = 720, width: int = 1280,
                   device="cpu", dtype=torch.bfloat16, seed: int = 0):
    """720p x 16 frames -> latent [16, 4, 90, 160] (VAE 4x temporal, 8x spatial), 14 400 tokens."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    lt = max(1, frames // 4)
    x = torch.randn(batch, params.in_dim, lt, height // 8, width // 8, generator=g).to(device=device, dtype=dtype)
    t = (torch.rand(batch, generator=g) * 1000).to(device=device, dtype=dtype)
    ctx = torch.randn(batch, params.text_len, params.text_dim, generator=g).to(device=device, dtype=dtype)
    return dict(x=x, timesteps=t, context=ctx)


def i2v_inputs(params: WanParams, batch: int, frames: int = 16, height: int = 720, width: int = 1280,
               device="cpu", dtype=torch.bfloat16, seed: int = 0):
    """Image-to-video step inputs: ``x = cat(noise, mask, image latent)`` along the channels, as ComfyUI builds it for
    WAN2.2 I2V.  The mask is ones on the first latent frame (the conditioning image) and zeros elsewhere."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    lt = max(1, frames // 4)
    hl, wl = height // 8, width // 8
    nc = params.out_dim
    mc = params.in_dim - 2 * nc
    noise = torch.randn(batch, nc, lt, hl, wl, generator=g)
    mask = torch.zeros(batch, mc, lt, hl, wl)
    mask[:, :, 0] = 1.0
    image = torch.randn(batch, nc, lt, hl, wl, generator=g)
    x = torch.cat([noise, mask, image], 1).to(device=device, dtype=dtype)
    t = (torch.rand(batch, generator=g) * 1000).to(device=device, dtype=dtype)
    ctx = torch.randn(batch, params.text_len, params.text_dim, generator=g).to(device=device, dtype=dtype)
    return dict(x=x, timesteps=t, context=ctx)


def clip_inputs(params: WanParams, batch: int, frames: int = 16, height: int = 720, width: int = 1280, device="cpu",
                dtype=torch.bfloat16, seed: int = 0, clip_tokens: Optional[int] = None):
    """``i2v_inputs`` plus ``clip_fea`` [B, Li, clip_dim]: CLIP vision features of the conditioning image (Li = 257), or of
    the first and last frame for FLF2V (Li = 514 = ``clip_pos_tokens``)."""
    out = i2v_inputs(params, batch, frames, height, width, device, dtype, seed)
    li = clip_tokens or params.clip_pos_tokens or 257
    g = torch.Generator(device="cpu").manual_seed(seed + 1)
    out["clip_fea"] = torch.randn(batch, li, params.clip_dim, generator=g).to(device=device, dtype=dtype)
    return out


def ti2v_inputs(params: WanParams, batch: int, frames: int = 121, height: int = 704, width: int = 1280, device="cpu",
                dtype=torch.bfloat16, seed: int = 0):
    """WAN2.2 TI2V image-to-video step inputs, as ComfyUI builds them for the 5B model: the WAN2.2 VAE latent
    [B, 48, (frames - 1) // 4 + 1, height / 16, width / 16] whose first frame holds the encoded start image, and one
    timestep per latent frame [B, T_lat]: 0 on the image frame, t on every other frame.  1280 x 704 x 121 frames is a
    31 x 44 x 80 latent (27 280 tokens)."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    lt = (frames - 1) // 4 + 1
    x = torch.randn(batch, params.in_dim, lt, height // 16, width // 16, generator=g)
    x[:, :, 0] = 0.5 * torch.randn(batch, params.in_dim, height // 16, width // 16, generator=g)    # "image latent"
    t = (torch.rand(batch, 1, generator=g) * 1000).expand(batch, lt).clone()
    t[:, 0] = 0.0
    ctx = torch.randn(batch, params.text_len, params.text_dim, generator=g)
    return dict(x=x.to(device=device, dtype=dtype), timesteps=t.to(device=device, dtype=dtype),
                context=ctx.to(device=device, dtype=dtype))
