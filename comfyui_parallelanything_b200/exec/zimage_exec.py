"""Z-Image / Lumina-2 "NextDiT" single-stream DiT on hand-written sm_100a kernels.

Same building blocks as the FLUX / WAN executors (tcgen05 GEMM with fused epilogues, TMEM attention) plus what this
family needs (SURVEY §2.6 "DiT attention + RoPE ... Z-Image"; the reference lists Z_IMAGE as tested,
/root/reference/README.md, and splits its ``layers`` list in pipeline mode, any_device_parallel.py:1156):

  * sandwich RMSNorms: ``rmsnorm_modulate`` is both the pre-norm (``rms(x) * w * (1 + scale)``) and the post-norm
    gated residual (``x += tanh(gate) * rms(y) * w``) - one memory pass each, no separate tanh / mul / add kernels;
  * SwiGLU: w1 and w3 are ONE GEMM over row-interleaved weights with ``silu(g) * a`` in the epilogue;
  * q/k per-head RMSNorm + 3-axis RoPE + head split in the QKV GEMM epilogue (shared with FLUX);
  * all (n_layers + n_refiner) x 4 + 1 AdaLN vectors of a step come from ONE GEMM over the concatenated weights;
  * caption path (RMSNorm + Linear + ``context_refiner`` blocks) depends only on the conditioning: computed once
    per sampling run and cached (the reference re-sends and re-computes constant conditioning every step);
  * the 2x2 patch embedding is the fused scatter kernel (peer loads + GEMM + timestep sinusoid); the head is
    LayerNorm * (1 + scale) + Linear + unpatchify (+ Euler update, + NVLink peer store) in one GEMM epilogue.
"""
from __future__ import annotations

from typing import Dict, Optional

import torch
import torch.nn as nn

from .. import ops
from . import bf16 as _bf, block_linear, conditioning_sig, quantize_block_weights, recognize
from .dit import DiTExecutor, head_gather, rope_layout
from ..models import flux as flux_model
from ..models import zimage as zimage_model


class ZImageExecutor(DiTExecutor):
    pa_family = "zimage"

    def __init__(self, model: "zimage_model.ZImageModel", device, cuda_graphs: bool = False, fp8: bool = False):
        super().__init__(model, device, cuda_graphs)
        d, p = self.device, self.params
        self.dim, self.heads = p.dim, p.n_heads
        if p.dim // p.n_heads != 128 or p.patch_size != 2 or p.in_channels != 16:
            raise ValueError("ZImageExecutor is specialised for head_dim 128, 2x2 patches, 16 latent channels")
        if p.ffn_hidden % 32 or p.dim % 8 or p.cap_feat_dim % 8:
            raise ValueError("unsupported sizes")
        W: Dict[str, Optional[torch.Tensor]] = {}
        C, ps, dim = p.in_channels, p.patch_size, p.dim
        # patch features: model order (ph, pw, c) -> scatter kernel order (c, ph, pw)
        W["img_in.w"] = _bf(model.x_embedder.weight.view(dim, ps, ps, C).permute(0, 3, 1, 2).reshape(dim, C * ps * ps), d)
        W["img_in.b"] = _bf(model.x_embedder.bias, d)
        W["cap_norm"] = _bf(model.cap_embedder[0].weight, d)
        W["cap.w"], W["cap.b"] = _bf(model.cap_embedder[1].weight, d), _bf(model.cap_embedder[1].bias, d)
        W["t0.w"], W["t0.b"] = _bf(model.t_embedder.mlp[0].weight, d), _bf(model.t_embedder.mlp[0].bias, d)
        W["t2.w"], W["t2.b"] = _bf(model.t_embedder.mlp[2].weight, d), _bf(model.t_embedder.mlp[2].bias, d)
        mod_w, mod_b = [], []
        self.mod_off: Dict[str, int] = {}

        def block(name: str, blk):
            a, f = blk.attention, blk.feed_forward
            W[name + ".qkv.w"] = _bf(a.qkv.weight, d)
            W[name + ".qs"], W[name + ".ks"] = _bf(recognize.norm_scale(a.q_norm), d), _bf(recognize.norm_scale(a.k_norm), d)
            W[name + ".out.w"] = _bf(a.out.weight, d)
            W[name + ".w13.w"] = ops.interleave_glu(_bf(f.w3.weight, d), _bf(f.w1.weight, d))     # out = w3x * silu(w1x)
            W[name + ".w2.w"] = _bf(f.w2.weight, d)
            for k_, m_ in (("n1", blk.attention_norm1), ("n2", blk.attention_norm2), ("f1", blk.ffn_norm1),
                           ("f2", blk.ffn_norm2)):
                W[f"{name}.{k_}"] = _bf(m_.weight, d)
            if getattr(blk, "modulation", hasattr(blk, "adaLN_modulation")):
                self.mod_off[name] = sum(w.shape[0] for w in mod_w)
                mod_w.append(_bf(blk.adaLN_modulation[1].weight, d))
                mod_b.append(_bf(blk.adaLN_modulation[1].bias, d))

        for i, blk in enumerate(model.context_refiner):
            block(f"cr{i}", blk)
        for i, blk in enumerate(model.noise_refiner):
            block(f"nr{i}", blk)
        for i, blk in enumerate(model.layers):
            block(f"l{i}", blk)
        self.mod_off["final"] = sum(w.shape[0] for w in mod_w)
        mod_w.append(_bf(model.final_layer.adaLN_modulation[1].weight, d))
        mod_b.append(_bf(model.final_layer.adaLN_modulation[1].bias, d))
        W["mod.w"], W["mod.b"] = torch.cat(mod_w, 0).contiguous(), torch.cat(mod_b, 0).contiguous()
        # head rows: (ph, pw, c) -> (c, ph, pw), the order the fused unpatchify epilogue writes
        fl = model.final_layer.linear
        W["final.w"] = _bf(fl.weight.view(ps, ps, C, dim).permute(2, 0, 1, 3).reshape(C * ps * ps, dim), d)
        W["final.b"] = _bf(fl.bias.view(ps, ps, C).permute(2, 0, 1).reshape(C * ps * ps), d)
        self.fp8 = bool(fp8)
        if self.fp8:
            # block GEMMs as MXFP8: 256-wide single-accumulator tiles where the epilogue needs whole heads (qkv) or
            # 64-column [a | g] groups (SwiGLU), double-buffered 224-wide tiles elsewhere
            blocks = [f"cr{i}" for i in range(len(model.context_refiner))] + \
                     [f"nr{i}" for i in range(len(model.noise_refiner))] + [f"l{i}" for i in range(len(model.layers))]
            names = [f"{b}.{n_}" for b in blocks for n_ in ("qkv", "out", "w13", "w2")]
            quantize_block_weights(W, names, lambda n_: 256 if n_.endswith((".qkv", ".w13")) else 224)
            torch.cuda.empty_cache()
        self.W = W
        self.n_cr, self.n_nr, self.n_layers = len(model.context_refiner), len(model.noise_refiner), len(model.layers)
        self.eps = p.norm_eps

    def rope(self, H: int, Wd: int, Lc: int) -> torch.Tensor:
        """fp32 [Lc + (H/2)*(W/2), 64, 2] RoPE table of the joint [caption | image] sequence."""
        ids = zimage_model.ZImageModel.make_ids(1, Lc, H // 2, Wd // 2, self.device)
        return rope_layout(flux_model.EmbedND(128, self.params.rope_theta, self.params.axes_dims)(ids))

    def _new_workspace(self, B: int, H: int, Wd: int, Lc: int) -> dict:
        d, dim, p = self.device, self.dim, self.params
        Li = (H // 2) * (Wd // 2)
        L = Lc + Li
        e = lambda *s: torch.empty(*s, dtype=torch.bfloat16, device=d)  # noqa: E731
        ws = dict(B=B, H=H, Wd=Wd, Lc=Lc, Li=Li, L=L)
        ws["X"], ws["XM"], ws["Y"], ws["ATT"] = e(B, L, dim), e(B, L, dim), e(B, L, dim), e(B, L, dim)
        ws["FF"] = e(B, L, p.ffn_hidden)
        for nm, n in (("", L), ("i", Li), ("t", Lc)):
            ws["Q" + nm], ws["K" + nm], ws["V" + nm] = (e(B, self.heads, n, 128) for _ in range(3))
        ws["CAPN"], ws["XT0"] = e(B, Lc, p.cap_feat_dim), e(B, Lc, dim)
        ws["T1"], ws["TH"] = e(B, 256), e(B, self.W["t0.w"].shape[0])
        ws["TE"], ws["STE"] = e(B, p.adaln_dim), e(B, p.adaln_dim)
        ws["MOD"] = e(B, self.W["mod.w"].shape[0])
        ws["OUT"] = e(B, p.in_channels, H, Wd)
        ws["ROPE"] = self.rope(H, Wd, Lc)
        ws["ROPE_I"] = ws["ROPE"][Lc:].contiguous()
        ws["ctx_sig"] = None
        return ws

    # ------------------------------------------------------------------ schedule
    def _block(self, ws, name: str, xs, xms, ys, att, ff, q, k, v, rope, modulated: bool) -> int:
        W, eps = self.W, self.eps
        sc_a = self._mod(ws, name, 0) if modulated else None
        g_a = self._mod(ws, name, 1) if modulated else None
        sc_m = self._mod(ws, name, 2) if modulated else None
        g_m = self._mod(ws, name, 3) if modulated else None
        n = 5
        ops.rmsnorm_modulate(xs, xms, weight=W[name + ".n1"], scale=sc_a, eps=eps)
        n += block_linear(W, xms, name + ".qkv", "qkv_rope", q=q, k=k, v=v, q_scale=W[name + ".qs"],
                          k_scale=W[name + ".ks"], rope=rope, seq_off=0, qk_eps=eps)
        ops.attention(q, k, v, out=att)
        n += block_linear(W, att, name + ".out", "bias", out=ys)
        ops.rmsnorm_modulate(ys, xs, weight=W[name + ".n2"], gate=g_a, residual=xs, eps=eps)
        ops.rmsnorm_modulate(xs, xms, weight=W[name + ".f1"], scale=sc_m, eps=eps)
        n += block_linear(W, xms, name + ".w13", "swiglu", out=ff)
        n += block_linear(W, ff, name + ".w2", "bias", out=ys)
        ops.rmsnorm_modulate(ys, xs, weight=W[name + ".f2"], gate=g_m, residual=xs, eps=eps)
        return n

    def _prepare_ctx(self, ws, ctx) -> int:
        """Caption path (RMSNorm + Linear + ``context_refiner`` blocks): a function of the conditioning only, so it
        runs EAGERLY and only when the conditioning changed - never inside the per-step CUDA graph, which reads the
        refined caption tokens from the workspace's fixed ``XT0`` buffer."""
        sig = conditioning_sig(ctx)
        if ws["ctx_sig"] == sig:
            return 0
        W, Lc, n = self.W, ws["Lc"], 2
        XM, Y, ATT, FF = ws["XM"], ws["Y"], ws["ATT"], ws["FF"]
        ops.rmsnorm_modulate(ctx, ws["CAPN"], weight=W["cap_norm"], eps=self.eps)
        xt0 = ws["XT0"]
        ops.gemm(ws["CAPN"], W["cap.w"], "bias", out=xt0, bias=W["cap.b"])
        for i in range(self.n_cr):
            n += self._block(ws, f"cr{i}", xt0, XM[:, :Lc], Y[:, :Lc], ATT[:, :Lc], FF[:, :Lc], ws["Qt"], ws["Kt"],
                             ws["Vt"], ws["ROPE"], False)
        ws["ctx_sig"] = sig
        return n

    def _run(self, ws, x_ptr: int, t, ctx, out, x_in=None, sigmas=None, out_ptr: Optional[int] = None,
             out_sample_off: int = 0, t_ptr: Optional[int] = None, x_copy=None):
        W, p, Lc = self.W, self.params, ws["Lc"]
        C = ops.require()
        n = 0
        X, XM, Y, ATT, FF = ws["X"], ws["XM"], ws["Y"], ws["ATT"], ws["FF"]
        Xt, Xi = X[:, :Lc], X[:, Lc:]
        # fused scatter: (peer) latent shard -> 2x2 patches -> x_embedder GEMM ; timestep sinusoid
        C.scatter_patch_embed(W["img_in.w"], W["img_in.b"], x_ptr, t_ptr if t_ptr is not None else t.data_ptr(), 0,
                              ws["T1"], None, x_copy, Xi, p.in_channels, ws["H"], ws["Wd"], float(p.t_scale))
        ops.gemm(ws["T1"], W["t0.w"], "silu", out=ws["TH"], bias=W["t0.b"])
        ops.gemm(ws["TH"], W["t2.w"], "bias", out=ws["TE"], bias=W["t2.b"])
        C.silu(ws["TE"], ws["STE"])
        ops.gemm(ws["STE"], W["mod.w"], "bias", out=ws["MOD"], bias=W["mod.b"])            # every AdaLN vector of the step
        n += 5
        C.copy_rows(ws["XT0"], Xt)
        n += 1
        for i in range(self.n_nr):
            n += self._block(ws, f"nr{i}", Xi, XM[:, Lc:], Y[:, Lc:], ATT[:, Lc:], FF[:, Lc:], ws["Qi"], ws["Ki"], ws["Vi"],
                             ws["ROPE_I"], True)
        for i in range(self.n_layers):
            n += self._block(ws, f"l{i}", X, XM, Y, ATT, FF, ws["Q"], ws["K"], ws["V"], ws["ROPE"], True)
        # head: LayerNorm * (1 + scale) + Linear + unpatchify (+ Euler, + peer store)
        ops.layernorm_modulate(Xi, XM[:, Lc:], scale=self._mod(ws, "final", 0), eps=1e-6)
        head_gather(XM[:, Lc:], W["final.w"], W["final.b"], p.in_channels, ws["H"], ws["Wd"], out=out, out_ptr=out_ptr,
                    out_sample_off=out_sample_off, x_in=x_in, sigmas=sigmas)
        n += 2
        self.launches_per_step = n
        return out

    @torch.no_grad()
    def forward(self, x, timesteps, context=None, num_tokens=None, attention_mask=None, transformer_options=None,
                **kwargs):
        return self._forward(x, timesteps, context)


def build_zimage_executor(model: nn.Module, device, **kw) -> ZImageExecutor:
    return ZImageExecutor(model, device, **kw)
