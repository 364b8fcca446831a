"""Sequence-parallel (Ulysses) WAN2.x step for batch == 1 on N GPUs of one process.

Video generation is the batch-1 workload: one 720p clip is 14k - 57k tokens through 40 blocks.  The reference's batch == 1
mode (/root/reference/any_device_parallel.py:24-87, 1295-1305) walks the blocks sequentially over the devices - same
latency as one GPU.  Here, as for FLUX (``flux_sp.py``):

  * every GPU owns ``L / N`` consecutive video tokens for the linear layers (patch embedding, LayerNorm+modulate, QKV,
    o, cross-attention q / o, FFN, head), including the full-width q/k RMSNorm + 3-D RoPE (RoPE rows = the slice's
    global positions);
  * self-attention runs on ``H / N`` heads over ALL tokens: one peer-pull exchange turns [my tokens, all heads] into
    [all tokens, my heads] before it and one turns the result back after it (csrc/comm/sp_a2a.cu, device-side flag
    handshake, epochs in device memory -> the whole share of a GPU is one CUDA graph);
  * per-frame timesteps (WAN2.2 TI2V): the replicated time path embeds one timestep per latent frame, and the
    LayerNorm / gated-residual lookups use the slice's global token index, so a slice that starts mid-frame reads the
    right frame's modulation vectors;
  * text cross-attention needs no exchange: every GPU holds the (step-invariant, cached) K/V of the 512 text tokens and
    attends with its own query tokens; WAN2.1 I2V / FLF2V hold the image K/V of the CLIP tokens the same way and run the
    executor's two-source cross-attention;
  * the head GEMM's unpatchify epilogue stores each GPU's token rows straight into the lead GPU's output (NVLink).
"""
from __future__ import annotations

from typing import List, Optional

import torch

from .. import ops
from . import block_linear
from .dit import head_gather
from .sp_common import UlyssesBase, attention_variant
from .wan_exec import frame_lookup, frame_steps


def supported(executors) -> Optional[str]:
    n = len(executors)
    if n < 2:
        return "needs at least 2 GPUs"
    C = ops.require()
    if n > C.SP_MAX_RANKS:
        return f"at most {C.SP_MAX_RANKS} GPUs"
    ex0 = executors[0]
    if any(getattr(e, "pa_family", None) != "wan" or not getattr(e, "pa_native", False) for e in executors):
        return "every replica must be a native WAN executor"
    if ex0.heads % n:
        return f"{ex0.heads} heads are not divisible by {n} GPUs"
    if 2 * ex0.n_blocks + 2 > C.SP_MAX_SLOTS:
        return "too many blocks for the flag table"
    return None


def exchange_tables(g: int, n: int, Ll: int, dim: int, hpg: int, ptrs):
    """Copy descriptors (src, dst, src_pitch, dst_pitch, rows, row_bytes) GPU ``g`` pulls with, bf16 buffers:
    ``ptrs[r]`` = base addresses of rank r's QKV [Ll, 3*dim] (its tokens, all heads), QF / KF / VF [L, hpg*128] (all
    tokens, its heads), ATTF [L, hpg*128] and ATT [Ll, dim].  Pure function of the geometry (CPU-testable)."""
    qkv, att = [], []
    for r in range(n):
        for sec, name_f in enumerate(("QF", "KF", "VF")):
            # heads of g inside r's token-major [Ll, 3*dim] -> rows [r*Ll, ...) of my [L, hpg*128]
            src = ptrs[r]["QKV"] + (sec * dim + g * hpg * 128) * 2
            dst = ptrs[g][name_f] + r * Ll * hpg * 256
            qkv.append((src, dst, 3 * dim * 2, hpg * 256, Ll, hpg * 256))
        # attention output of r's heads for MY token rows -> columns [r*hpg*128, ...) of my ATT rows
        src = ptrs[r]["ATTF"] + g * Ll * hpg * 256
        dst = ptrs[g]["ATT"] + r * hpg * 256
        att.append((src, dst, hpg * 256, dim * 2, Ll, hpg * 256))
    return qkv, att


class WanUlysses(UlyssesBase):
    family = "wan"

    def __init__(self, executors: List, timeout_ms: int = 20000):
        why = supported(executors)
        if why:
            raise ValueError(f"sequence-parallel WAN unavailable: {why}")
        super().__init__(executors, timeout_ms)

    # ------------------------------------------------------------------ engine-facing protocol
    def accepts(self, x, context) -> bool:
        if x.dim() != 5 or context.dim() != 3 or x.shape[1] != self.ex[0].params.in_dim:
            return False
        T, H, Wd = x.shape[2], x.shape[3], x.shape[4]
        if H % 2 or Wd % 2:
            return False
        L = T * (H // 2) * (Wd // 2)
        # a GPU's token slice must be whole 8-row groups (TMA swizzle atoms of the head-sliced views)
        return L % (8 * self.n) == 0

    def out_shape(self, x) -> tuple:
        return self.ex[0].out_shape(tuple(x.shape))

    def _clip(self, kwargs):
        """``clip_fea`` of the step when the replicas take CLIP image conditioning, else None."""
        if not getattr(self.ex[0], "conditioning_kwargs", ()):
            return None
        c = kwargs.get("clip_fea")
        return c if isinstance(c, torch.Tensor) else None

    def slot_buffers(self, device, x, timesteps, context, kwargs) -> dict:
        st = super().slot_buffers(device, x, timesteps, context, kwargs)
        tt = frame_steps(timesteps, x.shape)
        if tt > 1:
            st["t"] = torch.empty(1, tt, dtype=torch.bfloat16, device=device)      # one timestep per latent frame
        clip = self._clip(kwargs)
        if clip is not None:
            st["clip"], st["clip_src"] = torch.empty(tuple(clip.shape), dtype=torch.bfloat16, device=device), None
        return st

    def stage(self, st: dict, timesteps, context, kwargs, cache_conditioning: bool) -> None:
        super().stage(st, timesteps, context, kwargs, cache_conditioning)
        clip = self._clip(kwargs)
        if clip is not None:
            ident = (id(clip), clip.data_ptr(), clip._version)
            if not cache_conditioning or st["clip_src"] is None or st["clip_src"][0] != ident:
                st["clip"].copy_(clip, non_blocking=True)
                st["clip_src"] = (ident, clip)

    def io_key(self, x, timesteps, context, kwargs) -> tuple:
        clip = self._clip(kwargs)
        return (super().io_key(x, timesteps, context, kwargs) + ((tuple(clip.shape),) if clip is not None else ())
                + (frame_steps(timesteps, x.shape),))

    def geometry(self, x, timesteps, context, kwargs=None) -> tuple:
        clip = self._clip(kwargs or {})
        return (x.shape[2], x.shape[3], x.shape[4], context.shape[1], clip.shape[1] if clip is not None else 0,
                frame_steps(timesteps, x.shape))

    def workspace(self, T: int, H: int, Wd: int, Lc: int, Li: int = 0, Tt: int = 1) -> list:
        """``Tt`` timesteps (1, or one per latent frame): the replicated time path and modulation tables have Tt
        rows."""
        key = (T, H, Wd, Lc, Li, Tt)
        got = self._ws.get(key)
        if got is not None:
            return got
        n, ex0 = self.n, self.ex[0]
        dim, heads = ex0.dim, ex0.heads
        L = T * (H // 2) * (Wd // 2)
        Ll, hpg = L // n, heads // n
        wss = []
        for g, ex in enumerate(self.ex):
            d = ex.device
            e = lambda *s: torch.empty(*s, dtype=torch.bfloat16, device=d)  # noqa: E731
            ws = dict(g=g, B=1, T=T, H=H, Wd=Wd, L=L, Ll=Ll, Lc=Lc, hpg=hpg)
            ws["TOK"] = e(1, L, 4 * ex.params.in_dim)
            ws["X"], ws["XM"] = e(1, Ll, dim), e(1, Ll, dim)
            ws["QKV"] = e(1, Ll, 3 * dim)                            # my tokens, all heads
            ws["QF"], ws["KF"], ws["VF"] = e(1, L, hpg * 128), e(1, L, hpg * 128), e(1, L, hpg * 128)   # all tokens, my heads
            ws["ATTF"] = e(1, L, hpg * 128)
            ws["ATT"] = e(1, Ll, dim)
            ws["FF"] = e(1, Ll, ex.params.ffn_dim)
            ws["T1"], ws["E_H"], ws["E"], ws["SE"] = e(Tt, 256), e(Tt, dim), e(Tt, dim), e(Tt, dim)
            ws["E0"] = e(Tt, 6 * dim)
            ws["MOD"] = e(Tt, ex.n_blocks, 6 * dim)
            ws["HSHIFT"], ws["HSCALE"] = e(Tt, 1, dim), e(Tt, 1, dim)
            ws["CTX_H"], ws["CTX"] = e(1, Lc, dim), e(1, Lc, dim)
            ws["CQ"] = e(1, Ll, dim)
            ws["CKV"] = [e(1, Lc, 2 * dim) for _ in range(ex.n_blocks)]
            if getattr(ex, "conditioning_kwargs", ()):
                # CLIP image branch: projection scratch and every block's image K/V (from the text without clip_fea)
                ws["Li"] = Li
                if Li:
                    ws["CLIP_H"], ws["CLIP"] = e(1, Li, ex.clip_dim), e(1, Li, dim)
                ws["CKVI"] = [e(1, Li or Lc, 2 * dim) for _ in range(ex.n_blocks)]
            ws["ROPE"] = ex.rope(T, H, Wd)[g * Ll:(g + 1) * Ll].contiguous()       # RoPE rows of MY tokens
            ws["ctx_sig"] = None
            wss.append(ws)
        ptrs = [{k: ws[k].data_ptr() for k in ("QKV", "QF", "KF", "VF", "ATTF", "ATT")} for ws in wss]
        for g, ws in enumerate(wss):
            qkv, att = exchange_tables(g, n, Ll, dim, hpg, ptrs)
            ws["DESC_QKV"], ws["N_QKV"] = self._table(qkv, ws["X"].device), len(qkv)
            ws["DESC_ATT"], ws["N_ATT"] = self._table(att, ws["X"].device), len(att)
        self._ws[key] = wss
        return wss

    def pre_step(self, g: int, wss, st: dict) -> None:
        # text embedding + every block's cross-attention K/V (and the image K/V of a CLIP model): only when the
        # conditioning changed, never in the graph
        if "CKVI" in wss[g]:
            self.ex[g]._prepare_ctx(wss[g], st["ctx"], st.get("clip"))
        else:
            self.ex[g]._prepare_ctx(wss[g], st["ctx"])

    # ------------------------------------------------------------------ one GPU's share of the step
    def run_rank(self, g: int, wss, x_ptr: int, st: dict, out_ptr: int) -> int:
        ex, ws, C = self.ex[g], wss[g], self.C
        W, dim = ex.W, ex.dim
        L, Ll, hpg = ws["L"], ws["Ll"], ws["hpg"]
        X, XM, QKV, ATT, FF, MOD, ROPE = ws["X"], ws["XM"], ws["QKV"], ws["ATT"], ws["FF"], ws["MOD"], ws["ROPE"]
        TH = ws["T"] * ws["H"]
        t = st["t"].reshape(-1)
        fr = frame_lookup(ws, row_off=g * Ll)             # per-frame timesteps: frame of each global token row
        nl = 0
        # ---- embedders: patchify the whole clip (a T*H tall image), embed only my token slice; time path is replicated
        C.patchify(x_ptr, ws["TOK"], 1, ex.params.in_dim, TH, ws["Wd"], 2)
        ops.gemm(ws["TOK"][:, g * Ll:(g + 1) * Ll], W["patch.w"], "bias", out=X, bias=W["patch.b"])
        ops.timestep_embedding(t, 256, time_factor=1.0, out=ws["T1"])
        ops.gemm(ws["T1"], W["time0.w"], "silu", out=ws["E_H"], bias=W["time0.b"])
        ops.gemm(ws["E_H"], W["time2.w"], "bias", out=ws["E"], bias=W["time2.b"])
        C.silu(ws["E"], ws["SE"])
        ops.gemm(ws["SE"], W["tproj.w"], "bias", out=ws["E0"], bias=W["tproj.b"])
        C.bcast_add(ws["E0"], W["mod_table"], MOD)
        C.bcast_add(ws["E"], W["head_shift"], ws["HSHIFT"])
        C.bcast_add(ws["E"], W["head_scale"], ws["HSCALE"])
        nl += 10

        def mod(i, j):
            return MOD[:, i, j * dim:(j + 1) * dim]

        def heads_of(tk: torch.Tensor, nh: int) -> torch.Tensor:      # token-major [1, rows, nh*128] -> [1, nh, rows, 128] view
            return tk.view(1, tk.shape[1], nh, 128).permute(0, 2, 1, 3)

        att_variant = attention_variant(hpg, L)
        slot = 0
        for i in range(ex.n_blocks):
            # ---- self attention: token-sliced QKV + q/k norm + RoPE, head-sliced attention between two exchanges
            ops.layernorm_modulate(X, XM, scale=mod(i, 1), shift=mod(i, 0), eps=ex.eps, **fr["ln"])
            nl += block_linear(W, XM, f"b{i}.qkv", "bias", out=QKV)
            C.rms_rope(QKV[:, :, :dim], W[f"b{i}.nq"], ROPE, ex.eps)
            C.rms_rope(QKV[:, :, dim:2 * dim], W[f"b{i}.nk"], ROPE, ex.eps)
            self._exchange(g, ws, slot, "QKV")
            ops.attention(heads_of(ws["QF"], hpg), heads_of(ws["KF"], hpg), heads_of(ws["VF"], hpg), out=ws["ATTF"],
                          variant=att_variant)
            self._exchange(g, ws, slot + 1, "ATT")
            slot += 2
            nl += 8 + block_linear(W, ATT, f"b{i}.o", "gate_res", out=X, residual=X, gate=mod(i, 2), **fr["gate"])
            # ---- cross attention: my query tokens against the replicated text (and image) K/V
            ops.layernorm_modulate(X, XM, gamma=W[f"b{i}.n3.g"], beta=W[f"b{i}.n3.b"], eps=ex.eps)
            nl += block_linear(W, XM, f"b{i}.cq", "bias", out=ws["CQ"])
            C.rms_rope(ws["CQ"], W[f"b{i}.cnq"], None, ex.eps)
            ex._cross_attention(ws, i, ATT)
            nl += 3 + block_linear(W, ATT, f"b{i}.co", "res", out=X, residual=X)
            # ---- FFN
            ops.layernorm_modulate(X, XM, scale=mod(i, 4), shift=mod(i, 3), eps=ex.eps, **fr["ln"])
            nl += 1 + block_linear(W, XM, f"b{i}.f0", "gelu", out=FF)
            nl += block_linear(W, FF, f"b{i}.f2", "gate_res", out=X, residual=X, gate=mod(i, 5), **fr["gate"])
        # ---- head on my tokens: AdaLN + Linear + unpatchify, rows stored into the LEAD GPU's output
        ops.layernorm_modulate(X, XM, scale=ws["HSCALE"][:, 0], shift=ws["HSHIFT"][:, 0], eps=ex.eps, **fr["ln"])
        head_gather(XM, W["head.w"], W["head.b"], ex.params.out_dim, TH, ws["Wd"], out_ptr=out_ptr, tok_off=g * Ll)
        self._end_step(g)
        nl += 3
        return nl
