"""Sequence-parallel (Ulysses) Z-Image / NextDiT step for batch == 1 on N GPUs of one process.

Same scheme as ``flux_sp.py`` (the joint [caption | image] sequence of a NextDiT layer is a FLUX single-stream block
without the parallel MLP): every GPU owns ``Lc / N`` caption tokens and ``Li / N`` image tokens for the linear layers
and the RMSNorm / gate kernels, ``H / N`` heads over the whole sequence for attention, with one peer-pull exchange
(csrc/comm/sp_a2a.cu) before and one after it.  The ``noise_refiner`` layers attend over the image tokens only and use
their own (image-only) exchange tables; the caption path (``context_refiner``) depends on the conditioning only and is
computed by every GPU for itself, eagerly and only when the prompt changes (``ZImageExecutor._prepare_ctx``).

Replaces the reference's batch == 1 layer split (/root/reference/any_device_parallel.py:24-87, 1295-1305).  Z-Image-Turbo has
30 heads: chains of 2, 3, 5 or 6 GPUs qualify.
"""
from __future__ import annotations

from typing import List, Optional

import torch

from .. import ops
from . import block_linear
from .dit import head_gather
from .flux_sp import exchange_tables
from .sp_common import UlyssesBase, attention_variant


def supported(executors) -> Optional[str]:
    n = len(executors)
    if n < 2:
        return "needs at least 2 GPUs"
    C = ops.require()
    if n > C.SP_MAX_RANKS:
        return f"at most {C.SP_MAX_RANKS} GPUs"
    ex0 = executors[0]
    if any(getattr(e, "pa_family", None) != "zimage" or not getattr(e, "pa_native", False) for e in executors):
        return "every replica must be a native Z-Image executor"
    if ex0.heads % n:
        return f"{ex0.heads} heads are not divisible by {n} GPUs"
    if 2 * (ex0.n_nr + ex0.n_layers) + 2 > C.SP_MAX_SLOTS:
        return "too many blocks for the flag table"
    return None


class ZImageUlysses(UlyssesBase):
    family = "zimage"

    def __init__(self, executors: List, timeout_ms: int = 20000):
        why = supported(executors)
        if why:
            raise ValueError(f"sequence-parallel Z-Image unavailable: {why}")
        super().__init__(executors, timeout_ms)

    # ------------------------------------------------------------------ engine-facing protocol
    def accepts(self, x, context) -> bool:
        if x.dim() != 4 or context.dim() != 3 or x.shape[1] != self.ex[0].params.in_channels:
            return False
        n = self.n
        H, Wd, Lc = x.shape[2], x.shape[3], context.shape[1]
        return H % 2 == 0 and Wd % 2 == 0 and Lc % n == 0 and ((H // 2) * (Wd // 2)) % n == 0 and Lc >= n

    def geometry(self, x, timesteps, context, kwargs=None) -> tuple:
        return (x.shape[2], x.shape[3], context.shape[1])

    def workspace(self, H: int, Wd: int, Lc: int) -> list:
        key = (H, Wd, Lc)
        got = self._ws.get(key)
        if got is not None:
            return got
        n, ex0 = self.n, self.ex[0]
        p, dim, heads = ex0.params, ex0.dim, ex0.heads
        Li = (H // 2) * (Wd // 2)
        L = Lc + Li
        Lcl, Lil = Lc // n, Li // n
        Ll, hpg = Lcl + Lil, heads // n
        wss = []
        for g, ex in enumerate(self.ex):
            d = ex.device
            e = lambda *s: torch.empty(*s, dtype=torch.bfloat16, device=d)  # noqa: E731
            ws = dict(g=g, H=H, Wd=Wd, Lc=Lc, Li=Li, L=L, Lcl=Lcl, Lil=Lil, Ll=Ll, hpg=hpg)
            ws["X"], ws["XM"], ws["Y"] = e(1, Ll, dim), e(1, Ll, dim), e(1, Ll, dim)
            ws["CAT"] = e(1, Ll, dim)                                 # pulled attention output: all heads, my tokens
            ws["FF"] = e(1, Ll, p.ffn_hidden)
            ws["Q"], ws["K"], ws["V"] = (e(1, heads, Ll, 128) for _ in range(3))          # joint layers: all heads, my tokens
            ws["QF"], ws["KF"], ws["VF"] = (e(1, hpg, L, 128) for _ in range(3))          # my heads, all tokens
            ws["ATTF"] = e(1, L, hpg * 128)
            # noise refiner: image tokens only
            ws["CATi"] = e(1, Lil, dim)
            ws["Qi"], ws["Ki"], ws["Vi"] = (e(1, heads, Lil, 128) for _ in range(3))
            ws["QFi"], ws["KFi"], ws["VFi"] = (e(1, hpg, Li, 128) for _ in range(3))
            ws["ATTFi"] = e(1, Li, hpg * 128)
            ws["TOK"] = e(1, Li, 4 * p.in_channels)
            ws["T1"], ws["TH"], ws["TE"], ws["STE"] = e(1, 256), e(1, ex.W["t0.w"].shape[0]), e(1, p.adaln_dim), e(1, p.adaln_dim)
            ws["MOD"] = e(1, ex.W["mod.w"].shape[0])
            ws["ROPE"] = ex.rope(H, Wd, Lc)
            ws["ROPE_I"] = ws["ROPE"][Lc:].contiguous()
            # scratch of the (replicated, eager) caption path: what ZImageExecutor._prepare_ctx expects of a workspace
            ws["CTXWS"] = dict(Lc=Lc, XM=e(1, Lc, dim), Y=e(1, Lc, dim), ATT=e(1, Lc, dim), FF=e(1, Lc, p.ffn_hidden),
                               Qt=e(1, heads, Lc, 128), Kt=e(1, heads, Lc, 128), Vt=e(1, heads, Lc, 128), ROPE=ws["ROPE"],
                               CAPN=e(1, Lc, p.cap_feat_dim), XT0=e(1, Lc, dim), ctx_sig=None)
            wss.append(ws)
        joint = [{k: ws[k].data_ptr() for k in ("Q", "K", "V", "QF", "KF", "VF", "ATTF", "CAT")} for ws in wss]
        image = [{k: ws[k + "i"].data_ptr() for k in ("Q", "K", "V", "QF", "KF", "VF", "ATTF", "CAT")} for ws in wss]
        for g, ws in enumerate(wss):
            for tag, (lt, ptrs) in (("", (Lc, joint)), ("_I", (0, image))):
                qkv, att = exchange_tables(g, n, lt, Li, dim, 0, hpg, ptrs)
                qkv = [r for r in qkv if r[4] > 0 and r[5] > 0]       # image-only tables have no caption segment
                att = [r for r in att if r[4] > 0 and r[5] > 0]
                ws["DESC_QKV" + tag], ws["N_QKV" + tag] = self._table(qkv, ws["X"].device), len(qkv)
                ws["DESC_ATT" + tag], ws["N_ATT" + tag] = self._table(att, ws["X"].device), len(att)
        self._ws[key] = wss
        return wss

    def pre_step(self, g: int, wss, st: dict) -> None:
        self.ex[g]._prepare_ctx(wss[g]["CTXWS"], st["ctx"])

    # ------------------------------------------------------------------ one GPU's share of the step
    def _block(self, g, ws, slot, name, xs, xms, ys, cat, ff, q, k, v, qf, kf, vf, attf, tag, modulated, att_variant, **rope_kw):
        ex = self.ex[g]
        W, eps = ex.W, ex.eps
        sc_a = ex._mod(ws, name, 0) if modulated else None
        g_a = ex._mod(ws, name, 1) if modulated else None
        sc_m = ex._mod(ws, name, 2) if modulated else None
        g_m = ex._mod(ws, name, 3) if modulated else None
        nl = 9
        ops.rmsnorm_modulate(xs, xms, weight=W[name + ".n1"], scale=sc_a, eps=eps)
        nl += block_linear(W, xms, name + ".qkv", "qkv_rope", q=q, k=k, v=v, q_scale=W[name + ".qs"], k_scale=W[name + ".ks"],
                           seq_off=0, qk_eps=eps, **rope_kw)
        self._exchange(g, ws, slot, "QKV" + tag)                   # all heads / my tokens -> my heads / all tokens
        ops.attention(qf, kf, vf, out=attf, variant=att_variant)
        self._exchange(g, ws, slot + 1, "ATT" + tag)               # my heads / all tokens -> all heads / my tokens
        nl += block_linear(W, cat, name + ".out", "bias", out=ys)
        ops.rmsnorm_modulate(ys, xs, weight=W[name + ".n2"], gate=g_a, residual=xs, eps=eps)
        ops.rmsnorm_modulate(xs, xms, weight=W[name + ".f1"], scale=sc_m, eps=eps)
        nl += block_linear(W, xms, name + ".w13", "swiglu", out=ff)
        nl += block_linear(W, ff, name + ".w2", "bias", out=ys)
        ops.rmsnorm_modulate(ys, xs, weight=W[name + ".f2"], gate=g_m, residual=xs, eps=eps)
        return nl

    def run_rank(self, g: int, wss, x_ptr: int, st: dict, out_ptr: int) -> int:
        ex, ws, C = self.ex[g], wss[g], self.C
        W, p = ex.W, ex.params
        Lc, Lcl, Lil, hpg = ws["Lc"], ws["Lcl"], ws["Lil"], ws["hpg"]
        X, XM, Y, FF = ws["X"], ws["XM"], ws["Y"], ws["FF"]
        Xt, Xi = X[:, :Lcl], X[:, Lcl:]
        nl = 0
        # ---- embedders: patchify the whole latent, embed my image band; my slice of the (cached) refined caption tokens
        C.patchify(x_ptr, ws["TOK"], 1, p.in_channels, ws["H"], ws["Wd"], 2)
        ops.gemm(ws["TOK"][:, g * Lil:(g + 1) * Lil], W["img_in.w"], "bias", out=Xi, bias=W["img_in.b"])
        ops.timestep_embedding(st["t"], 256, time_factor=float(p.t_scale), out=ws["T1"])
        ops.gemm(ws["T1"], W["t0.w"], "silu", out=ws["TH"], bias=W["t0.b"])
        ops.gemm(ws["TH"], W["t2.w"], "bias", out=ws["TE"], bias=W["t2.b"])
        C.silu(ws["TE"], ws["STE"])
        ops.gemm(ws["STE"], W["mod.w"], "bias", out=ws["MOD"], bias=W["mod.b"])
        C.copy_rows(ws["CTXWS"]["XT0"][:, g * Lcl:(g + 1) * Lcl], Xt)
        nl += 8
        slot = 0
        for i in range(ex.n_nr):            # image tokens only; RoPE row of local image row r = g*Lil + r of the image table
            nl += self._block(g, ws, slot, f"nr{i}", Xi, XM[:, Lcl:], Y[:, Lcl:], ws["CATi"], FF[:, Lcl:], ws["Qi"], ws["Ki"],
                              ws["Vi"], ws["QFi"], ws["KFi"], ws["VFi"], ws["ATTFi"], "_I", True,
                              attention_variant(hpg, ws["Li"]), rope=ws["ROPE_I"], rope_off=g * Lil)
            slot += 2
        for i in range(ex.n_layers):        # joint sequence, local layout [caption slice | image slice]
            nl += self._block(g, ws, slot, f"l{i}", X, XM, Y, ws["CAT"], FF, ws["Q"], ws["K"], ws["V"], ws["QF"], ws["KF"],
                              ws["VF"], ws["ATTF"], "", True, attention_variant(hpg, ws["L"]), rope=ws["ROPE"],
                              rope_off=g * Lcl, rope_off2=Lc + g * Lil - Lcl, seg_rows=Lcl)
            slot += 2
        # ---- head on my image tokens: LayerNorm * (1 + scale) + Linear + unpatchify, rows stored into the LEAD GPU's output
        ops.layernorm_modulate(Xi, XM[:, Lcl:], scale=ex._mod(ws, "final", 0), eps=1e-6)
        head_gather(XM[:, Lcl:], W["final.w"], W["final.b"], p.in_channels, ws["H"], ws["Wd"], out_ptr=out_ptr,
                    tok_off=g * Lil)
        self._end_step(g)
        nl += 3
        return nl
