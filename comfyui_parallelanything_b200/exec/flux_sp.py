"""Sequence-parallel (Ulysses) FLUX step for batch == 1 on N GPUs of one process.

The reference's batch == 1 mode walks the transformer blocks of ONE sample sequentially over the devices
(/root/reference/any_device_parallel.py:24-87, 1295-1305): every device already holds the full model, so it spreads
activation memory but buys no latency.  Here every GPU of the chain works on the sample at the same time:

  * linear layers (LayerNorm+modulate, QKV, proj, MLP, linear1/2, final layer) run on a token slice: GPU g owns
    ``Lt/N`` text tokens and ``Li/N`` image tokens (a horizontal band of the latent), local layout [txt slice | img slice];
  * attention runs on a head slice: GPU g owns ``H/N`` heads over the FULL sequence;
  * between the two layouts the data moves with ONE peer-pull kernel per GPU and exchange (csrc/comm/sp_a2a.cu): after a
    device-side flag handshake it reads the other GPUs' q/k/v (resp. attention-output) slabs straight out of their HBM
    over NVLink.  Epoch counters live in device memory, so each GPU's whole step (57 blocks x 2 exchanges) is one CUDA
    graph replayed by the engine's native host threads.

Weights are replicated (exactly what the reference does - every device holds the full model), activations and FLOPs are
split N ways.  Per block a GPU sends/receives ~4 x L/N x hid x (N-1)/N bf16 (FLUX-dev, N = 8: ~12 MB), i.e. < 1 ms of
NVLink time per step next to ~6 ms of compute.
"""
from __future__ import annotations

from typing import List, Optional

import torch

from .. import ops
from . import block_linear
from .dit import head_gather
from .sp_common import UlyssesBase, attention_variant


def supported(executors) -> Optional[str]:
    """None if the chain's native FLUX replicas can run sequence-parallel, else the reason they cannot."""
    n = len(executors)
    if n < 2:
        return "needs at least 2 GPUs"
    C = ops.require()
    if n > C.SP_MAX_RANKS:
        return f"at most {C.SP_MAX_RANKS} GPUs"
    ex0 = executors[0]
    if any(getattr(e, "pa_family", None) != "flux" or not getattr(e, "pa_native", False) for e in executors):
        return "every replica must be a native FLUX executor"
    if ex0.heads % n:
        return f"{ex0.heads} heads are not divisible by {n} GPUs"
    if 2 * (ex0.n_double + ex0.n_single) + 2 > C.SP_MAX_SLOTS:
        return "too many blocks for the flag table"
    return None


def exchange_tables(g: int, n: int, Lt: int, Li: int, hid: int, mlp: int, hpg: int, ptrs):
    """Copy descriptors (src, dst, src_pitch, dst_pitch, rows, row_bytes) GPU ``g`` pulls with, bf16 buffers:
    ``ptrs[r]`` = base addresses of rank r's Q / K / V [H, Ll, 128] (all heads, its [txt | img] token slice), QF / KF / VF
    [hpg, L, 128] (its heads, all tokens in global [txt | img] order), ATTF [L, hpg*128] and CAT [Ll, hid+mlp].
    Pure function of the geometry (CPU-testable)."""
    Ltl, Lil = Lt // n, Li // n
    Ll, L = Ltl + Lil, Lt + Li
    qkv, att = [], []
    for r in range(n):
        for name_l, name_f in (("Q", "QF"), ("K", "KF"), ("V", "VF")):
            src_base = ptrs[r][name_l] + g * hpg * Ll * 256          # heads of g inside r's [H, Ll, 128]
            dst_base = ptrs[g][name_f]
            # txt slice of r -> global rows [r*Ltl, ...), img slice -> global rows [Lt + r*Lil, ...)
            qkv.append((src_base, dst_base + (r * Ltl) * 256, Ll * 256, L * 256, hpg, Ltl * 256))
            qkv.append((src_base + Ltl * 256, dst_base + (Lt + r * Lil) * 256, Ll * 256, L * 256, hpg, Lil * 256))
        # attention output of r's heads for MY token rows -> columns [r*hpg*128, ...) of my CAT rows
        src = ptrs[r]["ATTF"]
        dst = ptrs[g]["CAT"] + r * hpg * 256
        ld = (hid + mlp) * 2
        att.append((src + (g * Ltl) * hpg * 256, dst, hpg * 256, ld, Ltl, hpg * 256))
        att.append((src + (Lt + g * Lil) * hpg * 256, dst + Ltl * ld, hpg * 256, ld, Lil, hpg * 256))
    return qkv, att


class FluxUlysses(UlyssesBase):
    """Wires N FluxExecutors (one per GPU, same process) for sequence-parallel batch-1 steps."""
    family = "flux"

    def __init__(self, executors: List, timeout_ms: int = 20000):
        why = supported(executors)
        if why:
            raise ValueError(f"sequence-parallel FLUX unavailable: {why}")
        super().__init__(executors, timeout_ms)

    # ------------------------------------------------------------------ engine-facing protocol
    def accepts(self, x, context) -> bool:
        if x.dim() != 4 or context.dim() != 3:
            return False
        n = self.n
        H, Wd, Lt = x.shape[2], x.shape[3], context.shape[1]
        return H % 2 == 0 and Wd % 2 == 0 and Lt % n == 0 and ((H // 2) * (Wd // 2)) % n == 0 and Lt >= n

    def geometry(self, x, timesteps, context, kwargs=None) -> tuple:
        return (x.shape[2], x.shape[3], context.shape[1])

    def io_key(self, x, timesteps, context, kwargs) -> tuple:
        y = kwargs.get("y")
        return ("sp", tuple(x.shape), tuple(context.shape), None if y is None else tuple(y.shape),
                kwargs.get("guidance") is not None)

    def slot_buffers(self, device, x, timesteps, context, kwargs) -> dict:
        st = super().slot_buffers(device, x, timesteps, context, kwargs)
        bf = torch.bfloat16
        st["y"] = torch.zeros(1, self.ex[0].params.vec_in_dim, dtype=bf, device=device)
        st["g"] = torch.ones(1, dtype=bf, device=device)
        return st

    def stage(self, st, timesteps, context, kwargs, cache_conditioning: bool) -> None:
        super().stage(st, timesteps, context, kwargs, cache_conditioning)
        y, guidance = kwargs.get("y"), kwargs.get("guidance")
        if y is not None:
            st["y"].copy_(y[:, :st["y"].shape[1]], non_blocking=True)
        if guidance is not None:
            st["g"].copy_(guidance.reshape(-1)[:1], non_blocking=True)
        elif self.ex[0].params.guidance_embed:
            raise ValueError("guidance-distilled model needs a guidance strength")

    # ------------------------------------------------------------------ geometry / buffers
    def workspace(self, H: int, Wd: int, Lt: int) -> list:
        key = (H, Wd, Lt)
        got = self._ws.get(key)
        if got is not None:
            return got
        n, ex0 = self.n, self.ex[0]
        Li = (H // 2) * (Wd // 2)
        if Lt % n or Li % n:
            raise ValueError(f"text ({Lt}) / image ({Li}) token counts must divide by {n} GPUs")
        Ltl, Lil = Lt // n, Li // n
        Ll, L = Ltl + Lil, Lt + Li
        hid, mlp, heads = ex0.hid, ex0.mlp, ex0.heads
        hpg = heads // n
        wss = []
        for g, ex in enumerate(self.ex):
            d = ex.device
            e = lambda *s: torch.empty(*s, dtype=torch.bfloat16, device=d)  # noqa: E731
            ws = dict(g=g, H=H, Wd=Wd, Lt=Lt, Li=Li, L=L, Ltl=Ltl, Lil=Lil, Ll=Ll, hpg=hpg)
            ws["X"], ws["XM"] = e(1, Ll, hid), e(1, Ll, hid)
            ws["CAT"] = e(1, Ll, hid + mlp)                          # [attention (pulled) | GELU(mlp)] of the local tokens
            ws["Q"], ws["K"], ws["V"] = e(1, heads, Ll, 128), e(1, heads, Ll, 128), e(1, heads, Ll, 128)   # all heads, local tokens
            ws["QF"], ws["KF"], ws["VF"] = e(1, hpg, L, 128), e(1, hpg, L, 128), e(1, hpg, L, 128)        # my heads, all tokens
            ws["ATTF"] = e(1, L, hpg * 128)                          # attention output of my heads, all tokens
            ws["TOK"] = e(1, Li, ex.params.in_channels)
            ws["T1"], ws["T2"] = e(1, 256), e(1, 256)
            ws["HC"] = e(1, ex.W["vec_out.w"].shape[1])
            ws["SVEC"], ws["MOD"] = e(1, hid), e(1, ex.mod_total)
            ws["ROPE"] = ex.rope(H, Wd, Lt)
            wss.append(ws)
        # descriptor tables (static addresses -> built once, baked into the graphs)
        ptrs = [{k: ws[k].data_ptr() for k in ("Q", "K", "V", "QF", "KF", "VF", "ATTF", "CAT")} for ws in wss]
        for g, ws in enumerate(wss):
            qkv, att = exchange_tables(g, n, Lt, Li, hid, mlp, hpg, ptrs)
            ws["DESC_QKV"], ws["N_QKV"] = self._table(qkv, ws["X"].device), len(qkv)
            ws["DESC_ATT"], ws["N_ATT"] = self._table(att, ws["X"].device), len(att)
        self._ws[key] = wss
        return wss

    # ------------------------------------------------------------------ one GPU's share of the step
    def run_rank(self, g: int, wss, x_ptr: int, st: dict, out_ptr: int) -> int:
        """Everything GPU g does for one step; ``x_ptr`` / ``out_ptr`` are the lead GPU's latent / output buffers
        (peer mappings), ``st`` the step inputs staged on GPU g (t / ctx / y / guidance).  Returns the launch count."""
        ex, ws, C = self.ex[g], wss[g], self.C
        t, ctx, y = st["t"], st["ctx"], st["y"]
        guidance = st["g"] if ex.params.guidance_embed else None
        W, hid, mlp, n = ex.W, ex.hid, ex.mlp, self.n
        Lt, Li, Ltl, Lil, Ll, hpg = ws["Lt"], ws["Li"], ws["Ltl"], ws["Lil"], ws["Ll"], ws["hpg"]
        X, XM, CAT, Q, K, V, ROPE = ws["X"], ws["XM"], ws["CAT"], ws["Q"], ws["K"], ws["V"], ws["ROPE"]
        Xt, Xi, XMt, XMi = X[:, :Ltl], X[:, Ltl:], XM[:, :Ltl], XM[:, Ltl:]
        ATT, MH = CAT[:, :, :hid], CAT[:, :, hid:]
        ro_t, ro_i = g * Ltl, Lt + g * Lil - Ltl            # global RoPE row = local row + offset
        nl = 0
        p = ex.params
        ge = p.guidance_embed
        # ---- embedders (tiny): patchify the whole latent, embed only my token band; vec / modulations are replicated
        C.patchify(x_ptr, ws["TOK"], 1, p.in_channels // 4, ws["H"], ws["Wd"], 2)
        ops.gemm(ws["TOK"][:, g * Lil:(g + 1) * Lil], W["img_in.w"], "bias", out=Xi, bias=W["img_in.b"])
        ops.gemm(ctx[:, g * Ltl:(g + 1) * Ltl], W["txt_in.w"], "bias", out=Xt, bias=W["txt_in.b"])
        ops.timestep_embedding(t, 256, out=ws["T1"])
        HC = ws["HC"]
        ops.gemm(ws["T1"], W["time_in.in.w"], "silu", out=HC[:, :hid], bias=W["time_in.in.b"])
        col = hid
        nl += 5
        if ge:
            ops.timestep_embedding(guidance, 256, out=ws["T2"])
            ops.gemm(ws["T2"], W["guidance_in.in.w"], "silu", out=HC[:, col:col + hid], bias=W["guidance_in.in.b"])
            col += hid
            nl += 2
        ops.gemm(y, W["vector_in.in.w"], "silu", out=HC[:, col:col + hid], bias=W["vector_in.in.b"])
        ops.gemm(HC, W["vec_out.w"], "silu", out=ws["SVEC"], bias=W["vec_out.b"])
        nl += 2 + block_linear(W, ws["SVEC"], "mod", "bias", out=ws["MOD"])

        att_variant = attention_variant(hpg, ws["L"])
        slot = 0
        for i in range(ex.n_double):
            for s, xs, xms, off, ro in (("img", Xi, XMi, Ltl, ro_i), ("txt", Xt, XMt, 0, ro_t)):
                k = ("d", i, s)
                ops.layernorm_modulate(xs, xms, scale=ex._mod(ws, k, 1), shift=ex._mod(ws, k, 0))
                nl += 1 + block_linear(W, xms, f"d{i}.{s}.qkv", "qkv_rope", q=Q, k=K, v=V, q_scale=W[f"d{i}.{s}.qs"],
                                       k_scale=W[f"d{i}.{s}.ks"], rope=ROPE, seq_off=off, rope_off=ro)
            self._exchange(g, ws, slot, "QKV")                      # all heads / my tokens -> my heads / all tokens
            ops.attention(ws["QF"], ws["KF"], ws["VF"], out=ws["ATTF"], variant=att_variant)
            self._exchange(g, ws, slot + 1, "ATT")                  # my heads / all tokens -> all heads / my tokens
            slot += 2
            nl += 5
            for s, xs, xms, a, mh in (("img", Xi, XMi, ATT[:, Ltl:], MH[:, Ltl:]), ("txt", Xt, XMt, ATT[:, :Ltl], MH[:, :Ltl])):
                k = ("d", i, s)
                nl += block_linear(W, a, f"d{i}.{s}.proj", "gate_res", out=xs, residual=xs, gate=ex._mod(ws, k, 2))
                ops.layernorm_modulate(xs, xms, scale=ex._mod(ws, k, 4), shift=ex._mod(ws, k, 3))
                nl += block_linear(W, xms, f"d{i}.{s}.mlp0", "gelu", out=mh)
                nl += block_linear(W, mh, f"d{i}.{s}.mlp2", "gate_res", out=xs, residual=xs, gate=ex._mod(ws, k, 5))
                nl += 1
        for i in range(ex.n_single):
            k = ("s", i)
            ops.layernorm_modulate(X, XM, scale=ex._mod(ws, k, 1), shift=ex._mod(ws, k, 0))
            nl += 1 + block_linear(W, XM, f"s{i}.l1", "qkv_rope", q=Q, k=K, v=V, q_scale=W[f"s{i}.qs"],
                                   k_scale=W[f"s{i}.ks"], rope=ROPE, seq_off=0, rope_off=ro_t, rope_off2=ro_i,
                                   seg_rows=Ltl, out=CAT, mlp_col_off=hid)
            self._exchange(g, ws, slot, "QKV")
            ops.attention(ws["QF"], ws["KF"], ws["VF"], out=ws["ATTF"], variant=att_variant)
            self._exchange(g, ws, slot + 1, "ATT")
            slot += 2
            nl += 5 + block_linear(W, CAT, f"s{i}.l2", "gate_res", out=X, residual=X, gate=ex._mod(ws, k, 2))
        # ---- final layer on my image tokens: AdaLN + Linear + unpatchify, rows stored into the LEAD GPU's output
        k = ("final",)
        ops.layernorm_modulate(Xi, XMi, scale=ex._mod(ws, k, 1), shift=ex._mod(ws, k, 0))
        head_gather(XMi, W["final.w"], W["final.b"], p.out_channels // 4, ws["H"], ws["Wd"], out_ptr=out_ptr,
                    tok_off=g * Lil)
        # (no closing handshake: the engine orders the lead's staging-buffer rewrite after every GPU's stream, and a GPU
        # cannot run ahead into the next step's first exchange before all peers signalled it)
        self._end_step(g)
        nl += 3
        return nl
