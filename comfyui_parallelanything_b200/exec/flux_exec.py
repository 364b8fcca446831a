"""FLUX.1 MM-DiT forward on hand-written sm_100a kernels (the per-replica hot path).

Replaces what the reference reaches through ``forward_fn(x_in, t_in, context=c_in, **k_in)``
(/root/reference/any_device_parallel.py:1390: thousands of stock torch launches) by a static
schedule over packed weights:

  * every Linear is the persistent tcgen05/TMEM/TMA GEMM (csrc/kernels/gemm_tcgen05.cuh) with the
    following work fused into its epilogue: bias, GELU, AdaLN gated residual, the QKV head split +
    q/k RMSNorm + RoPE (+ the GELU'd MLP half of a single block), and for the last layer
    unpatchify + Euler update + (NVLink peer) store — the fused "gather";
  * txt/img streams live in ONE residual buffer ``X[B, Lt+Li, hid]``; the double blocks address
    the two row ranges as strided 3-D TMA tensors, so no cat/split/chunk kernels exist;
  * all 96 modulation projections are one GEMM over the concatenated modulation weights;
  * attention is csrc/kernels/attention.cu (S/O accumulators in TMEM), writing straight into the
    concat buffer that ``linear2`` of a single block consumes.

Per step: 19*13 + 38*4 + ~12 = ~410 kernel launches, optionally replayed as one CUDA graph.
"""
from __future__ import annotations

import os
from typing import Dict, Optional

import torch
import torch.nn as nn

from .. import ops
from . import bf16, block_linear, quantize_block_weights
from .dit import DiTExecutor, head_gather, rope_layout
from ..models import flux as flux_model
from ..utils.log import nvtx_range


class FluxExecutor(DiTExecutor):
    pa_family = "flux"

    def __init__(self, model: "flux_model.Flux", device, cuda_graphs: bool = False, fp8: bool = False):
        super().__init__(model, device, cuda_graphs)
        p = self.params
        self.hid, self.heads = p.hidden_size, p.num_heads
        if self.hid // self.heads != 128:
            raise ValueError("FluxExecutor is specialised for head_dim 128")
        if p.patch_size != 2:
            raise ValueError("FluxExecutor is specialised for 2x2 patches")
        self.mlp = int(p.hidden_size * p.mlp_ratio)
        # fp8=True: the block GEMMs (qkv / proj / mlp / linear1 / linear2 = 99.9 % of the FLOPs) run as MXFP8
        # block-scaled tcgen05 GEMMs (weights quantised once here, activations per GEMM); embedders,
        # modulation and the final layer stay bf16.
        self.fp8 = bool(fp8)
        # the fused scatter/patch-embed kernel is specialised for 16 latent channels x (2x2) patches
        self.fused_embed = (p.in_channels == 64)
        d = self.device
        W: Dict[str, torch.Tensor] = {}

        def lin(name, m):
            W[name + ".w"] = bf16(m.weight, d)
            W[name + ".b"] = bf16(m.bias, d) if m.bias is not None else None

        lin("img_in", model.img_in)
        lin("txt_in", model.txt_in)
        lin("time_in.in", model.time_in.in_layer)
        lin("vector_in.in", model.vector_in.in_layer)
        outs = [model.time_in.out_layer]
        if p.guidance_embed:
            lin("guidance_in.in", model.guidance_in.in_layer)
            outs.append(model.guidance_in.out_layer)
        outs.append(model.vector_in.out_layer)
        # vec = sum_i out_i(h_i)  ==  [h_t | h_g | h_y] @ [W_t | W_g | W_y]^T + (b_t + b_g + b_y)
        W["vec_out.w"] = torch.cat([bf16(o.weight, d) for o in outs], dim=1).contiguous()
        W["vec_out.b"] = sum(o.bias.detach().float().to(d) for o in outs).to(torch.bfloat16)
        mods, self.mod_off = [], {}
        off = 0
        for i, blk in enumerate(model.double_blocks):
            for s in ("img", "txt"):
                m = getattr(blk, s + "_mod").lin
                mods.append(m)
                self.mod_off[("d", i, s)] = off
                off += m.weight.shape[0]
                lin(f"d{i}.{s}.qkv", getattr(blk, s + "_attn").qkv)
                lin(f"d{i}.{s}.proj", getattr(blk, s + "_attn").proj)
                lin(f"d{i}.{s}.mlp0", getattr(blk, s + "_mlp")[0])
                lin(f"d{i}.{s}.mlp2", getattr(blk, s + "_mlp")[2])
                W[f"d{i}.{s}.qs"] = bf16(getattr(blk, s + "_attn").norm.query_norm.scale, d)
                W[f"d{i}.{s}.ks"] = bf16(getattr(blk, s + "_attn").norm.key_norm.scale, d)
        for i, blk in enumerate(model.single_blocks):
            mods.append(blk.modulation.lin)
            self.mod_off[("s", i)] = off
            off += blk.modulation.lin.weight.shape[0]
            lin(f"s{i}.l1", blk.linear1)
            lin(f"s{i}.l2", blk.linear2)
            W[f"s{i}.qs"] = bf16(blk.norm.query_norm.scale, d)
            W[f"s{i}.ks"] = bf16(blk.norm.key_norm.scale, d)
        fin = model.final_layer.adaLN_modulation[1]
        mods.append(fin)
        self.mod_off[("final",)] = off
        off += fin.weight.shape[0]
        self.mod_total = off
        W["mod.w"] = torch.cat([bf16(m.weight, d) for m in mods], dim=0).contiguous()
        W["mod.b"] = torch.cat([bf16(m.bias, d) for m in mods], dim=0).contiguous()
        lin("final", model.final_layer.linear)
        self.W = W
        if self.fp8:
            names = [k[:-2] for k in W if k.endswith(".w") and (k.startswith("d") or k.startswith("s"))
                     and k.split(".")[-2] in ("qkv", "proj", "mlp0", "mlp2", "l1", "l2")]
            # the modulation table (all blocks' adaLN linears, 1 056 768 x 3072 for FLUX.1-dev) is a pure weight stream
            # (6.5 GB in bf16 for <= 8 rows of activations): as MXFP8 it is half the bytes
            if os.environ.get("PA_FP8_MOD", "1") != "0":
                names.append("mod")
            # B-tile width the GEMM will use: 256 (single accumulator) for the fused QKV epilogues,
            # 224 (double-buffered accumulators) for everything else
            quantize_block_weights(W, names, lambda n: 256 if n.split(".")[-1] in ("qkv", "l1") else 224)
            torch.cuda.empty_cache()
        self.n_double, self.n_single = len(model.double_blocks), len(model.single_blocks)
        # fork the txt / img chains of the double blocks onto two streams with disjoint SM budgets (PA_DUAL_STREAM=0: off)
        self.dual_stream = os.environ.get("PA_DUAL_STREAM", "1") != "0"
        # fp8: attention / GELU epilogues emit the next GEMM's MXFP8 A operand themselves (PA_FP8_FUSED_QUANT=0: separate
        # quantise kernels in front of every GEMM)
        self.fused_quant = os.environ.get("PA_FP8_FUSED_QUANT", "1") != "0"
        self._side = self._ev_fork = self._ev_join = None

    # ------------------------------------------------------------------ workspaces
    def rope(self, H: int, Wd: int, Lt: int) -> torch.Tensor:
        """fp32 [Lt + (H/2)*(W/2), 64, 2] RoPE table of the joint [txt | img] sequence."""
        ids = flux_model.position_ids(1, H // 2, Wd // 2, Lt, self.device)
        return rope_layout(flux_model.EmbedND(128, self.params.theta, self.params.axes_dim)(ids))

    def _new_workspace(self, B: int, H: int, Wd: int, Lt: int) -> dict:
        d, hid, mlp = self.device, self.hid, self.mlp
        Li = (H // 2) * (Wd // 2)
        L = Lt + Li
        e = lambda *s: torch.empty(*s, dtype=torch.bfloat16, device=d)  # noqa: E731
        ws = dict(B=B, H=H, Wd=Wd, Lt=Lt, Li=Li, L=L)
        ws["X"] = e(B, L, hid)
        ws["XM"] = e(B, L, hid)
        ws["CAT"] = e(B, L, hid + mlp)
        ws["Q"], ws["K"], ws["V"] = e(B, self.heads, L, 128), e(B, self.heads, L, 128), e(B, self.heads, L, 128)
        ws["TOK"] = e(B, Li, self.params.in_channels)
        ws["T1"], ws["T2"] = e(B, 256), e(B, 256)
        ws["HC"] = e(B, self.W["vec_out.w"].shape[1])
        ws["SVEC"] = e(B, hid)
        ws["MOD"] = e(B, self.mod_total)
        ws["OUT"] = e(B, self.params.out_channels // 4, H, Wd)
        if self.fp8 and self.fused_quant:
            # MXFP8 operands written directly by the producing epilogues (attention, GELU): e4m3 bytes + UE8M0 scale
            # chunks (zero-initialised once: scale bytes of rows beyond the sequence are never written)
            u8 = lambda *s: torch.zeros(*s, dtype=torch.uint8, device=d)  # noqa: E731
            sfb = lambda rows, k: u8(B * ((rows + 127) // 128) * (k // 128) * 512)  # noqa: E731
            ws["CAT8"], ws["CAT8_SF"] = u8(B, L, hid + mlp), sfb(L, hid + mlp)
            ws["MH8I"], ws["MH8I_SF"] = u8(B, Li, mlp), sfb(Li, mlp)
            ws["MH8T"], ws["MH8T_SF"] = u8(B, Lt, mlp), sfb(Lt, mlp)
            ws["XM8"], ws["XM8_SF"] = u8(B, L, hid), sfb(L, hid)            # LayerNorm+modulate outputs, per chain
            ws["XM8I"], ws["XM8I_SF"] = u8(B, Li, hid), sfb(Li, hid)
            ws["XM8T"], ws["XM8T_SF"] = u8(B, Lt, hid), sfb(Lt, hid)
        ws["ROPE"] = self.rope(H, Wd, Lt)
        return ws

    # ------------------------------------------------------------------ schedule
    def _run(self, ws, x_ptr: int, t, ctx, y, guidance, out, x_in=None, sigmas=None, out_ptr: Optional[int] = None,
             out_sample_off: int = 0, t_ptr: Optional[int] = None, g_ptr: Optional[int] = None, x_copy=None):
        W, hid, mlp, Lt, B = self.W, self.hid, self.mlp, ws["Lt"], ws["B"]
        C = ops.require()
        n = 0
        X, XM, CAT, Q, K, V, ROPE = ws["X"], ws["XM"], ws["CAT"], ws["Q"], ws["K"], ws["V"], ws["ROPE"]
        Xi, Xt = X[:, Lt:], X[:, :Lt]
        XMi, XMt = XM[:, Lt:], XM[:, :Lt]
        ATT = CAT[:, :, :hid]
        MH = CAT[:, :, hid:]
        # ---- embedders
        HC = ws["HC"]
        ge = self.params.guidance_embed
        if self.fused_embed:
            # fused scatter: (peer) latent shard -> patchify -> img_in GEMM, + timestep/guidance embeddings
            C.scatter_patch_embed(W["img_in.w"], W["img_in.b"], x_ptr, t_ptr if t_ptr is not None else t.data_ptr(),
                                  (g_ptr if g_ptr is not None else guidance.data_ptr()) if ge else 0, ws["T1"],
                                  ws["T2"] if ge else None, x_copy, Xi, self.params.in_channels // 4, ws["H"],
                                  ws["Wd"], 1000.0)
            n += 1
        else:
            C.patchify(x_ptr, ws["TOK"], B, self.params.in_channels // 4, ws["H"], ws["Wd"], 2)
            ops.gemm(ws["TOK"], W["img_in.w"], "bias", out=Xi, bias=W["img_in.b"])
            ops.timestep_embedding(t, 256, out=ws["T1"])
            n += 3
            if ge:
                ops.timestep_embedding(guidance, 256, out=ws["T2"])
                n += 1
        ops.gemm(ctx, W["txt_in.w"], "bias", out=Xt, bias=W["txt_in.b"])
        ops.gemm(ws["T1"], W["time_in.in.w"], "silu", out=HC[:, :hid], bias=W["time_in.in.b"])
        col = hid
        n += 2
        if ge:
            ops.gemm(ws["T2"], W["guidance_in.in.w"], "silu", out=HC[:, col:col + hid], bias=W["guidance_in.in.b"])
            col += hid
            n += 1
        ops.gemm(y, W["vector_in.in.w"], "silu", out=HC[:, col:col + hid], bias=W["vector_in.in.b"])
        ops.gemm(HC, W["vec_out.w"], "silu", out=ws["SVEC"], bias=W["vec_out.b"])          # silu(vec)
        n += 2 + block_linear(W, ws["SVEC"], "mod", "bias", out=ws["MOD"])                   # all modulations
        # ---- double-stream blocks
        # Between two joint attentions the txt and img chains are independent.  Run back to back, the 512-row txt
        # GEMMs fill 24-96 of the 74 CTA-pair slots and the img GEMMs end in a partial wave; forked onto two streams
        # with disjoint SM budgets (share of SMs = share of rows) both chains finish together and every wave is full.
        dual = self.dual_stream and self.n_double > 0
        if dual:
            sms = C.num_sms()
            txt_sms = min(sms // 2, max(2, int(round(sms * Lt / float(ws["L"]) / 2.0)) * 2))
            main = torch.cuda.current_stream(self.device)
            if self._side is None:
                self._side = torch.cuda.Stream(device=self.device)
                self._ev_fork, self._ev_join = torch.cuda.Event(), torch.cuda.Event()
            side = self._side

        fused8 = self.fp8 and self.fused_quant and hid % 256 == 0

        def ln8(xs, s, sc, sh):
            """LayerNorm + modulate straight to the MXFP8 A operand of the following GEMM."""
            a8 = (ws["XM8I"], ws["XM8I_SF"]) if s == "img" else ((ws["XM8T"], ws["XM8T_SF"]) if s == "txt"
                                                                  else (ws["XM8"], ws["XM8_SF"]))
            C.layernorm_modulate_fp8(xs, a8[0], a8[1], sc, sh, 1e-6)
            return a8

        def pre(i, s, xs, xms, seq_off):
            k = ("d", i, s)
            if fused8 and f"d{i}.{s}.qkv.q" in W:
                a8 = ln8(xs, s, self._mod(ws, k, 1), self._mod(ws, k, 0))
                return 1 + block_linear(W, None, f"d{i}.{s}.qkv", "qkv_rope", a8=a8, q=Q, k=K, v=V,
                                        q_scale=W[f"d{i}.{s}.qs"], k_scale=W[f"d{i}.{s}.ks"], rope=ROPE, seq_off=seq_off)
            ops.layernorm_modulate(xs, xms, scale=self._mod(ws, k, 1), shift=self._mod(ws, k, 0))
            return 1 + block_linear(W, xms, f"d{i}.{s}.qkv", "qkv_rope", q=Q, k=K, v=V, q_scale=W[f"d{i}.{s}.qs"],
                                    k_scale=W[f"d{i}.{s}.ks"], rope=ROPE, seq_off=seq_off)

        # joint attention of the double blocks straight to MXFP8: the txt / img proj GEMMs read row ranges of ONE
        # [B, L, hid] e4m3 buffer (scale chunks: L/128 per sample, the img range starts at chunk Lt/128)
        att8 = fused8 and Lt % 128 == 0 and ws["L"] % 128 == 0 and os.environ.get("PA_FP8_ATT_PROJ", "1") != "0"
        if att8:
            sf_img = ws["XM8_SF"][(Lt // 128) * (hid // 128) * 512:]
            A8 = {"img": (ws["XM8"][:, Lt:], sf_img), "txt": (ws["XM8"][:, :Lt], ws["XM8_SF"])}

        def post(i, s, xs, xms, a, mh):
            k = ("d", i, s)
            if att8 and f"d{i}.{s}.proj.q" in W:
                m = block_linear(W, None, f"d{i}.{s}.proj", "gate_res", a8=A8[s], sfa_mtiles=ws["L"] // 128, out=xs,
                                 residual=xs, gate=self._mod(ws, k, 2))
            else:
                m = block_linear(W, a, f"d{i}.{s}.proj", "gate_res", out=xs, residual=xs, gate=self._mod(ws, k, 2))
            if fused8 and f"d{i}.{s}.mlp0.q" in W and f"d{i}.{s}.mlp2.q" in W:
                a8 = ln8(xs, s, self._mod(ws, k, 4), self._mod(ws, k, 3))
                m8 = (ws["MH8I"], ws["MH8I_SF"]) if s == "img" else (ws["MH8T"], ws["MH8T_SF"])
                m += block_linear(W, None, f"d{i}.{s}.mlp0", "gelu", a8=a8, out8=m8[0], sf8=m8[1])  # GELU + MX quant.
                m += block_linear(W, None, f"d{i}.{s}.mlp2", "gate_res", a8=m8, out=xs, residual=xs,
                                  gate=self._mod(ws, k, 5))
                return m + 1
            ops.layernorm_modulate(xs, xms, scale=self._mod(ws, k, 4), shift=self._mod(ws, k, 3))
            m += block_linear(W, xms, f"d{i}.{s}.mlp0", "gelu", out=mh)
            m += block_linear(W, mh, f"d{i}.{s}.mlp2", "gate_res", out=xs, residual=xs, gate=self._mod(ws, k, 5))
            return m + 1

        def both(f_img, f_txt):
            """img chain on the main stream, txt chain on the side stream, disjoint SM budgets; join before returning."""
            if not dual:
                return f_img() + f_txt()
            self._ev_fork.record(main)
            side.wait_event(self._ev_fork)
            try:
                with torch.cuda.stream(side):
                    C.set_sm_limit(txt_sms)
                    m = f_txt()
                    self._ev_join.record(side)
                C.set_sm_limit(sms - txt_sms)
                m += f_img()
            finally:
                C.set_sm_limit(0)
            main.wait_event(self._ev_join)
            return m

        for i in range(self.n_double):
          with nvtx_range(f"flux.double[{i}]"):
            n += both(lambda: pre(i, "img", Xi, XMi, Lt), lambda: pre(i, "txt", Xt, XMt, 0))
            if att8 and f"d{i}.img.proj.q" in W and f"d{i}.txt.proj.q" in W:
                C.attention_fp8out(Q, K, V, ws["XM8"], ws["XM8_SF"], 128 ** -0.5)
            else:
                ops.attention(Q, K, V, out=ATT)
            n += 1
            n += both(lambda: post(i, "img", Xi, XMi, ATT[:, Lt:], MH[:, Lt:]),
                      lambda: post(i, "txt", Xt, XMt, ATT[:, :Lt], MH[:, :Lt]))
        # ---- single-stream blocks
        for i in range(self.n_single):
            k = ("s", i)
            if fused8 and f"s{i}.l1.q" in W and f"s{i}.l2.q" in W:
                # linear2's A operand [attention | GELU(mlp)] is written as MXFP8 by its two producers
                c8 = (ws["CAT8"], ws["CAT8_SF"])
                a8 = ln8(X, "all", self._mod(ws, k, 1), self._mod(ws, k, 0))
                n += block_linear(W, None, f"s{i}.l1", "qkv_rope", a8=a8, q=Q, k=K, v=V, q_scale=W[f"s{i}.qs"],
                                  k_scale=W[f"s{i}.ks"], rope=ROPE, seq_off=0, out8=c8[0], sf8=c8[1], out8_col_off=hid)
                C.attention_fp8out(Q, K, V, c8[0], c8[1], 128 ** -0.5)
                n += block_linear(W, None, f"s{i}.l2", "gate_res", a8=c8, out=X, residual=X, gate=self._mod(ws, k, 2))
                n += 2
                continue
            ops.layernorm_modulate(X, XM, scale=self._mod(ws, k, 1), shift=self._mod(ws, k, 0))
            n += block_linear(W, XM, f"s{i}.l1", "qkv_rope", q=Q, k=K, v=V, q_scale=W[f"s{i}.qs"], k_scale=W[f"s{i}.ks"],
                              rope=ROPE, seq_off=0, out=CAT, mlp_col_off=hid)
            ops.attention(Q, K, V, out=ATT)
            n += block_linear(W, CAT, f"s{i}.l2", "gate_res", out=X, residual=X, gate=self._mod(ws, k, 2))
            n += 2
        # ---- final layer: AdaLN + Linear + unpatchify (+ Euler update, + peer store)
        k = ("final",)
        ops.layernorm_modulate(Xi, XMi, scale=self._mod(ws, k, 1), shift=self._mod(ws, k, 0))
        head_gather(XMi, W["final.w"], W["final.b"], self.params.out_channels // 4, ws["H"], ws["Wd"], out=out,
                    out_ptr=out_ptr, out_sample_off=out_sample_off, x_in=x_in, sigmas=sigmas)
        n += 2
        self.launches_per_step = n
        return out

    # ------------------------------------------------------------------ public entry points
    def _inputs(self, B: int, timesteps, context, y, guidance) -> tuple:
        timesteps, context = super()._inputs(B, timesteps, context)
        p, d = self.params, self.device
        if y is None:
            y = torch.zeros(B, p.vec_in_dim, device=d, dtype=torch.bfloat16)
        y = y[:, :p.vec_in_dim].to(device=d, dtype=torch.bfloat16).contiguous()
        if p.guidance_embed:
            if guidance is None:
                raise ValueError("guidance-distilled model needs a guidance strength")
            guidance = guidance.to(device=d, dtype=torch.bfloat16).contiguous()
        return timesteps, context, y, guidance

    def _prep(self, x, timesteps, context, y, guidance):
        x = x.to(device=self.device, dtype=torch.bfloat16).contiguous()
        return (x,) + self._inputs(x.shape[0], timesteps, context, y, guidance)

    @torch.no_grad()
    def forward(self, x, timesteps, context=None, y=None, guidance=None, control=None, transformer_options=None,
                **kwargs):
        """Same contract as ``models.flux.Flux.forward``: returns the velocity [B, 16, H, W]."""
        return self._forward(x, timesteps, context, y, guidance)

    @torch.no_grad()
    def forward_shard(self, x_src_ptr: int, shape, timesteps, context, out_ptr: int, out_sample_off: int, y=None,
                      guidance=None, **_ignored):
        """``DiTExecutor.forward_shard`` with the pooled text vector ``y`` and the guidance strength."""
        self._forward_shard(x_src_ptr, shape, out_ptr, out_sample_off, timesteps, context, y, guidance)

    def shard_graph_handle(self, x_src_ptr: int, shape, timesteps, context, out_ptr: int, out_sample_off: int, y=None,
                           guidance=None, **_ignored) -> int:
        return self._graph_handle(x_src_ptr, shape, out_ptr, out_sample_off, timesteps, context, y, guidance)

    @torch.no_grad()
    def denoise_step(self, x, timesteps, context, y, guidance, sigmas, out=None, out_ptr=None, out_sample_off=0,
                     x_src_ptr: Optional[int] = None, t_src_ptr: Optional[int] = None,
                     g_src_ptr: Optional[int] = None):
        """``DiTExecutor.denoise_step``; ``g_src_ptr`` lets the first kernel pull the guidance strength from a peer
        mapping as well."""
        return self._denoise(x, (timesteps, context, y, guidance), sigmas, out, out_ptr, out_sample_off, x_src_ptr,
                             t_src_ptr, g_ptr=g_src_ptr)


def build_flux_executor(model: nn.Module, device, **kw) -> FluxExecutor:
    return FluxExecutor(model, device, **kw)
