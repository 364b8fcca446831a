"""SDXL-class latent-diffusion UNet on hand-written sm_100a kernels (channels-last bf16 end to end).

What stock torch runs behind the reference's ``forward_fn(...)`` (/root/reference/any_device_parallel.py:1390)
as cuDNN convs + ATen GroupNorm/SiLU/LayerNorm + SDPA + many elementwise kernels becomes:

  * every 3x3 / 1x1 convolution = the tcgen05 implicit GEMM (TMA does the im2col with shifted 4-D boxes,
    zero padding from out-of-bounds fill, stride-2 via TMA element strides); the time-embedding add
    (``bias_bcast``), the ResBlock skip add and the transformer residuals (``res``) are GEMM epilogues;
  * GroupNorm(+SiLU) is one fused NHWC kernel pair; LayerNorm reuses the AdaLN kernel (affine, no mod);
  * attention (head_dim 64) reads q/k/v straight from the fused QKV GEMM output through strided 4-D TMA
    views; cross-attention K/V of the (step-invariant) text context are one GEMM per layer;
  * GEGLU is a GEMM epilogue over row-interleaved weights;
  * all ResBlock time-embedding projections are ONE GEMM over the concatenated weights;
  * the gather (``denoise_step``): NHWC eps -> CFG (cond/uncond pairs kept on one rank) -> Euler ->
    NCHW store straight into the lead GPU's buffer.
Head dims other than 64/128 (SD1.5: 40/80/160) are not covered — the engine then uses a torch replica.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Tuple

import torch
import torch.nn as nn

from .. import ops
from . import bf16 as _bf, conditioning_sig, recognize
from .graphs import GraphCache


def _pad32(t: torch.Tensor) -> torch.Tensor:
    n = t.shape[0]
    m = (n + 31) // 32 * 32
    if m == n:
        return t
    out = torch.zeros((m,) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
    out[:n] = t
    return out


class _Conv:
    def __init__(self, m: nn.Conv2d, d):
        self.taps = m.kernel_size[0] * m.kernel_size[1]
        self.stride = m.stride[0]
        self.cout = m.out_channels
        self.w = ops.pack_conv_weight(m.weight.detach().to(d))
        self.b = _pad32(_bf(m.bias, d)) if m.bias is not None else None

    def __call__(self, x4: torch.Tensor, mode: str = "bias", **kw) -> torch.Tensor:
        return ops.conv2d_nhwc(x4, self.w, self.taps, self.stride, mode, bias=self.b, **kw)


class _Lin:
    def __init__(self, m: nn.Linear, d):
        self.w = _bf(m.weight, d)
        self.b = _bf(m.bias, d) if m.bias is not None else None

    def __call__(self, x: torch.Tensor, mode: str = "bias", out: Optional[torch.Tensor] = None, **kw) -> torch.Tensor:
        if out is None:
            out = torch.empty(x.shape[:-1] + (self.w.shape[0],), dtype=torch.bfloat16, device=x.device)
        ops.gemm(x, self.w, mode, out=out, bias=self.b, **kw)
        return out


class _GN:
    def __init__(self, m: nn.GroupNorm, d):
        self.g, self.b, self.groups, self.eps = _bf(m.weight, d), _bf(m.bias, d), m.num_groups, m.eps

    def __call__(self, x3: torch.Tensor, silu: bool) -> torch.Tensor:
        return ops.groupnorm_silu(x3, self.g, self.b, self.groups, self.eps, silu)


class _LN:
    def __init__(self, m: nn.LayerNorm, d):
        self.g, self.b, self.eps = _bf(m.weight, d), _bf(m.bias, d), m.eps

    def __call__(self, x3: torch.Tensor) -> torch.Tensor:
        return ops.layernorm_modulate(x3, gamma=self.g, beta=self.b, eps=self.eps)


class _Res:
    def __init__(self, m: nn.Module, d, emb_off: int):
        self.gn1, self.conv1 = _GN(m.in_layers[0], d), _Conv(m.in_layers[2], d)
        self.gn2, self.conv2 = _GN(m.out_layers[0], d), _Conv(m.out_layers[3], d)
        self.skip = None if isinstance(m.skip_connection, nn.Identity) else _Conv(m.skip_connection, d)
        self.emb_off, self.cout = emb_off, self.conv1.cout

    def __call__(self, x3, hw, emb_all):
        b, (h, w) = x3.shape[0], hw
        t = self.gn1(x3, True)
        t = self.conv1(t.view(b, h, w, -1), "bias_bcast", gate=emb_all[:, self.emb_off:self.emb_off + self.cout])
        t = self.gn2(t, True)
        skip = x3 if self.skip is None else self.skip(x3.view(b, h, w, -1))
        return self.conv2(t.view(b, h, w, -1), "res", residual=skip)


class _TBlock:
    def __init__(self, m: nn.Module, d):
        a1, a2 = m.attn1, m.attn2
        self.heads, self.dh = a1.heads, a1.dim_head
        self.ln1, self.ln2, self.ln3 = _LN(m.norm1, d), _LN(m.norm2, d), _LN(m.norm3, d)
        self.wqkv = torch.cat([_bf(a1.to_q.weight, d), _bf(a1.to_k.weight, d), _bf(a1.to_v.weight, d)], 0).contiguous()
        self.o1 = _Lin(a1.to_out[0], d)
        self.wq2 = _bf(a2.to_q.weight, d)
        self.wkv2 = torch.cat([_bf(a2.to_k.weight, d), _bf(a2.to_v.weight, d)], 0).contiguous()
        self.o2 = _Lin(a2.to_out[0], d)
        proj = m.ff.net[0].proj
        half = proj.weight.shape[0] // 2
        wa, wg = _bf(proj.weight[:half], d), _bf(proj.weight[half:], d)
        k = wa.shape[1]
        self.wff1 = torch.stack([wa.view(half // 32, 32, k), wg.view(half // 32, 32, k)], 1).reshape(2 * half, k).contiguous()
        ba, bg = _bf(proj.bias[:half], d), _bf(proj.bias[half:], d)
        self.bff1 = torch.stack([ba.view(half // 32, 32), bg.view(half // 32, 32)], 1).reshape(2 * half).contiguous()
        self.ff2 = _Lin(m.ff.net[2], d)
        self._kv = None          # cross-attention K/V of the (step-invariant) text context
        self._kv_sig = None

    def prepare_ctx(self, ctx) -> int:
        """K/V projections of the conditioning depend only on ``ctx``: computed once per sampling run, EAGERLY (never
        inside the per-step CUDA graph, which reads the persistent ``_kv`` buffer; SURVEY K3 - the reference
        re-sends and re-projects the constant conditioning every step).  Returns the number of launches."""
        sig = conditioning_sig(ctx)
        if self._kv_sig == sig:
            return 0
        inner = self.wkv2.shape[0] // 2
        if self._kv is None or self._kv.shape[:2] != ctx.shape[:2]:
            self._kv = torch.empty(ctx.shape[0], ctx.shape[1], 2 * inner, dtype=torch.bfloat16, device=ctx.device)
        ops.gemm(ctx, self.wkv2, "bias", out=self._kv)
        self._kv_sig = sig
        return 1

    def __call__(self, h, ctx):
        b, l, inner = h.shape
        H, D = self.heads, self.dh
        e = lambda *s: torch.empty(*s, dtype=torch.bfloat16, device=h.device)  # noqa: E731
        n = self.ln1(h)
        qkv = e(b, l, 3 * inner)
        ops.gemm(n, self.wqkv, "bias", out=qkv)
        v5 = qkv.view(b, l, 3, H, D)
        a = ops.attention(v5[:, :, 0].permute(0, 2, 1, 3), v5[:, :, 1].permute(0, 2, 1, 3), v5[:, :, 2].permute(0, 2, 1, 3))
        self.o1(a, "res", out=h, residual=h)
        n = self.ln2(h)
        q = e(b, l, inner)
        ops.gemm(n, self.wq2, "bias", out=q)
        kv5 = self._kv.view(b, ctx.shape[1], 2, H, D)
        a = ops.attention(q.view(b, l, H, D).permute(0, 2, 1, 3), kv5[:, :, 0].permute(0, 2, 1, 3),
                          kv5[:, :, 1].permute(0, 2, 1, 3))
        self.o2(a, "res", out=h, residual=h)
        n = self.ln3(h)
        f = e(b, l, self.wff1.shape[0] // 2)
        ops.gemm(n, self.wff1, "geglu", out=f, bias=self.bff1)
        self.ff2(f, "res", out=h, residual=h)
        return h


class _ST:
    def __init__(self, m: nn.Module, d):
        self.gn = _GN(m.norm, d)
        if isinstance(m.proj_in, nn.Linear):
            self.pin, self.pout = _Lin(m.proj_in, d), _Lin(m.proj_out, d)
        else:       # 1x1 convs on NHWC rows are plain linears
            self.pin, self.pout = _Lin(_as_linear(m.proj_in), d), _Lin(_as_linear(m.proj_out), d)
        self.blocks = [_TBlock(b, d) for b in m.transformer_blocks]

    def __call__(self, x3, ctx):
        h = self.pin(self.gn(x3, False))
        for blk in self.blocks:
            h = blk(h, ctx)
        return self.pout(h, "res", residual=x3)


def _as_linear(conv: nn.Conv2d) -> nn.Linear:
    lin = nn.Linear(conv.in_channels, conv.out_channels, bias=conv.bias is not None)
    lin.weight = nn.Parameter(conv.weight.detach().reshape(conv.out_channels, conv.in_channels))
    if conv.bias is not None:
        lin.bias = nn.Parameter(conv.bias.detach())
    return lin


class UNetExecutor(nn.Module):
    pa_family = "unet"
    pa_native = True

    def __init__(self, model: nn.Module, device, cuda_graphs: bool = False, fp8: bool = False):
        super().__init__()
        ops.require()
        d = self.device = torch.device(device)
        p = self.params = recognize.params_of(model, "unet")        # from conv / linear shapes, not class identity
        if not p.supported:
            raise ValueError("UNetExecutor needs attention head_dim 64/128 and GroupNorm channels % 32 == 0")
        self.mc, self.in_ch, self.out_ch = p.model_channels, p.in_channels, p.out_channels
        self.adm = p.adm_in_channels
        self.ctx_dim = p.context_dim
        self.t1, self.t2 = _Lin(model.time_embed[0], d), _Lin(model.time_embed[2], d)
        if self.adm is not None:
            self.l1, self.l2 = _Lin(model.label_emb[0][0], d), _Lin(model.label_emb[0][2], d)
        emb_w, emb_b, off = [], [], 0

        def conv_layers(seq) -> List[Tuple[str, object]]:
            nonlocal off
            out = []
            for layer in seq:
                if recognize.is_resblock(layer):
                    lin = layer.emb_layers[1]
                    emb_w.append(_bf(lin.weight, d))
                    emb_b.append(_bf(lin.bias, d))
                    out.append(("res", _Res(layer, d, off)))
                    off += lin.weight.shape[0]
                elif recognize.is_spatial_transformer(layer):
                    out.append(("st", _ST(layer, d)))
                elif recognize.is_downsample(layer):
                    out.append(("down", _Conv(layer.op, d)))
                elif recognize.is_upsample(layer):
                    out.append(("up", _Conv(layer.conv, d)))
                elif isinstance(layer, nn.Conv2d):
                    out.append(("conv", _Conv(layer, d)))
                else:
                    raise TypeError(f"unsupported UNet layer {type(layer).__name__}")
            return out

        self.inp = [conv_layers(b) for b in model.input_blocks]
        self.mid = conv_layers(model.middle_block)
        self.outb = [conv_layers(b) for b in model.output_blocks]
        self.emb_w = torch.cat(emb_w, 0).contiguous()
        self.emb_b = torch.cat(emb_b, 0).contiguous()
        self.gn_out, self.conv_out = _GN(model.out[0], d), _Conv(model.out[2], d)
        self.cin_pad = (self.in_ch + 7) // 8 * 8
        # fused scatter: (peer) NCHW latent shard -> im2col -> conv_in GEMM + timestep sinusoid in ONE kernel
        # (csrc/comm/scatter_conv.cu); needs the stock first layer: a lone 3x3 / stride-1 conv over 4 latent channels
        cin = model.input_blocks[0][0]
        self.fused_in = (len(self.inp[0]) == 1 and self.inp[0][0][0] == "conv" and isinstance(cin, nn.Conv2d)
                         and cin.kernel_size == (3, 3) and cin.stride == (1, 1) and cin.padding == (1, 1)
                         and self.in_ch == 4 and self.mc % 32 == 0 and cin.bias is not None)
        if self.fused_in:
            self.cin_w = ops.pack_conv_in_weight(cin.weight.detach().to(d))
            self.cin_b = _bf(cin.bias, d)
        self.cuda_graphs = cuda_graphs
        self._graphs = GraphCache(d, enabled=cuda_graphs)
        self._tblocks: List[_TBlock] = []
        for seq in self.inp + [self.mid] + self.outb:
            for kind, op in seq:
                if kind == "st":
                    self._tblocks.extend(op.blocks)
        self._io: Dict[Tuple, dict] = {}
        self.launches_per_step = 0

    def parameters(self, recurse: bool = True):  # type: ignore[override]
        return iter(())

    def invalidate_conditioning(self) -> None:
        """Forget the cached cross-attention K/V (call when the prompt buffer is rewritten in place)."""
        for tb in self._tblocks:
            tb._kv_sig = None

    def _prepare_ctx(self, ctx) -> int:
        return sum(tb.prepare_ctx(ctx) for tb in self._tblocks)

    def _ctx_ready(self, ctx) -> bool:
        sig = conditioning_sig(ctx)
        return all(tb._kv_sig == sig for tb in self._tblocks)

    def release(self) -> None:
        self.inp, self.mid, self.outb, self._tblocks = [], [], [], []
        self._graphs.clear()
        self._io.clear()

    # ------------------------------------------------------------------ schedule
    def _seq(self, layers, h, hw, emb_all, ctx):
        C = ops.require()
        for kind, op in layers:
            b = h.shape[0]
            if kind == "res":
                h = op(h, hw, emb_all)
            elif kind == "st":
                h = op(h, ctx)
            elif kind == "conv":
                h = op(h.view(b, hw[0], hw[1], -1))
            elif kind == "down":
                h = op(h.view(b, hw[0], hw[1], -1))
                hw = ((hw[0] + 1) // 2, (hw[1] + 1) // 2)
            elif kind == "up":
                up = torch.empty(b, 2 * hw[0], 2 * hw[1], h.shape[-1], dtype=torch.bfloat16, device=h.device)
                C.upsample2x(h.view(b, hw[0], hw[1], -1), up)
                hw = (2 * hw[0], 2 * hw[1])
                h = op(up)
        return h, hw

    def _eps_nhwc(self, x_ptr: int, B: int, H: int, W: int, t, ctx, y, t_ptr: Optional[int] = None, x_copy=None):
        C = ops.require()
        d = self.device
        e = lambda *s: torch.empty(*s, dtype=torch.bfloat16, device=d)  # noqa: E731
        if self.fused_in:
            h0, temb = e(B, H * W, self.mc), e(B, self.mc)
            C.scatter_conv_in(self.cin_w, self.cin_b, x_ptr, t_ptr if t_ptr is not None else t.data_ptr(), temb, x_copy,
                              h0, self.in_ch, H, W, 1.0, 10000.0)
            first = 1
        else:
            xh = e(B, H, W, self.cin_pad)
            C.nchw_to_nhwc_pad(x_ptr, xh, B, self.in_ch, H * W)
            temb = ops.timestep_embedding(t, self.mc, time_factor=1.0)
            h0, first = xh.view(B, H * W, self.cin_pad), 0
        emb = self.t2(self.t1(temb, "silu"))
        if self.adm is not None:
            emb = self.l2(self.l1(y, "silu"), "res", residual=emb)
        semb = torch.empty_like(emb)
        C.silu(emb, semb)
        emb_all = e(B, self.emb_w.shape[0])
        ops.gemm(semb, self.emb_w, "bias", out=emb_all, bias=self.emb_b)
        hs: List[Tuple[torch.Tensor, Tuple[int, int]]] = []
        h, hw = h0, (H, W)
        if first:
            hs.append((h, hw))
        for layers in self.inp[first:]:
            h, hw = self._seq(layers, h, hw, emb_all, ctx)
            hs.append((h, hw))
        h, hw = self._seq(self.mid, h, hw, emb_all, ctx)
        for layers in self.outb:
            skip, _ = hs.pop()
            cat = e(B, hw[0] * hw[1], h.shape[-1] + skip.shape[-1])
            C.concat_channels(h, skip, cat)
            h, hw = self._seq(layers, cat, hw, emb_all, ctx)
        h = self.gn_out(h, True)
        return self.conv_out(h.view(B, hw[0], hw[1], -1))            # [B, HW, 32] (first out_ch are real)

    def _prep(self, x, timesteps, context, y):
        d = self.device
        bf = lambda t: t.to(device=d, dtype=torch.bfloat16).contiguous()  # noqa: E731
        return bf(x), bf(timesteps), bf(context), (bf(y) if y is not None else None)

    @torch.no_grad()
    def forward(self, x, timesteps=None, context=None, y=None, control=None, transformer_options=None, **kwargs):
        with torch.cuda.device(self.device):
            x, timesteps, context, y = self._prep(x, timesteps, context, y)
            B, _, H, W = x.shape
            self._prepare_ctx(context)
            eps = self._eps_nhwc(x.data_ptr(), B, H, W, timesteps, context, y)
            out = torch.empty(B, self.out_ch, H, W, dtype=torch.bfloat16, device=self.device)
            ops.require().unet_out_gather(eps, None, out.data_ptr(), None, B, self.out_ch, False, 1.0, 0, 0)
            return out

    def out_shape(self, shape) -> Tuple[int, ...]:
        """Output shape for an input of ``shape`` (in_ch and out_ch are independent, e.g. 9-channel inpaint UNets)."""
        return (shape[0], self.out_ch) + tuple(shape[2:])

    def _shard_args(self, x_src_ptr, shape, timesteps, context, out_ptr, out_sample_off, y):
        d = self.device
        bf = lambda t: t.to(device=d, dtype=torch.bfloat16).contiguous()  # noqa: E731
        timesteps, context = bf(timesteps), bf(context)
        y = bf(y) if y is not None else None
        key = ("shard", tuple(shape), x_src_ptr, timesteps.data_ptr(), context.data_ptr(), tuple(context.shape),
               y.data_ptr() if y is not None else 0, out_ptr, out_sample_off)
        return key, timesteps, context, y

    @torch.no_grad()
    def forward_shard(self, x_src_ptr: int, shape, timesteps, context, out_ptr: int, out_sample_off: int, y=None,
                      **_ignored):
        with torch.cuda.device(self.device):
            key, timesteps, context, y = self._shard_args(x_src_ptr, shape, timesteps, context, out_ptr,
                                                          out_sample_off, y)
            self._prepare_ctx(context)

            def body():
                eps = self._eps_nhwc(x_src_ptr, shape[0], shape[2], shape[3], timesteps, context, y)
                ops.require().unet_out_gather(eps, None, out_ptr, None, shape[0], self.out_ch, False, 1.0, 0,
                                              out_sample_off)
            self._graphs.run(key, body)

    def shard_graph_handle(self, x_src_ptr: int, shape, timesteps, context, out_ptr: int, out_sample_off: int, y=None,
                           **_ignored) -> int:
        with torch.cuda.device(self.device):
            key, _t, context, _y = self._shard_args(x_src_ptr, shape, timesteps, context, out_ptr, out_sample_off, y)
            if not self._ctx_ready(context):
                return 0
        return self._graphs.exec_handle(key)

    @torch.no_grad()
    def denoise_step(self, x, timesteps, context, y, sigmas, cfg_scale: float = 1.0, cfg_pairs: bool = False,
                     out=None, out_ptr: Optional[int] = None, out_sample_off: int = 0,
                     x_src_ptr: Optional[int] = None, t_src_ptr: Optional[int] = None):
        """eps forward + (CFG) + Euler update, stored NCHW into ``out`` / a peer buffer.  With ``cfg_pairs``
        the local batch is [cond(n) | uncond(n)] and ``x``/``sigmas`` describe the n samples.  With ``x_src_ptr``
        (and ``t_src_ptr``) the first kernel pulls the latent shard (and timesteps) from the lead GPU over NVLink and
        fills ``x`` with the local copy the Euler epilogue reads."""
        with torch.cuda.device(self.device):
            B, _, H, W = x.shape
            n = B // 2 if cfg_pairs else B
            if out is None and out_ptr is None:
                io = self._io.get((n, H, W))
                if io is None:
                    io = self._io[(n, H, W)] = {"OUT": torch.empty(n, self.out_ch, H, W, dtype=torch.bfloat16,
                                                                   device=self.device)}
                out = io["OUT"]
            self._prepare_ctx(context)
            pull = x_src_ptr is not None
            local_copy = x if (pull and self.fused_in and x.data_ptr() != x_src_ptr) else None
            if pull and not self.fused_in:
                raise ValueError("peer-pulled latents need the fused conv_in path (4 latent channels)")

            def body():
                eps = self._eps_nhwc(x_src_ptr if pull else x.data_ptr(), B, H, W, timesteps, context, y,
                                     t_ptr=t_src_ptr, x_copy=local_copy)
                ops.require().unet_out_gather(eps, x, out_ptr if out_ptr is not None else out.data_ptr(), sigmas, n,
                                              self.out_ch, cfg_pairs, float(cfg_scale), 1, out_sample_off)

            key = (tuple(x.shape), x.data_ptr(), timesteps.data_ptr(), context.data_ptr(), tuple(context.shape),
                   y.data_ptr() if y is not None else 0, sigmas.data_ptr(), out.data_ptr() if out is not None else 0,
                   out_ptr or 0, out_sample_off, x_src_ptr or 0, t_src_ptr or 0, bool(cfg_pairs), float(cfg_scale))
            self._graphs.run(key, body)
            return out


def build_unet_executor(model: nn.Module, device, **kw) -> UNetExecutor:
    return UNetExecutor(model, device, **kw)


def supports(model: nn.Module) -> bool:
    """Structure of an SD/SDXL-class UNet with head_dim 64/128 attention and channel counts that are multiples of 32."""
    got = recognize.identify(model)
    return got is not None and got[0] == "unet" and bool(got[1].supported)
