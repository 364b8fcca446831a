"""Python surface of the native sm_100a library (``_C.so``, built in-tree by
``tools/build.py`` / ``__graft_entry__.build()``).

On a machine with a CUDA device the extension is mandatory: ``require()`` raises if
it cannot be loaded — there is deliberately no silent eager fallback for the native
executors.  On the GPU-less dev box the import is attempted too (it links against
libtorch only), so build breakage is caught by the CPU test-suite.
"""
from __future__ import annotations

import importlib
import os
from typing import Optional

import torch

_C = None
_err: Optional[BaseException] = None
try:  # noqa: SIM105
    _C = importlib.import_module(__name__ + "._C")
except BaseException as e:  # pragma: no cover - depends on build state
    _err = e


def available() -> bool:
    return _C is not None


def load_error() -> Optional[BaseException]:
    return _err


def require():
    if _C is None:
        raise RuntimeError(
            "comfyui_parallelanything_b200 native library is not built/loaded "
            f"({_err!r}); run `python tools/build.py` (or __graft_entry__.build())")
    return _C


def native_ok(device) -> bool:
    """True when ``device`` is a Blackwell (sm_100) GPU and the library is loaded."""
    if _C is None or not torch.cuda.is_available():
        return False
    d = torch.device(device)
    if d.type != "cuda":
        return False
    return torch.cuda.get_device_capability(d)[0] == 10


EPI = {
    "bias": 0, "gelu": 1, "silu": 2, "gate_res": 3, "qkv_rope": 4, "euler_unpatch": 5, "geglu": 6, "res": 7, "bias_bcast": 8, "swiglu": 9,
    "gelu_erf": 10,     # exact erf GELU (nn.GELU()); "gelu" is the tanh approximation
}


def gemm(a: torch.Tensor, w: torch.Tensor, mode: str = "bias", **kw) -> None:
    """``out = epilogue(a @ w.T)`` on tcgen05 tensor cores.  ``a``: [M,K] or [B,rows,K] view
    (last dim contiguous), ``w``: [N,K].  See csrc/bind.cpp for the keyword arguments; ``gate_res`` with
    ``gate_rows=`` / ``gate_row_off=`` reads one gate row per group of rows, like ``layernorm_modulate``'s
    ``mod_rows``."""
    require().gemm(a, w, EPI[mode], **kw)


def pack_conv_weight(w: torch.Tensor) -> torch.Tensor:
    """OIHW conv weight -> [Cout_pad32, taps * Cin_pad64] bf16, tap-major (kh, kw), zero padded — the
    K-major B operand of the implicit-GEMM convolution."""
    co, ci, kh, kw = w.shape
    cpad = (ci + 63) // 64 * 64
    copad = (co + 31) // 32 * 32
    out = torch.zeros(copad, kh * kw, cpad, dtype=torch.bfloat16, device=w.device)
    out[:co, :, :ci] = w.permute(0, 2, 3, 1).reshape(co, kh * kw, ci).to(torch.bfloat16)
    return out.reshape(copad, kh * kw * cpad).contiguous()


def pack_conv_in_weight(w: torch.Tensor) -> torch.Tensor:
    """OIHW 3x3 weight of a UNet's first convolution -> [Cout, 64] bf16, k = tap*Cin + c (tap-major, zero padded):
    the B operand of the fused scatter + conv_in kernel (csrc/comm/scatter_conv.cu), which builds the matching
    im2col rows from the lead GPU's NCHW latent."""
    co, ci, kh, kw = w.shape
    if (kh, kw) != (3, 3) or 9 * ci > 64:
        raise ValueError("fused conv_in needs a 3x3 kernel with 9*Cin <= 64")
    out = torch.zeros(co, 64, dtype=torch.bfloat16, device=w.device)
    out[:, :9 * ci] = w.permute(0, 2, 3, 1).reshape(co, 9 * ci).to(torch.bfloat16)
    return out.contiguous()


def conv2d_nhwc(x: torch.Tensor, w_packed: torch.Tensor, taps: int, stride: int = 1, mode: str = "bias",
                out: Optional[torch.Tensor] = None, **kw) -> torch.Tensor:
    """3x3 (pad 1) or 1x1 convolution on NHWC bf16 as an implicit GEMM on tcgen05 (TMA does the im2col:
    shifted 4-D boxes, zero padding from out-of-bounds fill).  Returns [N, Ho*Wo, Cout_pad]."""
    n, h, wd, _ = x.shape
    pad, k = (1, 3) if taps == 9 else (0, 1)
    ho, wo = (h + 2 * pad - k) // stride + 1, (wd + 2 * pad - k) // stride + 1
    if out is None:
        out = torch.empty(n, ho * wo, w_packed.shape[0], dtype=torch.bfloat16, device=x.device)
    require().conv(x, w_packed, taps, stride, EPI[mode], out=out, **kw)
    return out


def linear(a: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor] = None, act: str = "bias",
           out: Optional[torch.Tensor] = None) -> torch.Tensor:
    if out is None:
        out = torch.empty(a.shape[:-1] + (w.shape[0],), dtype=torch.bfloat16, device=a.device)
    gemm(a, w, act, out=out, bias=bias)
    return out


def layernorm_modulate(x, out=None, scale=None, shift=None, gamma=None, beta=None, eps: float = 1e-6,
                       mod_rows: int = 0, mod_row_off: int = 0):
    """``out = LayerNorm(x) [* gamma + beta] * (1 + scale) + shift`` per row; ``scale`` / ``shift``: per-sample [B, D]
    views.  ``mod_rows`` > 0: [G, D] views with one vector per group of ``mod_rows`` rows instead (a video frame's
    tokens); row r of sample b reads vector ``(b * rows + r + mod_row_off) // mod_rows``."""
    if out is None:
        out = torch.empty_like(x)
    require().layernorm_modulate(x, out, scale, shift, gamma, beta, eps, mod_rows, mod_row_off)
    return out


def rmsnorm_modulate(x, out=None, weight=None, scale=None, gate=None, residual=None, eps: float = 1e-5,
                     tanh_gate: bool = True):
    """``out = [residual +] [tanh](gate) * rms(x) * weight * (1 + scale)`` per row (NextDiT / Z-Image blocks);
    ``scale`` / ``gate``: per-sample [B, D] views.  ``out`` may alias ``residual``."""
    if out is None:
        out = torch.empty_like(x)
    require().rmsnorm_mod(x, out, weight, scale, gate, residual, eps, tanh_gate)
    return out


def interleave_glu(wa: torch.Tensor, wg: torch.Tensor) -> torch.Tensor:
    """Row-interleave value / gate projection weights (or biases) in groups of 32 for the ``geglu`` / ``swiglu``
    GEMM epilogues: output column n/2 = a * act(g)."""
    half = wa.shape[0]
    if wa.dim() == 1:
        return torch.stack([wa.view(half // 32, 32), wg.view(half // 32, 32)], 1).reshape(2 * half).contiguous()
    k = wa.shape[1]
    return torch.stack([wa.view(half // 32, 32, k), wg.view(half // 32, 32, k)], 1).reshape(2 * half, k).contiguous()


def timestep_embedding(t: torch.Tensor, dim: int = 256, time_factor: float = 1000.0, max_period: float = 10000.0,
                       out: Optional[torch.Tensor] = None) -> torch.Tensor:
    if out is None:
        out = torch.empty(t.shape[0], dim, dtype=torch.bfloat16, device=t.device)
    require().timestep_embedding(t, out, time_factor, max_period)
    return out


ATTENTION_VARIANT = int(os.environ.get("PA_ATTENTION", "2"))    # 1: one query tile per CTA, 2: ping-pong (two)


def attention(q, k, v, out=None, scale: Optional[float] = None, variant: Optional[int] = None, kv2=None):
    """q,k,v: [B,H,L,D] bf16 views (D = 64 / 128, innermost contiguous) -> out [B, Lq, H*D].

    ``kv2 = (k2, v2)``: a second key/value source ([B, H, Lk2, 128] views, head dim 128 only); the result is then
    ``softmax(q k^T) v + softmax(q k2^T) v2``, computed in one launch of the two-source ping-pong kernel whatever
    ``variant`` / ``PA_ATTENTION`` select (WAN2.1 image-to-video: text plus CLIP image cross-attention)."""
    b, h, lq, d = q.shape
    if out is None:
        out = torch.empty(b, lq, h * d, dtype=torch.bfloat16, device=q.device)
    k2, v2 = kv2 if kv2 is not None else (None, None)
    require().attention(q, k, v, out, float(scale if scale is not None else d ** -0.5),
                        ATTENTION_VARIANT if variant is None else variant, k2, v2)
    return out


def groupnorm_silu(x_nhwc, gamma, beta, groups: int = 32, eps: float = 1e-5, silu: bool = True, out=None):
    if out is None:
        out = torch.empty_like(x_nhwc)
    require().groupnorm_silu(x_nhwc, out, gamma, beta, groups, eps, silu)
    return out


# ----------------------------------------------------------------------------- MXFP8 (block-scaled fp8)
def quantize_mxfp8(x: torch.Tensor, tile_rows: int = 128):
    """bf16 [.., rows, K] -> (e4m3 bytes, UE8M0 scale chunks) for the block-scaled tcgen05 GEMM (K % 128 == 0).
    ``tile_rows``: 128 for activations; for weights the B-tile width the GEMM will use (224 generic / 256 QKV)."""
    q, sf = require().quantize_mxfp8(x, tile_rows)
    return q, sf


def dequantize_mxfp8(q: torch.Tensor, sf: torch.Tensor, tile_rows: int = 128) -> torch.Tensor:
    """Reference decode of ``quantize_mxfp8`` output (fp32), used by the numerics checks."""
    if q.dim() == 2:
        q = q.unsqueeze(0)
    b, rows, k = q.shape
    cpt, kc = (tile_rows + 127) // 128, k // 128
    tiles = (rows + tile_rows - 1) // tile_rows
    e = sf.view(b, tiles, cpt, kc, 32, 4, 4).permute(0, 1, 2, 5, 4, 3, 6).reshape(b, tiles, cpt * 128, kc * 4)
    e = e[:, :, :tile_rows].reshape(b, tiles * tile_rows, kc * 4)[:, :rows].float() - 127.0
    vals = q.view(torch.float8_e4m3fn).float().view(b, rows, k // 32, 32)
    return (vals * torch.exp2(e)[..., None]).reshape(b, rows, k)


def gemm_fp8(a_q, sfa, w_q, sfb, mode: str = "bias", w_tile: int = 224, **kw) -> None:
    """Block-scaled fp8 GEMM: same epilogues / keyword arguments as ``gemm`` (bf16 outputs).  ``w_tile`` must be
    the ``tile_rows`` the weight was quantised with (224 generic, 256 for the fused QKV epilogue)."""
    require().gemm_fp8(a_q, sfa, w_q, sfb, EPI[mode], w_tile, **kw)
