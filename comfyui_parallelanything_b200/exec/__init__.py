"""Native (hand-written sm_100a) executors, one per model family.

``builder_for(module)`` returns ``build(module, device, **kw) -> executor`` when the
wrapped module is a family we have a static kernel schedule for, else ``None`` (the
engine then falls back to a torch replica of the module).
"""
from __future__ import annotations

from typing import Callable, Optional

import torch
import torch.nn as nn


WORKSPACE_LIMIT = 6     # distinct (batch, resolution, text length) activation workspaces kept per executor


def bf16(t: torch.Tensor, device) -> torch.Tensor:
    """A weight as a contiguous bf16 tensor on ``device``, detached from the source module."""
    return t.detach().to(device=device, dtype=torch.bfloat16).contiguous()


def conditioning_sig(ctx: torch.Tensor) -> tuple:
    """Identity of a conditioning tensor: results computed from it stay valid while this is unchanged (same buffer,
    same shape, not written in place since)."""
    return (ctx.data_ptr(), tuple(ctx.shape), ctx._version)


def cache_workspace(cache: dict, key, ws: dict, device=None, on_evict: Optional[Callable] = None) -> dict:
    """Insert ``ws`` into an executor's workspace cache, evicting the least recently used entry beyond
    ``WORKSPACE_LIMIT`` (a ComfyUI session that walks through many resolutions must not pin gigabytes of activation
    buffers per shape).  ``on_evict`` lets the executor drop anything that still points into the evicted buffers
    (captured CUDA graphs); the device is synchronised first so no in-flight kernel uses them."""
    cache[key] = ws
    while len(cache) > WORKSPACE_LIMIT:
        old = next(iter(cache))
        if old == key:
            break
        if device is not None:
            if torch.cuda.is_available():
                torch.cuda.synchronize(device)
        if on_evict is not None:
            on_evict(old)
        del cache[old]
    return ws


def touch_workspace(cache: dict, key):
    """LRU hit: move ``key`` to the most-recent end and return its workspace (or None)."""
    ws = cache.get(key)
    if ws is not None and next(reversed(cache)) != key:
        cache[key] = cache.pop(key)
    return ws


def quantize_block_weights(W: dict, names, tile_of: Callable[[str], int]) -> int:
    """MXFP8-quantise the block linears ``names`` of a packed weight table in place: ``name.w`` (bf16 [N, K]) becomes
    ``name.q`` (e4m3 bytes) + ``name.sf`` (UE8M0 scale chunks grouped for the GEMM's B-tile width) + ``name.tile``.
    Shapes that are not multiples of 128 stay bf16.  Returns the number of quantised matrices."""
    from .. import ops
    n = 0
    for name in names:
        w = W.get(name + ".w")
        if w is None or w.shape[0] % 128 or w.shape[1] % 128:
            continue
        tile = tile_of(name)
        W[name + ".q"], W[name + ".sf"] = ops.quantize_mxfp8(W.pop(name + ".w"), tile)
        W[name + ".tile"] = tile
        n += 1
    return n


def block_linear(W: dict, a, name: str, mode: str, a8=None, **kw) -> int:
    """One block Linear of a DiT executor: bf16 tcgen05 GEMM, or - when ``name`` was quantised - MX-quantise the
    activation (unless the producer already emitted ``a8 = (bytes, scales)``) and run the block-scaled fp8 GEMM; same
    epilogues either way.  Returns the number of kernel launches."""
    from .. import ops
    bias = W.get(name + ".b")
    if name + ".q" in W:
        n = 1
        if a8 is None:
            a8 = ops.quantize_mxfp8(a)
            n = 3
        ops.gemm_fp8(a8[0], a8[1], W[name + ".q"], W[name + ".sf"], mode, W[name + ".tile"], bias=bias, **kw)
        return n
    ops.gemm(a, W[name + ".w"], mode, bias=bias, **kw)
    return 1


def builder_for(module: nn.Module) -> Optional[Callable]:
    """Pick the native executor for ``module`` by its STRUCTURE (attribute names + parameter shapes, as ComfyUI's
    own model classes name them - ``exec/recognize.py``), never by ``isinstance`` of this repository's oracle classes:
    the reference accepts any ``diffusion_model`` (/root/reference/any_device_parallel.py:917-930) and so do we."""
    from . import recognize
    got = recognize.identify(module)
    if got is None:
        return None
    fam, p = got
    if fam == "flux":
        if p.hidden_size // p.num_heads == 128 and p.patch_size == 2 and p.hidden_size % 128 == 0:
            from .flux_exec import build_flux_executor
            return build_flux_executor
    elif fam == "wan":
        # (in_dim, out_dim) = (36, 16): WAN2.2 image-to-video ([noise | mask | image latent]); (48, 48): WAN2.2 TI2V-5B
        # (WAN2.2 VAE latent, per-frame timesteps).  A CLIP image embedding (WAN2.1 I2V / FLF2V, Fun-InP) gets the
        # executor with the image cross-attention only when its structure is complete; anything else with ``img_emb``
        # keeps the torch replica, which must not drop ``clip_fea``
        from .wan_exec import WAN_CHANNELS
        if (p.dim // p.num_heads == 128 and tuple(p.patch_size) == (1, 2, 2)
                and (p.in_dim, p.out_dim) in WAN_CHANNELS):
            if not p.has_img_emb and not p.img_cross_attn:
                from .wan_exec import build_wan_executor
                return build_wan_executor
            if p.clip_ok and p.clip_dim % 64 == 0:
                from .wan_exec import build_wan_clip_executor
                return build_wan_clip_executor
    elif fam == "zimage":
        if p.dim // p.n_heads == 128 and p.patch_size == 2 and p.in_channels == 16 and p.ffn_hidden % 32 == 0:
            from .zimage_exec import build_zimage_executor
            return build_zimage_executor
    elif fam == "vae":
        from .vae_exec import build_vae_executor
        return build_vae_executor
    elif fam == "unet":
        if p.supported:
            from .unet_exec import build_unet_executor
            return build_unet_executor
    return None


def family_of(module: nn.Module) -> Optional[str]:
    from . import recognize
    got = recognize.identify(module)
    return got[0] if got else None
