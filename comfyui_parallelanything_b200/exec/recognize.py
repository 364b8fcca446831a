"""Structural recognition of the model families that have a native sm_100a executor.

The reference wraps *whatever* ``diffusion_model`` it is handed (/root/reference/any_device_parallel.py:917-930) and
clones it by harvesting constructor arguments from well-known attribute names (ADP:284-350).  A native executor needs
more: the layer graph itself.  So the module is recognised by its **structure** — the attribute names and parameter
shapes ComfyUI's own model code uses (``double_blocks.N.img_attn.qkv.weight``, ``blocks.N.self_attn.norm_q.weight``,
``input_blocks.N.1.transformer_blocks.M.attn2.to_k.weight`` ...) — never by ``isinstance`` of this repository's
oracle classes.  A ``comfy.ldm.flux.model.Flux`` / ``comfy.ldm.wan.model.WanModel`` / ``comfy.ldm.lumina.model.NextDiT``
/ ``comfy.ldm.modules.diffusionmodules.openaimodel.UNetModel`` therefore gets the same native replicas as the
repository's own definitions, and anything that does not match falls back to a torch replica.

``identify(module)`` returns ``(family, params)`` or ``None``; ``params`` is a ``SimpleNamespace`` with exactly the
fields the executors read, derived from the weights (and cross-checked against ``module.params`` / module attributes
where those exist, because a few hyper-parameters — RoPE theta, axes split, eps — leave no trace in a weight shape).
"""
from __future__ import annotations

from types import SimpleNamespace
from typing import Any, Optional, Tuple

import torch
import torch.nn as nn


def _is_list(m: Any) -> bool:
    return isinstance(m, (nn.ModuleList, nn.Sequential)) and len(m) > 0


def _w(m: Any) -> Optional[torch.Tensor]:
    w = getattr(m, "weight", None)
    return w if isinstance(w, torch.Tensor) else None


def _has_linear(m: Any) -> bool:
    w = _w(m)
    return w is not None and w.dim() == 2


def norm_scale(m: Any) -> torch.Tensor:
    """RMSNorm scale parameter: ComfyUI's FLUX layers call it ``scale``, its generic ops (and WAN / NextDiT) ``weight``."""
    s = getattr(m, "scale", None)
    if isinstance(s, torch.Tensor):
        return s
    w = getattr(m, "weight", None)
    if isinstance(w, torch.Tensor):
        return w
    raise AttributeError(f"{type(m).__name__} has neither .scale nor .weight")


def _hint(module: Any, *names: str, default: Any = None) -> Any:
    """Hyper-parameter that cannot be read off a weight shape: look in ``module.params`` (dataclass / dict /
    namespace), then on the module itself (ComfyUI's WAN / NextDiT keep them as attributes)."""
    for holder in (getattr(module, "params", None), getattr(module, "config", None), module):
        if holder is None:
            continue
        for n in names:
            v = holder.get(n) if isinstance(holder, dict) else getattr(holder, n, None)
            if v is not None and not isinstance(v, (nn.Module, torch.Tensor)) and not callable(v):
                return v
    return default


# --------------------------------------------------------------------------------------------- FLUX (MM-DiT)
def _flux(m: nn.Module) -> Optional[SimpleNamespace]:
    need = ("img_in", "txt_in", "time_in", "vector_in", "double_blocks", "single_blocks", "final_layer")
    if not all(hasattr(m, a) for a in need):
        return None
    if not (_is_list(m.double_blocks) and _is_list(m.single_blocks) and _has_linear(m.img_in) and _has_linear(m.txt_in)):
        return None
    d0, s0 = m.double_blocks[0], m.single_blocks[0]
    try:
        ok = (_has_linear(d0.img_attn.qkv) and _has_linear(d0.txt_attn.proj) and _has_linear(d0.img_mod.lin)
              and _has_linear(d0.img_mlp[0]) and _has_linear(d0.img_mlp[2]) and _has_linear(s0.linear1)
              and _has_linear(s0.linear2) and _has_linear(s0.modulation.lin) and _has_linear(m.final_layer.linear)
              and _has_linear(m.final_layer.adaLN_modulation[1]) and _has_linear(m.time_in.in_layer)
              and _has_linear(m.vector_in.out_layer))
        head_dim = int(norm_scale(d0.img_attn.norm.query_norm).shape[0])
    except (AttributeError, IndexError, TypeError):
        return None
    if not ok:
        return None
    hidden = int(m.img_in.weight.shape[0])
    if d0.img_attn.qkv.weight.shape != (3 * hidden, hidden) or hidden % head_dim:
        return None
    mlp = int(d0.img_mlp[0].weight.shape[0])
    if s0.linear1.weight.shape[0] != 3 * hidden + mlp or s0.linear2.weight.shape[1] != hidden + mlp:
        return None
    if d0.img_mod.lin.weight.shape[0] != 6 * hidden or s0.modulation.lin.weight.shape[0] != 3 * hidden:
        return None
    in_ch = int(m.img_in.weight.shape[1])
    patch = int(_hint(m, "patch_size", default=2))
    g = getattr(m, "guidance_in", None)
    guidance = g is not None and hasattr(g, "in_layer") and _has_linear(g.in_layer)
    axes = list(_hint(m, "axes_dim", default=[head_dim - 2 * (7 * head_dim // 16), 7 * head_dim // 16, 7 * head_dim // 16]))
    return SimpleNamespace(
        in_channels=in_ch, out_channels=int(m.final_layer.linear.weight.shape[0]), vec_in_dim=int(m.vector_in.in_layer.weight.shape[1]),
        context_in_dim=int(m.txt_in.weight.shape[1]), hidden_size=hidden, mlp_ratio=mlp / hidden,
        num_heads=hidden // head_dim, depth=len(m.double_blocks), depth_single_blocks=len(m.single_blocks),
        axes_dim=axes, theta=int(_hint(m, "theta", default=10_000)), patch_size=patch,
        qkv_bias=d0.img_attn.qkv.bias is not None, guidance_embed=bool(guidance))


# --------------------------------------------------------------------------------------------- WAN2.x video DiT
def _wan(m: nn.Module) -> Optional[SimpleNamespace]:
    need = ("patch_embedding", "text_embedding", "time_embedding", "time_projection", "blocks", "head")
    if not all(hasattr(m, a) for a in need) or not _is_list(m.blocks):
        return None
    pe = _w(m.patch_embedding)
    if pe is None or pe.dim() != 5:
        return None
    b0 = m.blocks[0]
    try:
        ok = (_has_linear(b0.self_attn.q) and _has_linear(b0.self_attn.o) and _has_linear(b0.cross_attn.k)
              and _has_linear(b0.ffn[0]) and _has_linear(b0.ffn[2]) and isinstance(b0.modulation, torch.Tensor)
              and _has_linear(m.head.head) and isinstance(m.head.modulation, torch.Tensor)
              and _has_linear(m.text_embedding[0]) and _has_linear(m.time_embedding[0])
              and _has_linear(m.time_projection[1]) and norm_scale(b0.self_attn.norm_q) is not None
              and _w(b0.norm3) is not None)
    except (AttributeError, IndexError, TypeError):
        return None
    if not ok:
        return None
    dim = int(pe.shape[0])
    heads = _hint(m, "num_heads")
    if heads is None:
        heads = getattr(b0.self_attn, "num_heads", None) or dim // 128
    patch = tuple(int(v) for v in pe.shape[2:])
    out_dim = int(m.head.head.weight.shape[0]) // (patch[0] * patch[1] * patch[2])
    clip_dim, clip_pos, clip_ok = _wan_clip(m, dim)
    return SimpleNamespace(
        in_dim=int(pe.shape[1]), out_dim=out_dim, dim=dim, ffn_dim=int(b0.ffn[0].weight.shape[0]), num_heads=int(heads),
        num_layers=len(m.blocks), text_dim=int(m.text_embedding[0].weight.shape[1]),
        text_len=int(_hint(m, "text_len", default=512)), freq_dim=int(m.time_embedding[0].weight.shape[1]),
        patch_size=patch, eps=float(_hint(m, "eps", default=1e-6)),
        # CLIP image projection of WAN2.1 I2V / FLF2V and the Fun models: their blocks add an image cross-attention
        has_img_emb=getattr(m, "img_emb", None) is not None,
        # clip_ok: ``img_emb.proj`` is exactly LayerNorm, Linear, GELU, Linear, LayerNorm and every block's cross-attention
        # has ``k_img`` / ``v_img`` / ``norm_k_img`` - the structure the native image cross-attention implements
        clip_dim=clip_dim, clip_pos_tokens=clip_pos, clip_ok=clip_ok,
        img_cross_attn=any(hasattr(blk.cross_attn, "k_img") for blk in m.blocks))


def _wan_clip(m: nn.Module, dim: int) -> Tuple[int, int, bool]:
    """(clip_dim, clip_pos_tokens, complete) of WAN's CLIP image branch; (0, 0, False) when there is none."""
    emb = getattr(m, "img_emb", None)
    proj = getattr(emb, "proj", None)
    if emb is None or not isinstance(proj, nn.Sequential) or len(proj) != 5:
        return 0, 0, False
    n0, l1, act, l3, n4 = proj
    if not (isinstance(n0, nn.LayerNorm) and isinstance(n4, nn.LayerNorm) and isinstance(act, nn.GELU)
            and getattr(act, "approximate", "none") == "none" and _has_linear(l1) and _has_linear(l3)
            and n0.elementwise_affine and n4.elementwise_affine):
        return 0, 0, False
    clip_dim = int(l1.weight.shape[1])
    if (tuple(n0.weight.shape) != (clip_dim,) or tuple(l1.weight.shape) != (clip_dim, clip_dim)
            or tuple(l3.weight.shape) != (dim, clip_dim) or tuple(n4.weight.shape) != (dim,)):
        return 0, 0, False
    pos = getattr(emb, "emb_pos", None)
    clip_pos = 0
    if isinstance(pos, torch.Tensor):
        if pos.dim() != 3 or pos.shape[2] != clip_dim:
            return 0, 0, False
        clip_pos = int(pos.shape[1])
    for blk in m.blocks:
        ca = blk.cross_attn
        if not (_has_linear(getattr(ca, "k_img", None)) and _has_linear(getattr(ca, "v_img", None))
                and isinstance(getattr(ca, "norm_k_img", None), nn.Module)
                and tuple(ca.k_img.weight.shape) == (dim, dim) and tuple(ca.v_img.weight.shape) == (dim, dim)
                and ca.k_img.bias is not None and ca.v_img.bias is not None
                and tuple(norm_scale(ca.norm_k_img).shape) == (dim,)):
            return clip_dim, clip_pos, False
    return clip_dim, clip_pos, True


# --------------------------------------------------------------------------------------------- Z-Image / NextDiT
def _zimage(m: nn.Module) -> Optional[SimpleNamespace]:
    need = ("x_embedder", "cap_embedder", "t_embedder", "noise_refiner", "context_refiner", "layers", "final_layer")
    if not all(hasattr(m, a) for a in need) or not _is_list(m.layers) or not _has_linear(m.x_embedder):
        return None
    l0 = m.layers[0]
    try:
        ok = (_has_linear(l0.attention.qkv) and _has_linear(l0.attention.out) and _has_linear(l0.feed_forward.w1)
              and _has_linear(l0.feed_forward.w2) and _has_linear(l0.feed_forward.w3)
              and _has_linear(l0.adaLN_modulation[1]) and _has_linear(m.cap_embedder[1])
              and _has_linear(m.t_embedder.mlp[0]) and _has_linear(m.t_embedder.mlp[2])
              and _has_linear(m.final_layer.linear) and _has_linear(m.final_layer.adaLN_modulation[1])
              and all(_w(getattr(l0, n)) is not None for n in ("attention_norm1", "attention_norm2", "ffn_norm1",
                                                               "ffn_norm2")))
        head_dim = int(norm_scale(l0.attention.q_norm).shape[0])
    except (AttributeError, IndexError, TypeError):
        return None
    if not ok:
        return None
    dim = int(m.x_embedder.weight.shape[0])
    if l0.attention.qkv.weight.shape[0] != 3 * dim or dim % head_dim:      # GQA variants are not covered
        return None
    patch = int(_hint(m, "patch_size", default=2))
    in_ch = int(m.x_embedder.weight.shape[1]) // (patch * patch)
    hd = head_dim
    return SimpleNamespace(
        patch_size=patch, in_channels=in_ch, dim=dim, n_layers=len(m.layers),
        n_refiner_layers=len(m.noise_refiner), n_heads=dim // head_dim, ffn_hidden=int(l0.feed_forward.w1.weight.shape[0]),
        norm_eps=float(_hint(m, "norm_eps", "eps", default=1e-5)), cap_feat_dim=int(m.cap_embedder[1].weight.shape[1]),
        axes_dims=list(_hint(m, "axes_dims", default=[hd // 4, 3 * hd // 8, 3 * hd // 8])),
        rope_theta=float(_hint(m, "rope_theta", default=256.0)), t_scale=float(_hint(m, "t_scale", "time_scale", default=1000.0)),
        adaln_dim=int(m.t_embedder.mlp[2].weight.shape[0]))


# --------------------------------------------------------------------------------------------- SD / SDXL UNet
def is_resblock(layer: Any) -> bool:
    return all(hasattr(layer, a) for a in ("in_layers", "emb_layers", "out_layers", "skip_connection"))


def is_spatial_transformer(layer: Any) -> bool:
    return all(hasattr(layer, a) for a in ("norm", "proj_in", "transformer_blocks", "proj_out"))


def is_downsample(layer: Any) -> bool:
    return isinstance(getattr(layer, "op", None), nn.Conv2d)


def is_upsample(layer: Any) -> bool:
    return isinstance(getattr(layer, "conv", None), nn.Conv2d) and not is_resblock(layer)


def _unet(m: nn.Module) -> Optional[SimpleNamespace]:
    need = ("input_blocks", "middle_block", "output_blocks", "time_embed", "out")
    if not all(hasattr(m, a) for a in need) or not _is_list(m.input_blocks) or not _is_list(m.output_blocks):
        return None
    try:
        conv_in = m.input_blocks[0][0]
        if not isinstance(conv_in, nn.Conv2d) or not _has_linear(m.time_embed[0]) or not isinstance(m.out[-1], nn.Conv2d):
            return None
    except (IndexError, TypeError):
        return None
    ctx_dim, heads_ok, n_res = None, True, 0
    for blocks in (m.input_blocks, [m.middle_block], m.output_blocks):
        for seq in blocks:
            for layer in (seq if isinstance(seq, (nn.Sequential, nn.ModuleList)) else [seq]):
                if is_resblock(layer):
                    n_res += 1
                elif is_spatial_transformer(layer):
                    for tb in layer.transformer_blocks:
                        if not all(hasattr(tb, a) for a in ("attn1", "attn2", "ff", "norm1", "norm2", "norm3")):
                            return None
                        a2 = tb.attn2
                        dh = getattr(a2, "dim_head", None)
                        if dh is None:
                            heads = getattr(a2, "heads", None)
                            dh = a2.to_q.weight.shape[0] // heads if heads else None
                        if dh not in (64, 128):
                            heads_ok = False
                        ctx_dim = int(a2.to_k.weight.shape[1])
                elif isinstance(layer, nn.Conv2d) or is_downsample(layer) or is_upsample(layer):
                    pass
                else:
                    return None
    if n_res == 0:
        return None
    for gn in m.modules():
        if isinstance(gn, nn.GroupNorm) and gn.num_channels % 32:
            heads_ok = False
    label = getattr(m, "label_emb", None)
    adm = None
    if label is not None:
        try:
            adm = int(label[0][0].weight.shape[1])
        except (IndexError, TypeError, AttributeError):
            adm = None
    return SimpleNamespace(
        model_channels=int(conv_in.weight.shape[0]), in_channels=int(conv_in.weight.shape[1]),
        out_channels=int(m.out[-1].weight.shape[0]), adm_in_channels=adm, context_dim=ctx_dim, supported=heads_ok)


# --------------------------------------------------------------------------------------------- SD VAE decoder
def _vae(m: nn.Module) -> Optional[SimpleNamespace]:
    need = ("conv_in", "mid", "up", "norm_out", "conv_out")
    if not all(hasattr(m, a) for a in need) or not isinstance(m.conv_in, nn.Conv2d):
        return None
    return SimpleNamespace(z_channels=int(m.conv_in.weight.shape[1]), out_channels=int(m.conv_out.weight.shape[0]))


_FAMILIES = (("flux", _flux), ("wan", _wan), ("zimage", _zimage), ("unet", _unet), ("vae", _vae))


def identify(module: nn.Module) -> Optional[Tuple[str, SimpleNamespace]]:
    """(family, derived params) if ``module`` has the layer structure of a supported family, else None."""
    if not isinstance(module, nn.Module):
        return None
    for fam, fn in _FAMILIES:
        try:
            p = fn(module)
        except Exception:               # a foreign module with surprising attribute types is simply "not ours"
            p = None
        if p is not None:
            return fam, p
    return None


def params_of(module: nn.Module, family: str) -> SimpleNamespace:
    """Derived params of ``module`` for ``family`` (raises if the structure does not match)."""
    got = identify(module)
    if got is None or got[0] != family:
        raise ValueError(f"{type(module).__name__} does not have the structure of a {family} model")
    return got[1]
