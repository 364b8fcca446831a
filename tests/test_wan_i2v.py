"""WAN2.2 image-to-video (36 input channels = noise | mask | image latent, 16 output channels) on the CPU: recognition,
builder choice and what the native executor packs.  The GPU side is in test_gpu_wan_i2v.py."""
import dataclasses

import torch
import torch.nn as nn

from comfyui_parallelanything_b200 import exec as native_exec
from comfyui_parallelanything_b200.exec import recognize
from comfyui_parallelanything_b200.models import wan
from comfyui_parallelanything_b200.utils.lookalike import launder


def _i2v_params():
    return dataclasses.replace(wan.wan_tiny_params(), in_dim=36)


def test_i2v_params_and_inputs():
    p = wan.wan22_i2v_a14b_params()
    assert (p.in_dim, p.out_dim) == (36, 16)
    assert dataclasses.replace(p, in_dim=16) == wan.wan22_a14b_params()
    inp = wan.i2v_inputs(_i2v_params(), 2, frames=8, height=32, width=48)
    x = inp["x"]
    assert tuple(x.shape) == (2, 36, 2, 4, 6)
    mask = x[:, 16:20].float()
    assert torch.equal(mask[:, :, 0], torch.ones_like(mask[:, :, 0]))
    assert torch.equal(mask[:, :, 1:], torch.zeros_like(mask[:, :, 1:]))


def test_i2v_model_and_lookalike_select_wan_builder():
    torch.manual_seed(0)
    m = wan.WanModel(_i2v_params())
    for mod in (m, launder(m)):
        fam, dp = recognize.identify(mod)
        assert fam == "wan" and (dp.in_dim, dp.out_dim) == (36, 16) and not dp.has_img_emb
        b = native_exec.builder_for(mod)
        assert b is not None and b.__name__ == "build_wan_executor"


def test_clip_image_embedding_keeps_torch_replica():
    """WAN2.1 I2V / FLF2V and the Fun models carry ``img_emb`` (CLIP image projection for an image cross-attention the
    executor does not implement): they must not get a native executor that would ignore ``clip_fea``."""
    for p in (_i2v_params(), wan.wan_tiny_params()):
        lm = launder(wan.WanModel(p))
        lm.img_emb = nn.Sequential(nn.LayerNorm(32), nn.Linear(32, p.dim))
        fam, dp = recognize.identify(lm)
        assert fam == "wan" and dp.has_img_emb
        assert native_exec.builder_for(lm) is None


def test_i2v_executor_packs_wide_patch_embedding():
    from comfyui_parallelanything_b200.exec.wan_exec import WanExecutor
    torch.manual_seed(0)
    p = _i2v_params()
    m = wan.WanModel(p).to(torch.bfloat16)
    ex = WanExecutor(m, "cpu")
    assert torch.equal(ex.W["patch.w"], m.patch_embedding.weight.reshape(p.dim, 144))
    assert ex.W["patch.w"].is_contiguous() and ex.W["patch.w"].stride(0) * 2 % 16 == 0   # TMA row pitch
    ws = ex.workspace(1, 2, 8, 8, 8)
    assert tuple(ws["OUT"].shape) == (1, 16, 2, 8, 8)
    assert ex.out_shape((3, 36, 2, 8, 8)) == (3, 16, 2, 8, 8)
    t2v = WanExecutor(wan.WanModel(wan.wan_tiny_params()).to(torch.bfloat16), "cpu")
    assert t2v.out_shape((3, 16, 2, 8, 8)) == (3, 16, 2, 8, 8)
