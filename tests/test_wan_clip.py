"""WAN2.1 image-to-video / first-last-frame models (CLIP image cross-attention) on the CPU: oracle semantics,
recognition, builder choice, packing, workspace shapes and the step entry points.  The GPU side is in
test_gpu_wan_clip.py and the self-checks (tests/test_gpu_kernels.py)."""
import dataclasses
import inspect

import pytest
import torch
import torch.nn as nn

from comfyui_parallelanything_b200 import exec as native_exec
from comfyui_parallelanything_b200.exec import recognize
from comfyui_parallelanything_b200.models import wan
from comfyui_parallelanything_b200.utils.lookalike import launder


def _clip_params(flf2v=False):
    return dataclasses.replace(wan.wan_tiny_params(), in_dim=36, clip_dim=128, clip_pos_tokens=514 if flf2v else 0)


def _model(flf2v=False, seed=0):
    torch.manual_seed(seed)
    return wan.WanModel(_clip_params(flf2v)).eval()


def test_param_constructors():
    p, f = wan.wan21_i2v_14b_params(), wan.wan21_flf2v_14b_params()
    assert (p.in_dim, p.out_dim, p.dim, p.num_heads, p.num_layers, p.clip_dim, p.clip_pos_tokens) == (36, 16, 5120, 40, 40,
                                                                                                      1280, 0)
    assert dataclasses.replace(f, clip_pos_tokens=0) == p and f.clip_pos_tokens == 514
    inp = wan.clip_inputs(_clip_params(True), 2, frames=8, height=32, width=48)
    assert tuple(inp["clip_fea"].shape) == (2, 514, 128) and tuple(inp["x"].shape) == (2, 36, 2, 4, 6)
    assert tuple(wan.clip_inputs(_clip_params(), 1, frames=8, height=32, width=48)["clip_fea"].shape) == (1, 257, 128)


def test_t2v_and_i2v_models_draw_the_same_random_numbers():
    torch.manual_seed(0)
    a = wan.WanModel(dataclasses.replace(wan.wan_tiny_params(), in_dim=36))
    b = _model()
    sb = b.state_dict()
    for k, v in a.state_dict().items():
        assert torch.equal(v, sb[k]), k


def test_no_clip_fea_is_the_text_as_image_branch():
    m = _model()
    inp = wan.clip_inputs(m.params, 1, frames=4, height=32, width=32, dtype=torch.float32)
    with torch.no_grad():
        got = m(inp["x"], inp["timesteps"], context=inp["context"])
        # by hand: every block's image branch attends over the embedded text
        ctx = m.text_embedding(inp["context"])
        ca = m.blocks[0].cross_attn
        x = torch.randn(1, 8, m.params.dim)
        full = ca(x, ctx, None)
        q = ca.norm_q(ca.q(x)).view(1, 8, 2, 128).transpose(1, 2)
        att = lambda k, v: torch.nn.functional.scaled_dot_product_attention(  # noqa: E731
            q, k.view(1, -1, 2, 128).transpose(1, 2), v.view(1, -1, 2, 128).transpose(1, 2))
        want = ca.o((att(ca.norm_k(ca.k(ctx)), ca.v(ctx)) + att(ca.norm_k_img(ca.k_img(ctx)), ca.v_img(ctx)))
                    .transpose(1, 2).reshape(1, 8, -1))
    assert torch.allclose(full, want, atol=1e-5)
    assert torch.isfinite(got).all()
    with torch.no_grad():
        with_clip = m(**inp)
    assert not torch.allclose(with_clip, got)


@pytest.mark.parametrize("li", [257, 514])
def test_flf2v_emb_pos_slicing(li):
    m = _model(flf2v=True)
    emb = m.img_emb
    fea = torch.randn(2, li, 128)
    with torch.no_grad():
        got = emb(fea)
        want = emb.proj(fea[:, :514] + emb.emb_pos[:, :li])
    assert got.shape == (2, li, m.params.dim) and torch.equal(got, want)
    gelu = emb.proj[2]
    assert isinstance(gelu, nn.GELU) and gelu.approximate == "none"


@pytest.mark.parametrize("flf2v", [False, True])
def test_laundered_models_select_clip_builder(flf2v):
    m = _model(flf2v)
    for mod in (m, launder(m)):
        fam, dp = recognize.identify(mod)
        assert fam == "wan" and dp.has_img_emb and dp.clip_ok
        assert (dp.clip_dim, dp.clip_pos_tokens) == (128, 514 if flf2v else 0)
        b = native_exec.builder_for(mod)
        assert b is not None and b.__name__ == "build_wan_clip_executor"


def test_partial_structures_select_nothing():
    # img_emb without k_img
    lm = launder(wan.WanModel(dataclasses.replace(wan.wan_tiny_params(), in_dim=36)))
    lm.img_emb = launder(_model()).img_emb
    assert recognize.identify(lm)[1].has_img_emb and native_exec.builder_for(lm) is None
    # k_img without img_emb
    lm = launder(_model())
    del lm.img_emb
    assert native_exec.builder_for(lm) is None
    # a proj that is not the five layers
    lm = launder(_model())
    lm.img_emb.proj = nn.Sequential(*list(lm.img_emb.proj)[:4])
    assert not recognize.identify(lm)[1].clip_ok and native_exec.builder_for(lm) is None
    # tanh GELU is not ComfyUI's MLPProj
    lm = launder(_model())
    lm.img_emb.proj[2] = nn.GELU(approximate="tanh")
    assert native_exec.builder_for(lm) is None


@pytest.mark.parametrize("flf2v", [False, True])
def test_packing_and_workspace(flf2v):
    from comfyui_parallelanything_b200.exec.wan_exec import WanClipExecutor
    m = _model(flf2v).to(torch.bfloat16)
    ex = WanClipExecutor(m, "cpu")
    proj = m.img_emb.proj
    assert torch.equal(ex.W["img.l1.w"], proj[1].weight) and torch.equal(ex.W["img.l3.b"], proj[3].bias)
    assert torch.equal(ex.W["img.n0.g"], proj[0].weight) and torch.equal(ex.W["img.n4.b"], proj[4].bias)
    assert (ex.W["img.emb_pos"] is not None) == flf2v
    if flf2v:
        assert torch.equal(ex.W["img.emb_pos"], m.img_emb.emb_pos)
    for i, blk in enumerate(m.blocks):
        ca = blk.cross_attn
        assert torch.equal(ex.W[f"b{i}.ckvi.w"], torch.cat([ca.k_img.weight, ca.v_img.weight], 0))
        assert torch.equal(ex.W[f"b{i}.ckvi.b"], torch.cat([ca.k_img.bias, ca.v_img.bias], 0))
        assert torch.equal(ex.W[f"b{i}.cnki"], ca.norm_k_img.weight)
        assert torch.equal(ex.W[f"b{i}.ckv.w"], torch.cat([ca.k.weight, ca.v.weight], 0))
    li = 514 if flf2v else 257
    ws = ex.workspace(2, 2, 8, 8, 16, li)
    assert tuple(ws["CLIP_H"].shape) == (2, li, 128) and tuple(ws["CLIP"].shape) == (2, li, 256)
    assert len(ws["CKVI"]) == 2 and tuple(ws["CKVI"][0].shape) == (2, li, 512)
    assert tuple(ws["OUT"].shape) == (2, 16, 2, 8, 8)
    ws0 = ex.workspace(2, 2, 8, 8, 16, 0)                   # no clip_fea: image K/V from the 16 text tokens
    assert tuple(ws0["CKVI"][0].shape) == (2, 16, 512) and "CLIP" not in ws0
    x = torch.zeros(2, 36, 2, 8, 8)
    ctx, clip = torch.zeros(2, 16, 64), torch.zeros(2, li, 128)
    assert ex._geometry(x.shape, ctx, clip) == (2, 2, 8, 8, 16, li)
    assert ex._geometry(x.shape, ctx, None) == (2, 2, 8, 8, 16, 0)


def test_entry_points_and_batch_mismatch():
    from comfyui_parallelanything_b200.exec.wan_exec import WanClipExecutor, WanExecutor
    names = lambda f: list(inspect.signature(f).parameters)  # noqa: E731
    assert names(WanClipExecutor.denoise_step)[:6] == ["self", "x", "timesteps", "context", "clip_fea", "sigmas"]
    assert "clip_fea" in names(WanClipExecutor.forward_shard) and "clip_fea" in names(WanClipExecutor.shard_graph_handle)
    assert names(WanClipExecutor._prep) == ["self", "x", "timesteps", "context", "clip_fea"]
    assert WanClipExecutor.conditioning_kwargs == ("clip_fea",) and not hasattr(WanExecutor, "conditioning_kwargs")
    ex = WanClipExecutor(_model().to(torch.bfloat16), "cpu")
    with pytest.raises(ValueError):
        ex._inputs(2, torch.zeros(2), torch.zeros(2, 16, 64), torch.zeros(1, 257, 128))


def test_fused_staging_identity_survives_batch_split():
    """The fused data-parallel path receives fresh split views of the same conditioning every step: the staged copy
    must be reused (cache hit) while the sampler's tensor is unchanged, and refreshed after an in-place write."""
    from types import SimpleNamespace
    from comfyui_parallelanything_b200.engine import ParallelEngine
    from comfyui_parallelanything_b200.parallel import split
    counts = {}
    fake = SimpleNamespace(config=SimpleNamespace(cache_conditioning=True),
                           metrics=SimpleNamespace(incr=lambda k: counts.__setitem__(k, counts.get(k, 0) + 1)))
    clip = torch.randn(5, 257, 16)
    st, buf = {}, torch.empty(2, 257, 16)
    for _ in range(3):
        chunk = split.split_kwargs({"clip_fea": clip}, [3, 2], 5)[1]["clip_fea"]
        ParallelEngine._stage_conditioning(fake, st, "kw:clip_fea", buf, chunk)
    assert counts.get("cond_cache_hits") == 2 and torch.equal(buf, clip[3:])
    clip.mul_(2.0)
    chunk = split.split_kwargs({"clip_fea": clip}, [3, 2], 5)[1]["clip_fea"]
    ParallelEngine._stage_conditioning(fake, st, "kw:clip_fea", buf, chunk)
    assert counts.get("cond_cache_hits") == 2 and torch.equal(buf, clip[3:])
