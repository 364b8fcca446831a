"""WAN2.2 TI2V-5B (48 latent channels in and out, one timestep per latent frame) on the CPU: recognition, builder
choice, the oracle's per-frame timestep path, batch splitting and what the native executor packs.  The GPU side is in
test_gpu_wan_ti2v.py and the ``*_per_frame`` / ``wan_ti2v_*`` self-checks."""
import dataclasses

import pytest
import torch

from comfyui_parallelanything_b200 import exec as native_exec
from comfyui_parallelanything_b200.exec import recognize
from comfyui_parallelanything_b200.models import wan
from comfyui_parallelanything_b200.parallel import split
from comfyui_parallelanything_b200.utils.lookalike import launder


def _ti2v_params():
    return dataclasses.replace(wan.wan_tiny_params(), in_dim=48, out_dim=48)


def _rel(a, b):
    return ((a - b).abs().mean() / b.abs().mean()).item()


def _oracle_and_inputs(seed=0):
    torch.manual_seed(seed)
    p = _ti2v_params()
    m = wan.WanModel(p).eval()
    inp = wan.ti2v_inputs(p, 2, frames=9, height=256, width=320, dtype=torch.float32, seed=seed)
    return m, inp


def test_ti2v_params_and_inputs():
    p = wan.wan22_ti2v_5b_params()
    assert (p.in_dim, p.out_dim, p.dim, p.ffn_dim, p.num_heads, p.num_layers) == (48, 48, 3072, 14336, 24, 30)
    assert (p.text_dim, p.freq_dim, p.dim // p.num_heads) == (4096, 256, 128)
    inp = wan.ti2v_inputs(p, 2, frames=121, height=704, width=1280, dtype=torch.float32)
    assert tuple(inp["x"].shape) == (2, 48, 31, 44, 80)              # 27 280 tokens
    t = inp["timesteps"]
    assert tuple(t.shape) == (2, 31)
    assert torch.equal(t[:, 0], torch.zeros(2)) and bool((t[:, 1:] > 0).all())
    assert torch.equal(t[:, 1:], t[:, 1:2].expand(2, 30))
    assert tuple(inp["context"].shape) == (2, 512, 4096)


def test_ti2v_model_and_lookalike_select_wan_builder():
    torch.manual_seed(0)
    m = wan.WanModel(_ti2v_params())
    for mod in (m, launder(m)):
        fam, dp = recognize.identify(mod)
        assert fam == "wan" and (dp.in_dim, dp.out_dim) == (48, 48) and not dp.has_img_emb
        b = native_exec.builder_for(mod)
        assert b is not None and b.__name__ == "build_wan_executor"


@pytest.mark.parametrize("dims", [(48, 16), (36, 48), (16, 48)])
def test_other_channel_pairs_keep_torch_replica(dims):
    p = dataclasses.replace(wan.wan_tiny_params(), in_dim=dims[0], out_dim=dims[1])
    m = wan.WanModel(p)
    assert recognize.identify(m)[0] == "wan"
    assert native_exec.builder_for(m) is None
    from comfyui_parallelanything_b200.exec.wan_exec import WanExecutor
    with pytest.raises(ValueError):
        WanExecutor(m.to(torch.bfloat16), "cpu")


def test_oracle_equal_frame_timesteps_match_per_sample():
    m, inp = _oracle_and_inputs()
    t1 = torch.tensor([310.0, 870.0])
    T = inp["x"].shape[2]
    with torch.no_grad():
        want = m(inp["x"], t1, context=inp["context"])
        same = m(inp["x"], t1[:, None].expand(2, T).contiguous(), context=inp["context"])
        col = m(inp["x"], t1[:, None], context=inp["context"])
    assert torch.equal(col, want), "[B, 1] timesteps must take the [B] path"
    assert torch.allclose(same, want, rtol=1e-4, atol=1e-5), (same - want).abs().max()


def test_oracle_per_frame_timesteps_change_the_result():
    """Frame 0 at t = 0 (the start image) must differ from one timestep per sample by far more than the GPU checks'
    tolerances (0.03 bf16, 0.05 fp8), frame by frame, so those checks (which compare each frame) can tell a per-sample
    modulation lookup from a per-frame one."""
    m, inp = _oracle_and_inputs()
    t = inp["timesteps"]
    t[:, 1:] = torch.tensor([[700.0], [450.0]])
    with torch.no_grad():
        per_frame = m(inp["x"], t, context=inp["context"])
        at_t = m(inp["x"], t[:, 1], context=inp["context"])
        at_0 = m(inp["x"], t[:, 0], context=inp["context"])
    assert tuple(per_frame.shape) == tuple(inp["x"].shape)
    # wrong on frame 0 if every frame took t, wrong on the other frames if every frame took frame 0's timestep
    assert _rel(per_frame[:, :, :1], at_t[:, :, :1]) > 0.15
    assert _rel(per_frame[:, :, 1:], at_0[:, :, 1:]) > 0.15
    # each frame follows its own timestep (attention mixes frames, so only approximately)
    assert _rel(per_frame[:, :, :1], at_0[:, :, :1]) < 0.02
    assert _rel(per_frame[:, :, 1:], at_t[:, :, 1:]) < 0.02


def test_oracle_rejects_frame_count_mismatch():
    m, inp = _oracle_and_inputs()
    with pytest.raises(ValueError):
        m(inp["x"], inp["timesteps"][:, :2], context=inp["context"])


def test_split_value_keeps_frames_together():
    t = torch.arange(5 * 7, dtype=torch.float32).view(5, 7)
    chunks = split.split_value(t, [3, 2])
    assert [tuple(c.shape) for c in chunks] == [(3, 7), (2, 7)]
    assert torch.equal(torch.cat(chunks), t)


def test_executor_packing_and_timestep_geometry():
    from comfyui_parallelanything_b200.exec.wan_exec import WanExecutor, frame_lookup, frame_steps
    torch.manual_seed(0)
    p = _ti2v_params()
    m = wan.WanModel(p).to(torch.bfloat16)
    ex = WanExecutor(m, "cpu")
    assert torch.equal(ex.W["patch.w"], m.patch_embedding.weight.reshape(p.dim, 192))
    # head rows (pt, ph, pw, c) -> (c, ph, pw): row 4*c + k of the packed head is row k*48 + c of the model's
    hw, hb = m.head.head.weight, m.head.head.bias
    for c in (0, 17, 47):
        for k in range(4):
            assert torch.equal(ex.W["head.w"][4 * c + k], hw[k * 48 + c])
            assert torch.equal(ex.W["head.b"][4 * c + k], hb[k * 48 + c])
    assert ex.out_shape((2, 48, 3, 16, 20)) == (2, 48, 3, 16, 20)
    shape = (2, 48, 3, 16, 20)
    assert frame_steps(torch.zeros(2), shape) == 1
    assert frame_steps(torch.zeros(2, 1), shape) == 1
    assert frame_steps(torch.zeros(2, 3), shape) == 3
    for bad in (torch.zeros(2, 4), torch.zeros(3, 3), torch.zeros(2, 3, 1)):
        with pytest.raises(ValueError):
            frame_steps(bad, shape)
    ctx = torch.zeros(2, 16, 64)
    t2 = ex._inputs(2, torch.zeros(2, 3), ctx)[0]
    assert ex._geometry_of(shape, (t2, ctx)) == (2, 3, 16, 20, 16, 3)
    assert ex._geometry_of(shape, ex._inputs(2, torch.zeros(2, 1), ctx)) == (2, 3, 16, 20, 16, 1)
    ws = ex.workspace(2, 3, 16, 20, 16, 3)
    for k in ("T1", "E_H", "E", "SE", "E0", "MOD", "HSHIFT", "HSCALE"):
        assert ws[k].shape[0] == 6, k
    assert tuple(ws["OUT"].shape) == shape
    fr = frame_lookup(ws)
    assert fr == {"ln": dict(mod_rows=80, mod_row_off=0), "gate": dict(gate_rows=80, gate_row_off=0)}
    assert frame_lookup(ws, row_off=120)["gate"]["gate_row_off"] == 120
    ws1 = ex.workspace(2, 3, 16, 20, 16)
    assert ws1["MOD"].shape[0] == 2 and frame_lookup(ws1) == {"ln": {}, "gate": {}}
