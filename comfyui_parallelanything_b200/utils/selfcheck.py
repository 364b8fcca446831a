"""Numerics self-checks of every native kernel against plain PyTorch fp32 references.

Used three ways: ``pytest -m gpu`` (tests/test_gpu_kernels.py), ``tools/gpu_check.py``
(each check in its own process so a trapped kernel cannot poison the rest; JSON report
into ``gpurun_out/``) and ``__graft_entry__.smoke()``.
Every check returns ``dict(name, max_abs, max_rel, tol, ok, ...)``.
"""
from __future__ import annotations

import math
from typing import Callable, Dict

import torch
import torch.nn.functional as F

from .. import ops

CHECKS: Dict[str, Callable[[], dict]] = {}


def check(fn):
    CHECKS[fn.__name__] = fn
    return fn


def _cmp(name: str, got: torch.Tensor, want: torch.Tensor, tol: float, hard: float = 32.0, **extra) -> dict:
    """Pass = mean error < tol (relative to the typical magnitude of the reference), at most numel/10000 elements
    beyond 8*tol, AND no element at all beyond ``hard``*tol: a single wrong row / tile boundary of an otherwise
    correct result has errors of the order of the values themselves and fails the hard bound even when it is far
    too small a fraction to move the mean."""
    got, want = got.float(), want.float()
    diff = (got - want).abs()
    scale = want.abs().mean().item() + 1e-6
    max_abs = diff.max().item()
    # error relative to the typical magnitude of the reference (bf16 outputs: ~2^-8 relative)
    rel = max_abs / scale
    mean_rel = diff.mean().item() / scale
    bad = int((diff > tol * scale * 8).sum().item())
    ok = bool(mean_rel < tol and math.isfinite(max_abs) and bad <= max(1, diff.numel() // 10000)
              and rel <= hard * tol)
    return dict(name=name, max_abs=max_abs, max_rel=rel, mean_rel=mean_rel, tol=tol, hard_bound=hard * tol, ok=ok,
                outliers=bad, numel=diff.numel(), **extra)


def _dev():
    return torch.device("cuda", torch.cuda.current_device())


def _rand(*shape, scale=1.0, seed=0):
    g = torch.Generator(device="cpu").manual_seed(seed + sum(shape))
    return (torch.randn(*shape, generator=g) * scale).to(device=_dev(), dtype=torch.bfloat16)


# ------------------------------------------------------------------------------ GEMM
def _gemm_ref(a, w, bias=None):
    y = a.float() @ w.float().t()
    return y + bias.float() if bias is not None else y


@check
def gemm_bias_small():
    a, w, b = _rand(300, 256), _rand(512, 256, scale=0.06), _rand(512)
    out = torch.zeros(300, 512, dtype=torch.bfloat16, device=_dev())
    ops.gemm(a, w, "bias", out=out, bias=b)
    return _cmp("gemm_bias_small", out, _gemm_ref(a, w, b), 0.01)


@check
def gemm_bn_variants():
    a, w, b = _rand(384, 512), _rand(768, 512, scale=0.05), _rand(768)
    want = _gemm_ref(a, w, b)
    worst = None
    for bn in (64, 128, 256):
        out = torch.zeros(384, 768, dtype=torch.bfloat16, device=_dev())
        ops.gemm(a, w, "bias", out=out, bias=b, force_bn=bn)
        r = _cmp(f"gemm_bn{bn}", out, want, 0.01)
        if worst is None or r["mean_rel"] > worst["mean_rel"]:
            worst = r
    worst["name"] = "gemm_bn_variants"
    return worst


@check
def gemm_flux_shape():
    """One FLUX linear at full size: M=4608 tokens, K=3072, N=9216 (persistent multi-wave)."""
    a, w, b = _rand(4608, 3072), _rand(9216, 3072, scale=0.02), _rand(9216)
    out = torch.empty(4608, 9216, dtype=torch.bfloat16, device=_dev())
    ops.gemm(a, w, "bias", out=out, bias=b)
    return _cmp("gemm_flux_shape", out, _gemm_ref(a, w, b), 0.01)


@check
def gemm_batched_strided_views():
    x = _rand(3, 640, 256)                        # [B, txt(128)+img(512), D]
    w, b = _rand(256, 256, scale=0.06), _rand(256)
    out = torch.zeros(3, 640, 256, dtype=torch.bfloat16, device=_dev())
    ops.gemm(x[:, 128:], w, "bias", out=out[:, 128:], bias=b)
    ops.gemm(x[:, :128], w, "gelu", out=out[:, :128], bias=b)
    want = torch.empty(3, 640, 256, device=_dev())
    want[:, 128:] = _gemm_ref(x[:, 128:], w, b)
    want[:, :128] = F.gelu(_gemm_ref(x[:, :128], w, b), approximate="tanh")
    return _cmp("gemm_batched_strided_views", out, want, 0.012)


@check
def gemm_epilogues():
    a, w, b = _rand(2, 256, 512), _rand(512, 512, scale=0.04), _rand(512)
    res, gate = _rand(2, 256, 512), _rand(2, 512)
    y = _gemm_ref(a, w, b)
    outs, wants = [], []
    for mode, ref in (("silu", F.silu(y)), ("gelu", F.gelu(y, approximate="tanh")),
                      ("gate_res", res.float() + gate.float()[:, None] * y), ("res", res.float() + y)):
        out = torch.zeros(2, 256, 512, dtype=torch.bfloat16, device=_dev())
        ops.gemm(a, w, mode, out=out, bias=b, residual=res, gate=gate)
        outs.append(out.float())
        wants.append(ref)
    return _cmp("gemm_epilogues", torch.stack(outs), torch.stack(wants), 0.012)


@check
def gemm_skinny_m():
    a, w, b = _rand(8, 3072), _rand(18432, 3072, scale=0.02), _rand(18432)
    out = torch.zeros(8, 18432, dtype=torch.bfloat16, device=_dev())
    ops.gemm(a, w, "bias", out=out, bias=b)
    return _cmp("gemm_skinny_m", out, _gemm_ref(a, w, b), 0.01)


@check
def gemm_geglu():
    a = _rand(256, 256)
    wa, wg, ba, bg = _rand(512, 256, scale=0.06), _rand(512, 256, scale=0.06), _rand(512), _rand(512)
    want = _gemm_ref(a, wa, ba) * F.gelu(_gemm_ref(a, wg, bg))
    # interleave rows in groups of 32: [a0..31 | g0..31 | a32..63 | ...]
    w = torch.stack([wa.view(16, 32, 256), wg.view(16, 32, 256)], 1).reshape(1024, 256).contiguous()
    b = torch.stack([ba.view(16, 32), bg.view(16, 32)], 1).reshape(1024).contiguous()
    out = torch.zeros(256, 512, dtype=torch.bfloat16, device=_dev())
    ops.gemm(a, w, "geglu", out=out, bias=b)
    return _cmp("gemm_geglu", out, want, 0.012)


def _rope_table(L, dev):
    from ..models import flux
    ids = torch.zeros(1, L, 3, device=dev)
    ids[0, :, 1] = torch.arange(L, device=dev) // 16
    ids[0, :, 2] = torch.arange(L, device=dev) % 16
    pe = flux.EmbedND(128, 10000, [16, 56, 56])(ids)          # [1,1,L,64,2,2]
    table = torch.stack([pe[0, 0, :, :, 0, 0], pe[0, 0, :, :, 1, 0]], -1).contiguous()   # (cos, sin)
    return pe, table


@check
def gemm_qkv_rope():
    from ..models import flux
    B, L, H, D = 2, 384, 2, 128
    hid = H * D
    x, w, b = _rand(B, L, hid), _rand(3 * hid + 512, hid, scale=0.06), _rand(3 * hid + 512)
    qs, ks = (1 + 0.1 * _rand(D).float()).bfloat16(), (1 + 0.1 * _rand(D, seed=3).float()).bfloat16()
    pe, table = _rope_table(L + 64, _dev())
    q = torch.zeros(B, H, L + 64, D, dtype=torch.bfloat16, device=_dev())
    k, v = torch.zeros_like(q), torch.zeros_like(q)
    cat = torch.zeros(B, L, hid + 512, dtype=torch.bfloat16, device=_dev())
    ops.gemm(x, w, "qkv_rope", q=q, k=k, v=v, q_scale=qs, k_scale=ks, rope=table, seq_off=64, out=cat,
             mlp_col_off=hid, bias=b)
    y = _gemm_ref(x, w, b)
    qkv, mlp = y[..., :3 * hid], y[..., 3 * hid:]
    rq, rk, rv = qkv.view(B, L, 3, H, D).permute(2, 0, 3, 1, 4)

    def rms(t, s):
        return t * torch.rsqrt((t * t).mean(-1, keepdim=True) + 1e-6) * s.float()
    rq, rk = rms(rq, qs), rms(rk, ks)
    rq, rk = flux.apply_rope(rq, rk, pe[:, :, 64:])
    got = torch.cat([q[:, :, 64:].float().flatten(), k[:, :, 64:].float().flatten(), v[:, :, 64:].float().flatten(),
                     cat[..., hid:].float().flatten()])
    want = torch.cat([rq.flatten(), rk.flatten(), rv.flatten(), F.gelu(mlp, approximate="tanh").flatten()])
    r = _cmp("gemm_qkv_rope", got, want, 0.012)
    r["untouched_prefix_zero"] = bool(q[:, :, :64].abs().max().item() == 0)
    r["ok"] = r["ok"] and r["untouched_prefix_zero"]
    return r


@check
def gemm_euler_unpatch():
    B, C, Hl, Wl, hid = 2, 16, 32, 32, 256
    L = (Hl // 2) * (Wl // 2)
    h, w, b = _rand(B, L, hid), _rand(C * 4, hid, scale=0.06), _rand(C * 4)
    x = _rand(B, C, Hl, Wl)
    sig = torch.tensor([[1.0, 0.9], [0.5, 0.25]], device=_dev())
    xo = torch.zeros(B + 1, C, Hl, Wl, dtype=torch.bfloat16, device=_dev())
    ops.gemm(h, w, "euler_unpatch", bias=b, x_in=x, x_out=xo, xout_sample_off=1, sigmas=sig, C=C, Hl=Hl, Wl=Wl)
    v = _gemm_ref(h, w, b).view(B, Hl // 2, Wl // 2, C, 2, 2).permute(0, 3, 1, 4, 2, 5).reshape(B, C, Hl, Wl)
    want = x.float() + (sig[:, 1] - sig[:, 0])[:, None, None, None] * v
    r = _cmp("gemm_euler_unpatch", xo[1:], want, 0.012)
    xo2 = torch.zeros(B, C, Hl, Wl, dtype=torch.bfloat16, device=_dev())
    ops.gemm(h, w, "euler_unpatch", bias=b, x_out=xo2, C=C, Hl=Hl, Wl=Wl)
    r2 = _cmp("unpatch_only", xo2, v, 0.012)
    r["ok"] = r["ok"] and r2["ok"] and bool(xo[0].abs().max().item() == 0)
    r["unpatch_only_mean_rel"] = r2["mean_rel"]
    return r


@check
def euler_unpatch_xin_stride():
    """Euler update of the first 16 channels of a wider (36-channel, WAN I2V) input: ``xin_bstride`` = its sample size."""
    B, C, Cin, Hl, Wl, hid = 2, 16, 36, 32, 48, 256
    L = (Hl // 2) * (Wl // 2)
    h, w, b = _rand(B, L, hid), _rand(C * 4, hid, scale=0.06), _rand(C * 4)
    x = _rand(B, Cin, Hl, Wl)
    sig = torch.tensor([[1.0, 0.9], [0.5, 0.25]], device=_dev())
    xo = torch.zeros(B, C, Hl, Wl, dtype=torch.bfloat16, device=_dev())
    ops.gemm(h, w, "euler_unpatch", bias=b, x_in=x, xin_bstride=Cin * Hl * Wl, x_out=xo, sigmas=sig, C=C, Hl=Hl, Wl=Wl)
    v = _gemm_ref(h, w, b).view(B, Hl // 2, Wl // 2, C, 2, 2).permute(0, 3, 1, 4, 2, 5).reshape(B, C, Hl, Wl)
    want = x[:, :C].float() + (sig[:, 1] - sig[:, 0])[:, None, None, None] * v
    return _cmp("euler_unpatch_xin_stride", xo, want, 0.012)


# ------------------------------------------------------------------------------ attention
def _attn_case(name, B, H, Lq, Lk, tol=0.02):
    q, k, v = _rand(B, H, Lq, 128), _rand(B, H, Lk, 128, seed=1), _rand(B, H, Lk, 128, seed=2)
    want = F.scaled_dot_product_attention(q.float(), k.float(), v.float())
    want = want.transpose(1, 2).reshape(B, Lq, H * 128)
    worst = None
    for variant in (1, 2):                       # one query tile per CTA / ping-pong with two
        out = ops.attention(q, k, v, variant=variant)
        r = _cmp(name, out, want, tol)
        r["variant"] = variant
        if worst is None or not r["ok"] or (worst["ok"] and r["mean_rel"] > worst["mean_rel"]):
            worst = r
    return worst


@check
def attention_small():
    return _attn_case("attention_small", 1, 2, 256, 256)


@check
def attention_ragged():
    return _attn_case("attention_ragged", 2, 3, 200, 328)     # partial q tile + masked key padding


@check
def attention_flux_len():
    return _attn_case("attention_flux_len", 1, 4, 4608, 4608)


# ------------------------------------------------------------------------------ elementwise
@check
def layernorm_modulate():
    x, sc, sh = _rand(2, 300, 3072), _rand(2, 6, 3072, scale=0.3), _rand(2, 6, 3072, scale=0.3, seed=5)
    out = ops.layernorm_modulate(x[:, 44:], scale=sc[:, 1], shift=sh[:, 0])
    want = F.layer_norm(x[:, 44:].float(), (3072,), eps=1e-6) * (1 + sc[:, 1].float()[:, None]) + sh[:, 0].float()[:, None]
    r = _cmp("layernorm_modulate", out, want, 0.01)
    g, b = _rand(512), _rand(512, seed=9)
    x2 = _rand(64, 512)
    o2 = ops.layernorm_modulate(x2, gamma=g, beta=b, eps=1e-5)
    r2 = _cmp("ln_affine", o2, F.layer_norm(x2.float(), (512,), g.float(), b.float(), 1e-5), 0.01)
    r["ok"] = r["ok"] and r2["ok"]
    return r


@check
def timestep_embedding():
    from ..models import flux
    t = torch.tensor([0.0, 0.25, 0.5, 1.0], device=_dev(), dtype=torch.bfloat16)
    out = ops.timestep_embedding(t, 256)
    return _cmp("timestep_embedding", out, flux.timestep_embedding(t, 256), 0.01)


@check
def patchify():
    from ..models import flux
    m = flux.Flux.__new__(flux.Flux)
    m.patch_size = 2
    x = _rand(2, 16, 32, 48)
    out = torch.zeros(2, 16 * 24, 64, dtype=torch.bfloat16, device=_dev())
    ops.require().patchify(x.data_ptr(), out, 2, 16, 32, 48, 2)
    return _cmp("patchify", out, flux.Flux.patchify(m, x), 1e-6)


@check
def groupnorm_silu():
    x = _rand(2, 320, 24, 24)
    g, b = _rand(320), _rand(320, seed=4)
    nhwc = x.permute(0, 2, 3, 1).reshape(2, 576, 320).contiguous()
    out = ops.groupnorm_silu(nhwc, g, b, 32, 1e-5, True)
    want = F.silu(F.group_norm(x.float(), 32, g.float(), b.float(), 1e-5)).permute(0, 2, 3, 1).reshape(2, 576, 320)
    return _cmp("groupnorm_silu", out, want, 0.012)


@check
def cfg_euler_store():
    x, c, u = _rand(3, 4, 16, 16), _rand(3, 4, 16, 16, seed=1), _rand(3, 4, 16, 16, seed=2)
    sig = torch.tensor([[1.0, 0.8], [0.8, 0.6], [0.6, 0.1]], device=_dev())
    out = torch.zeros(5, 4, 16, 16, dtype=torch.bfloat16, device=_dev())
    ops.require().cfg_euler_store(x, c, u, out.data_ptr(), sig, 7.5, 2, 1)
    d = u.float() + 7.5 * (c.float() - u.float())
    want = x.float() + (sig[:, 1] - sig[:, 0])[:, None, None, None] * d
    r = _cmp("cfg_euler_store", out[2:], want, 0.012)
    r["ok"] = r["ok"] and bool(out[:2].abs().max().item() == 0)
    return r


@check
def flags_roundtrip():
    C = ops.require()
    flags = torch.zeros(16, dtype=torch.int32, device=_dev())
    err = torch.zeros(1, dtype=torch.int32, device=_dev())
    table = torch.tensor([flags.data_ptr()], dtype=torch.int64, device=_dev())
    C.signal_flags(table, 1, 3, 7)
    C.wait_flags(flags, 3, 1, 7, 2_000_000_000, err)
    C.wait_flags(flags, 4, 1, 1, 2_000_000, err)        # never signalled -> watchdog sets err, no hang
    torch.cuda.synchronize()
    e = err.item() & 0xFFFFFFFF
    ok = flags[3].item() == 7 and (e & 0xFFFF0000) == 0xDEAD0000 and (e & 0xFFFF) == 4
    return dict(name="flags_roundtrip", ok=bool(ok), flag=int(flags[3].item()), err=hex(e))


# ------------------------------------------------------------------------------ executors
def _flux_pair(params, seed=0):
    from ..exec.flux_exec import FluxExecutor
    from ..models import flux
    torch.manual_seed(seed)
    m = flux.Flux(params).to(device=_dev(), dtype=torch.bfloat16).eval()
    with torch.no_grad():
        for n_, p_ in m.named_parameters():          # non-trivial norm scales / biases
            if n_.endswith("scale"):
                p_.add_(0.1 * torch.randn_like(p_))
    ex = FluxExecutor(m, _dev())
    oracle = flux.Flux(params).to(device=_dev(), dtype=torch.float32).eval()
    oracle.load_state_dict({k: v.float() for k, v in m.state_dict().items()})
    return m, ex, oracle


@check
def flux_executor_tiny():
    from ..models import flux
    p = flux.flux_tiny_params()
    m, ex, oracle = _flux_pair(p)
    inp = flux.example_inputs(p, 2, 256, 256, txt_len=64, device=_dev(), dtype=torch.bfloat16)
    with torch.no_grad():
        got = ex(**inp)
        want = oracle(**{k: v.float() for k, v in inp.items()})
        eager = m(**inp)
    r = _cmp("flux_executor_tiny", got, want, 0.03)
    r["eager_bf16_mean_rel"] = _cmp("eager", eager, want, 1.0)["mean_rel"]   # what stock torch bf16 achieves
    r["launches"] = ex.launches_per_step
    # fused Euler step == x + dt * v
    sig = torch.tensor([[1.0, 0.75], [0.5, 0.25]], device=_dev())
    x, t, c, y, g = ex._prep(inp["x"], inp["timesteps"], inp["context"], inp["y"], inp["guidance"])
    with torch.no_grad():
        nxt = ex.denoise_step(x, t, c, y, g, sig).clone()
    want2 = inp["x"].float() + (sig[:, 1] - sig[:, 0])[:, None, None, None] * want
    r2 = _cmp("flux_euler", nxt, want2, 0.03)
    r["euler_mean_rel"] = r2["mean_rel"]
    r["ok"] = r["ok"] and r2["ok"]
    return r


@check
def flux_executor_mid():
    """Wider/deeper than tiny, ragged token counts (Lt=77, 24x40 latent) to exercise partial tiles."""
    from ..models import flux
    p = flux.FluxParams(in_channels=64, out_channels=64, vec_in_dim=768, context_in_dim=512, hidden_size=512,
                        mlp_ratio=4.0, num_heads=4, depth=2, depth_single_blocks=3)
    m, ex, oracle = _flux_pair(p, seed=1)
    inp = flux.example_inputs(p, 3, 192, 320, txt_len=77, device=_dev(), dtype=torch.bfloat16, seed=3)
    with torch.no_grad():
        got = ex(**inp)
        want = oracle(**{k: v.float() for k, v in inp.items()})
    return _cmp("flux_executor_mid", got, want, 0.03)


@check
def scatter_patch_embed():
    """Fused scatter kernel on one GPU (source pointers are local): patchify + img_in + temb."""
    from ..models import flux
    C_ = ops.require()
    n, Cc, Hl, Wl, N = 2, 16, 48, 40, 512
    Li = (Hl // 2) * (Wl // 2)
    x, w, b = _rand(n, Cc, Hl, Wl), _rand(N, 64, scale=0.1), _rand(N)
    t = torch.tensor([0.3, 0.9], device=_dev(), dtype=torch.bfloat16)
    g = torch.tensor([3.5, 1.0], device=_dev(), dtype=torch.bfloat16)
    X = torch.zeros(n, 77 + Li, N, dtype=torch.bfloat16, device=_dev())
    t_emb, g_emb = torch.zeros(n, 256, dtype=torch.bfloat16, device=_dev()), torch.zeros(n, 256, dtype=torch.bfloat16, device=_dev())
    xc = torch.zeros_like(x)
    C_.scatter_patch_embed(w, b, x.data_ptr(), t.data_ptr(), g.data_ptr(), t_emb, g_emb, xc, X[:, 77:], Cc, Hl, Wl, 1000.0)
    m = flux.Flux.__new__(flux.Flux)
    m.patch_size = 2
    want = _gemm_ref(flux.Flux.patchify(m, x), w, b)
    r = _cmp("scatter_patch_embed", X[:, 77:], want, 0.012)
    r2 = _cmp("temb", torch.cat([t_emb, g_emb]), torch.cat([flux.timestep_embedding(t, 256), flux.timestep_embedding(g, 256)]), 0.01)
    r["temb_mean_rel"] = r2["mean_rel"]
    r["ok"] = r["ok"] and r2["ok"] and bool(torch.equal(xc, x)) and bool(X[:, :77].abs().max().item() == 0)
    return r


@check
def scatter_patch_embed_wide():
    """Fused scatter kernel with latents wider than one 64-column K block (WAN2.2 I2V: 36 channels), 2..4 K blocks.
    One sample, so the output columns are split over several CTAs; 260 tokens = a partial last token tile."""
    from ..models import flux
    C_ = ops.require()
    m = flux.Flux.__new__(flux.Flux)
    m.patch_size = 2
    Hl, Wl, N = 26, 40, 768
    Li = (Hl // 2) * (Wl // 2)
    t = torch.tensor([0.7], device=_dev(), dtype=torch.bfloat16)
    worst = None
    for Cc in (20, 36, 64):
        x, w, b = _rand(1, Cc, Hl, Wl), _rand(N, 4 * Cc, scale=0.1), _rand(N)
        X = torch.zeros(1, 5 + Li, N, dtype=torch.bfloat16, device=_dev())
        t_emb = torch.zeros(1, 256, dtype=torch.bfloat16, device=_dev())
        xc = torch.zeros_like(x)
        C_.scatter_patch_embed(w, b, x.data_ptr(), t.data_ptr(), 0, t_emb, None, xc, X[:, 5:], Cc, Hl, Wl, 1.0)
        r = _cmp("scatter_patch_embed_wide", X[:, 5:], _gemm_ref(flux.Flux.patchify(m, x), w, b), 0.012, C=Cc)
        r["ok"] = r["ok"] and bool(torch.equal(xc, x)) and bool(X[:, :5].abs().max().item() == 0)
        if worst is None or not r["ok"] or (worst["ok"] and r["mean_rel"] > worst["mean_rel"]):
            worst = r
    return worst


# ------------------------------------------------------------------------------ convolution
def _conv_case(name, N, Cin, H, W, Cout, k, stride, mode="bias"):
    x = _rand(N, Cin, H, W)
    w = _rand(Cout, Cin, k, k, scale=(Cin * k * k) ** -0.5)
    b = _rand(Cout)
    xh = x.permute(0, 2, 3, 1).contiguous()
    wp = ops.pack_conv_weight(w)
    bp = torch.zeros(wp.shape[0], dtype=torch.bfloat16, device=_dev())
    bp[:Cout] = b
    kw = {}
    want = F.conv2d(x.float(), w.float(), b.float(), stride=stride, padding=k // 2)
    Ho, Wo = want.shape[2], want.shape[3]
    if mode == "res":
        res = _rand(N, Ho * Wo, wp.shape[0])
        kw["residual"] = res
        want = want + res[..., :Cout].float().view(N, Ho, Wo, Cout).permute(0, 3, 1, 2)
    if mode == "bias_bcast":
        emb = _rand(N, wp.shape[0])
        kw["gate"] = emb
        want = want + emb[:, :Cout].float()[:, :, None, None]
    out = ops.conv2d_nhwc(xh, wp, k * k, stride, mode, bias=bp, **kw)
    got = out[..., :Cout].float().view(N, Ho, Wo, Cout).permute(0, 3, 1, 2)
    return _cmp(name, got, want, 0.012)


@check
def conv3x3_basic():
    return _conv_case("conv3x3_basic", 2, 64, 32, 32, 128, 3, 1)


@check
def conv3x3_ragged():
    r1 = _conv_case("conv3x3_ragged", 1, 320, 24, 40, 320, 3, 1, "bias_bcast")    # Cin = 5x64, W not /16
    r2 = _conv_case("conv3x3_c8", 2, 8, 16, 16, 32, 3, 1)                          # tiny Cin (padded K)
    r3 = _conv_case("conv3x3_small_hw", 2, 128, 8, 8, 256, 3, 1, "res")            # 8x8 feature map
    r1["ok"] = r1["ok"] and r2["ok"] and r3["ok"]
    r1["c8_mean_rel"], r1["hw8_mean_rel"] = r2["mean_rel"], r3["mean_rel"]
    return r1


@check
def conv3x3_stride2():
    return _conv_case("conv3x3_stride2", 2, 128, 32, 48, 128, 3, 2)


@check
def conv1x1():
    return _conv_case("conv1x1", 2, 192, 16, 24, 320, 1, 1, "res")


@check
def attention_d64_strided():
    """head_dim 64 (SDXL) straight from a fused [B, L, 3*H*D] QKV GEMM output (strided 4-D TMA views),
    plus a short cross-attention (Lk = 77)."""
    B, H, L, D = 2, 10, 1024, 64
    qkv = _rand(B, L, 3, H, D)
    q, k, v = (qkv[:, :, i].permute(0, 2, 1, 3) for i in range(3))       # [B, H, L, D] views, no copies
    want = F.scaled_dot_product_attention(q.float(), k.float(), v.float()).transpose(1, 2).reshape(B, L, H * D)
    kc, vc = _rand(B, 77, H, D, seed=5).permute(0, 2, 1, 3), _rand(B, 77, H, D, seed=6).permute(0, 2, 1, 3)
    want2 = F.scaled_dot_product_attention(q.float(), kc.float(), vc.float()).transpose(1, 2).reshape(B, L, H * D)
    r = None
    for variant in (1, 2):
        ra = _cmp("attention_d64_strided", ops.attention(q, k, v, variant=variant), want, 0.02)
        rb = _cmp("cross77", ops.attention(q, kc, vc, variant=variant), want2, 0.02)
        ra["cross77_mean_rel"] = rb["mean_rel"]
        ra["variant"] = variant
        ra["ok"] = ra["ok"] and rb["ok"]
        if r is None or not ra["ok"]:
            r = ra
    return r


@check
def attention_pair():
    """CTA-pair attention kernel (variant 3): FLUX length, ragged key length, odd number of 256-row query blocks,
    strided q/k/v views."""
    res = {"name": "attention_pair", "ok": True}
    for tag, (B, H, Lq, Lk) in {"flux": (1, 4, 4608, 4608), "ragged": (2, 3, 700, 333), "short": (1, 2, 100, 77)}.items():
        qkv = _rand(B, max(Lq, Lk), 3, H, 128, seed=Lq)
        q = qkv[:, :Lq, 0].permute(0, 2, 1, 3)
        k = qkv[:, :Lk, 1].permute(0, 2, 1, 3)
        v = qkv[:, :Lk, 2].permute(0, 2, 1, 3)
        got = ops.attention(q, k, v, variant=3)
        want = F.scaled_dot_product_attention(q.float(), k.float(), v.float()).transpose(1, 2).reshape(B, Lq, H * 128)
        r = _cmp(tag, got, want, 0.02)
        res[tag + "_mean_rel"] = r["mean_rel"]
        res["ok"] = res["ok"] and r["ok"]
    return res


@check
def attention_speed():
    """Device-timed FLUX-shaped attention (B=2, 24 heads, 4608 tokens) for both kernel variants."""
    q, k, v = (_rand(2, 24, 4608, 128, seed=i) for i in range(3))
    out = torch.empty(2, 4608, 3072, dtype=torch.bfloat16, device=_dev())
    res = {"name": "attention_speed", "ok": True}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for variant in (1, 2, 3, 20, 151):   # 20 + DBG mask (attention2.cu); +128: one softmax warpgroup per tile (default)
        for _ in range(3):
            ops.attention(q, k, v, out=out, variant=variant)
        e0.record()
        for _ in range(10):
            ops.attention(q, k, v, out=out, variant=variant)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 10
        res[f"v{variant}_ms"] = round(ms, 4)
        res[f"v{variant}_tflops"] = round(4.0 * 2 * 24 * 4608 * 4608 * 128 / ms / 1e9, 1)
    return res


@check
def layout_kernels():
    C_ = ops.require()
    x = _rand(2, 4, 12, 20)
    nh = torch.zeros(2, 12 * 20, 8, dtype=torch.bfloat16, device=_dev())
    C_.nchw_to_nhwc_pad(x.data_ptr(), nh, 2, 4, 240)
    ok = torch.equal(nh[..., :4], x.permute(0, 2, 3, 1).reshape(2, 240, 4)) and nh[..., 4:].abs().max().item() == 0
    a = _rand(2, 6, 10, 32)
    up = torch.empty(2, 12, 20, 32, dtype=torch.bfloat16, device=_dev())
    C_.upsample2x(a, up)
    ok = ok and torch.equal(up, F.interpolate(a.permute(0, 3, 1, 2).float(), scale_factor=2.0, mode="nearest")
                            .permute(0, 2, 3, 1).to(torch.bfloat16))
    b = _rand(2, 60, 64, seed=3)
    cat = torch.empty(2, 60, 96, dtype=torch.bfloat16, device=_dev())
    C_.concat_channels(a.view(2, 60, 32), b, cat)
    ok = ok and torch.equal(cat, torch.cat([a.view(2, 60, 32), b], -1))
    # gather with CFG pairs + Euler
    eps = _rand(4, 240, 32)
    xs = _rand(2, 4, 12, 20, seed=7)
    sig = torch.tensor([[1.0, 0.7], [0.5, 0.4]], device=_dev())
    out = torch.zeros(3, 4, 12, 20, dtype=torch.bfloat16, device=_dev())
    C_.unet_out_gather(eps, xs, out.data_ptr(), sig, 2, 4, True, 5.0, 1, 1)
    e = eps[..., :4].float().view(4, 12, 20, 4).permute(0, 3, 1, 2)
    dref = e[2:] + 5.0 * (e[:2] - e[2:])
    want = xs.float() + (sig[:, 1] - sig[:, 0])[:, None, None, None] * dref
    r = _cmp("layout_kernels", out[1:], want, 0.012)
    r["ok"] = r["ok"] and bool(ok) and bool(out[0].abs().max().item() == 0)
    return r


@check
def unet_executor_mini():
    from ..exec.unet_exec import UNetExecutor
    from ..models import unet
    cfg = unet.mini_sdxl_config()
    torch.manual_seed(3)
    m = unet.UNetModel(**cfg).to(device=_dev(), dtype=torch.bfloat16).eval()
    ex = UNetExecutor(m, _dev())
    oracle = unet.UNetModel(**cfg).to(device=_dev(), dtype=torch.float32).eval()
    oracle.load_state_dict({k: v.float() for k, v in m.state_dict().items()})
    inp = unet.example_inputs(cfg, 2, 256, 384, ctx_len=77, device=_dev(), dtype=torch.bfloat16)
    with torch.no_grad():
        got = ex(**inp)
        want = oracle(**{k: v.float() for k, v in inp.items()})
        eager = m(**inp)
    r = _cmp("unet_executor_mini", got, want, 0.03)
    r["eager_bf16_mean_rel"] = _cmp("eager", eager, want, 1.0)["mean_rel"]
    # fused gather: CFG pairs + Euler
    sig = torch.tensor([[14.6, 10.0]], device=_dev())
    x2 = torch.cat([inp["x"][:1], inp["x"][:1]])
    t2 = torch.cat([inp["timesteps"][:1]] * 2)
    c2, y2 = inp["context"], inp["y"]
    nxt = ex.denoise_step(x2, t2, c2, y2, sig, cfg_scale=4.0, cfg_pairs=True)
    with torch.no_grad():
        e2 = oracle(x2.float(), t2.float(), context=c2.float(), y=y2.float())
    d = e2[1:] + 4.0 * (e2[:1] - e2[1:])
    want2 = x2[:1].float() + (sig[:, 1] - sig[:, 0]) * d
    r2 = _cmp("unet_euler", nxt, want2, 0.04)
    r["euler_mean_rel"] = r2["mean_rel"]
    r["ok"] = r["ok"] and r2["ok"]
    return r


@check
def wan_executor_tiny():
    from ..exec.wan_exec import WanExecutor
    from ..models import wan
    p = wan.wan_tiny_params()
    torch.manual_seed(2)
    m = wan.WanModel(p).to(device=_dev(), dtype=torch.bfloat16).eval()
    with torch.no_grad():
        for n_, p_ in m.named_parameters():
            if "norm" in n_ and n_.endswith("weight"):
                p_.add_(0.1 * torch.randn_like(p_))
    ex = WanExecutor(m, _dev())
    oracle = wan.WanModel(p).to(device=_dev(), dtype=torch.float32).eval()
    oracle.load_state_dict({k: v.float() for k, v in m.state_dict().items()})
    inp = wan.example_inputs(p, 2, frames=8, height=128, width=192, device=_dev(), dtype=torch.bfloat16)
    with torch.no_grad():
        got = ex(**inp)
        want = oracle(**{k: v.float() for k, v in inp.items()})
        eager = m(**inp)
    r = _cmp("wan_executor_tiny", got, want, 0.03)
    r["eager_bf16_mean_rel"] = _cmp("eager", eager, want, 1.0)["mean_rel"]
    r["launches"] = ex.launches_per_step
    sig = torch.tensor([[1.0, 0.8], [0.6, 0.5]], device=_dev())
    x, t, c = ex._prep(inp["x"], inp["timesteps"], inp["context"])
    nxt = ex.denoise_step(x, t, c, sig).clone()
    want2 = inp["x"].float() + (sig[:, 1] - sig[:, 0])[:, None, None, None, None] * want
    r2 = _cmp("wan_euler", nxt, want2, 0.03)
    r["euler_mean_rel"] = r2["mean_rel"]
    r["ok"] = r["ok"] and r2["ok"]
    return r


def _wan_i2v_case(fp8: bool) -> dict:
    """Tiny WAN2.2 I2V executor (36 input channels) against the fp32 oracle: ``forward``, then ``denoise_step`` eager,
    captured and replayed twice with the latent changed in place between the calls."""
    import dataclasses
    from ..exec.wan_exec import WanExecutor
    from ..models import wan
    p = dataclasses.replace(wan.wan_tiny_params(), in_dim=36)
    torch.manual_seed(3)
    m = wan.WanModel(p).to(device=_dev(), dtype=torch.bfloat16).eval()
    ex = WanExecutor(m, _dev(), cuda_graphs=True, fp8=fp8)
    oracle = wan.WanModel(p).to(device=_dev(), dtype=torch.float32).eval()
    oracle.load_state_dict({k: v.float() for k, v in m.state_dict().items()})
    inp = wan.i2v_inputs(p, 2, frames=8, height=128, width=192, device=_dev(), dtype=torch.bfloat16, seed=4)
    tol = 0.05 if fp8 else 0.03
    name = "wan_i2v_executor_tiny" + ("_fp8" if fp8 else "")
    with torch.no_grad():
        got = ex(**inp)
        want = oracle(**{k: v.float() for k, v in inp.items()})
    r = _cmp(name, got, want, tol)
    r["ok"] = r["ok"] and tuple(got.shape) == (2, 16) + tuple(inp["x"].shape[2:])
    sig = torch.tensor([[1.0, 0.8], [0.6, 0.5]], device=_dev())
    x, t, c = ex._prep(inp["x"], inp["timesteps"], inp["context"])
    worst = 0.0
    for it in range(4):                                 # eager, capture, replay, replay
        x[:, :16].mul_(0.9)                             # only the noise channels change between steps
        nxt = ex.denoise_step(x, t, c, sig).clone()
        with torch.no_grad():
            v = oracle(x.float(), t.float(), context=c.float())
        want2 = x[:, :16].float() + (sig[:, 1] - sig[:, 0])[:, None, None, None, None] * v
        r2 = _cmp(name + "_euler", nxt, want2, tol)
        worst = max(worst, r2["mean_rel"])
        r["ok"] = r["ok"] and r2["ok"]
    r["euler_worst_mean_rel"] = worst
    r["graphs"] = sorted(ex._graphs.state(k) for k in list(ex._graphs._graphs))
    r["ok"] = r["ok"] and "graph" in r["graphs"]
    return r


@check
def wan_i2v_executor_tiny():
    return _wan_i2v_case(False)


@check
def wan_i2v_executor_tiny_fp8():
    return _wan_i2v_case(True)


def _frames_ref(v: torch.Tensor, rows: int, off: int, B: int, L: int) -> torch.Tensor:
    """[G, D] per-group vectors -> [B, L, D] per-row vectors: row r of sample b reads group (b*L + r + off) // rows."""
    idx = (torch.arange(B * L, device=v.device) + off) // rows
    return v.float()[idx].view(B, L, -1)


@check
def layernorm_modulate_per_frame():
    """LayerNorm + modulate with one scale / shift row per video frame (``mod_rows``): 130 rows per frame (not a
    multiple of 128 or of the 8 warps per block), D = 3072, a [B*T, 6, D] table like the WAN modulation table, and a
    token slice that starts mid-frame (``mod_row_off``, sequence parallelism)."""
    B, T, HW, D = 2, 3, 130, 3072
    L = T * HW
    x = _rand(B, L, D)
    table = _rand(B * T, 6, D, scale=0.3, seed=3)
    sc, sh = table[:, 1], table[:, 0]
    out = ops.layernorm_modulate(x, scale=sc, shift=sh, mod_rows=HW)
    ln = F.layer_norm(x.float(), (D,), eps=1e-6)
    want = ln * (1 + _frames_ref(sc, HW, 0, B, L)) + _frames_ref(sh, HW, 0, B, L)
    r = _cmp("layernorm_modulate_per_frame", out, want, 0.01)
    # batch 1, rows [off, off + Ll) of the clip: the slice's first row is in the middle of frame 0
    off, Ll = 57, 200
    xs = x[:1, off:off + Ll]
    o2 = ops.layernorm_modulate(xs, scale=sc[:T], shift=sh[:T], mod_rows=HW, mod_row_off=off)
    w2 = (F.layer_norm(xs.float(), (D,), eps=1e-6) * (1 + _frames_ref(sc[:T], HW, off, 1, Ll))
          + _frames_ref(sh[:T], HW, off, 1, Ll))
    r2 = _cmp("slice", o2, w2, 0.01)
    # per sample (no mod_rows) must stay what it was: same bits as a [B, D] view
    o3 = ops.layernorm_modulate(x, scale=sc[::T], shift=sh[::T])
    w3 = ln * (1 + sc[::T].float()[:, None]) + sh[::T].float()[:, None]
    r3 = _cmp("per_sample", o3, w3, 0.01)
    r["slice_mean_rel"], r["per_sample_mean_rel"] = r2["mean_rel"], r3["mean_rel"]
    r["ok"] = r["ok"] and r2["ok"] and r3["ok"]
    return r


@check
def gemm_gate_res_per_frame():
    """Gated-residual epilogue with one gate row per video frame (``gate_rows``), frame boundaries inside 128-row
    tiles (80 and 130 rows per frame): bf16 one-CTA, CTA pair (force_bn=512), MXFP8 one-CTA and CTA-pair kernels (the
    pair kernels need >= 256 rows per sample: 320 and 260 here, the last tile ragged), and a token slice that starts
    mid-frame (``gate_row_off``)."""
    res = {"name": "gemm_gate_res_per_frame", "ok": True}
    worst = 0.0
    for HW, T in ((80, 4), (130, 2)):
        B, K, N = 2, 256, 512
        L = T * HW
        a, w, b = _rand(B, L, K, seed=1), _rand(N, K, scale=0.05, seed=2), _rand(N, seed=3)
        gates = _rand(B * T, 6, N, seed=4)[:, 2]                       # strided [B*T, N] view of a modulation table
        resid = _rand(B, L, N, seed=5)
        want = resid.float() + _frames_ref(gates, HW, 0, B, L) * _gemm_ref(a, w, b)
        cases = [("bf16", None), ("bf16_pair", 512)]
        for tag, bn in cases:
            out = resid.clone()
            kw = dict(force_bn=bn) if bn else {}
            ops.gemm(a, w, "gate_res", out=out, bias=b, residual=out, gate=gates, gate_rows=HW, **kw)
            r = _cmp(tag, out, want, 0.012)
            worst = max(worst, r["mean_rel"])
            res[f"{tag}_hw{HW}_ok"] = r["ok"]
            res["ok"] = res["ok"] and r["ok"]
        aq, sfa = ops.quantize_mxfp8(a)
        wq, sfb = ops.quantize_mxfp8(w, 224)
        exact = (resid.float() + _frames_ref(gates, HW, 0, B, L)
                 * (ops.dequantize_mxfp8(aq, sfa) @ ops.dequantize_mxfp8(wq, sfb, 224)[0].t() + b.float()))
        for pair in (0, 1):
            out = resid.clone()
            ops.gemm_fp8(aq, sfa, wq, sfb, "gate_res", 224, out=out, bias=b, residual=out, gate=gates, gate_rows=HW,
                         pair=pair)
            r = _cmp(f"mxfp8_pair{pair}", out, exact, 0.012)
            worst = max(worst, r["mean_rel"])
            res[f"mxfp8_pair{pair}_hw{HW}_ok"] = r["ok"]
            res["ok"] = res["ok"] and r["ok"]
    # batch-1 token slice starting mid-frame, as a sequence-parallel rank sees it
    HW, T, off, Ll, K, N = 80, 3, 120, 120, 256, 512
    a, w, b = _rand(1, Ll, K, seed=6), _rand(N, K, scale=0.05, seed=7), _rand(N, seed=8)
    gates, resid = _rand(T, N, seed=9), _rand(1, Ll, N, seed=10)
    out = resid.clone()
    ops.gemm(a, w, "gate_res", out=out, bias=b, residual=out, gate=gates, gate_rows=HW, gate_row_off=off)
    r = _cmp("slice", out, resid.float() + _frames_ref(gates, HW, off, 1, Ll) * _gemm_ref(a, w, b), 0.012)
    res["slice_ok"] = r["ok"]
    res["ok"] = res["ok"] and r["ok"]
    res["mean_rel"] = max(worst, r["mean_rel"])
    return res


@check
def scatter_patch_embed_per_frame_t():
    """Fused scatter kernel of a 48-channel WAN2.2 TI2V latent (three 64-column K blocks, K = 192) with one timestep
    per latent frame: ``n_t`` = B*T sinusoids."""
    from ..models import flux
    C_ = ops.require()
    m = flux.Flux.__new__(flux.Flux)
    m.patch_size = 2
    B, Cc, T, Hl, Wl, N = 2, 48, 3, 16, 20, 768
    x = _rand(B, Cc, T * Hl, Wl)                      # [B, C, T, H, W] as the kernel reads it: a T*H tall image
    w, b = _rand(N, 4 * Cc, scale=0.1), _rand(N)
    t = torch.tensor([[0.0, 700.0, 700.0], [0.0, 450.0, 450.0]], device=_dev(), dtype=torch.bfloat16)
    Li = T * (Hl // 2) * (Wl // 2)
    X = torch.zeros(B, Li, N, dtype=torch.bfloat16, device=_dev())
    t_emb = torch.zeros(B * T, 256, dtype=torch.bfloat16, device=_dev())
    xc = torch.zeros_like(x)
    C_.scatter_patch_embed(w, b, x.data_ptr(), t.data_ptr(), 0, t_emb, None, xc, X, Cc, T * Hl, Wl, 1.0, B * T)
    r = _cmp("scatter_patch_embed_per_frame_t", X, _gemm_ref(flux.Flux.patchify(m, x), w, b), 0.012)
    r2 = _cmp("temb", t_emb, flux.timestep_embedding(t.reshape(-1), 256, time_factor=1.0), 0.01)
    r["temb_mean_rel"] = r2["mean_rel"]
    r["ok"] = r["ok"] and r2["ok"] and bool(torch.equal(xc, x))
    return r


@check
def euler_unpatch_c48():
    """Head GEMM with the Euler / unpatchify epilogue for 48 latent channels (N = 192, WAN2.2 TI2V)."""
    B, C, Hl, Wl, hid = 2, 48, 32, 40, 256
    L = (Hl // 2) * (Wl // 2)
    h, w, b = _rand(B, L, hid), _rand(C * 4, hid, scale=0.06), _rand(C * 4)
    x = _rand(B, C, Hl, Wl)
    sig = torch.tensor([[1.0, 0.9], [0.5, 0.25]], device=_dev())
    xo = torch.zeros(B, C, Hl, Wl, dtype=torch.bfloat16, device=_dev())
    ops.gemm(h, w, "euler_unpatch", bias=b, x_in=x, x_out=xo, sigmas=sig, C=C, Hl=Hl, Wl=Wl)
    v = _gemm_ref(h, w, b).view(B, Hl // 2, Wl // 2, C, 2, 2).permute(0, 3, 1, 4, 2, 5).reshape(B, C, Hl, Wl)
    want = x.float() + (sig[:, 1] - sig[:, 0])[:, None, None, None] * v
    return _cmp("euler_unpatch_c48", xo, want, 0.012)


def _per_frame_cmp(name: str, got: torch.Tensor, want: torch.Tensor, tol: float) -> dict:
    """``_cmp`` of the whole clip and of every latent frame on its own (dim 2): a per-sample modulation lookup is wrong
    on some frames only, which the whole-clip mean could hide."""
    r = _cmp(name, got, want, tol)
    frames = [_cmp(f"{name}_f{f}", got[:, :, f], want[:, :, f], tol) for f in range(got.shape[2])]
    r["frame_mean_rel"] = [round(fr["mean_rel"], 5) for fr in frames]
    r["ok"] = r["ok"] and all(fr["ok"] for fr in frames)
    return r


def _wan_ti2v_case(fp8: bool) -> dict:
    """Tiny WAN2.2 TI2V executor (48 channels in and out, per-frame timesteps, 80 tokens per frame) against the fp32
    oracle: ``forward``, then ``denoise_step`` eager, captured and replayed twice with the latent AND the per-frame
    timesteps changed in place between the calls (the graph must read both)."""
    import dataclasses
    from ..exec.wan_exec import WanExecutor
    from ..models import wan
    p = dataclasses.replace(wan.wan_tiny_params(), in_dim=48, out_dim=48)
    torch.manual_seed(5)
    m = wan.WanModel(p).to(device=_dev(), dtype=torch.bfloat16).eval()
    ex = WanExecutor(m, _dev(), cuda_graphs=True, fp8=fp8)
    oracle = wan.WanModel(p).to(device=_dev(), dtype=torch.float32).eval()
    oracle.load_state_dict({k: v.float() for k, v in m.state_dict().items()})
    inp = wan.ti2v_inputs(p, 2, frames=9, height=256, width=320, device=_dev(), dtype=torch.bfloat16, seed=6)
    inp["timesteps"][:, 1:] = torch.tensor([[700.0], [450.0]], device=_dev(), dtype=torch.bfloat16)
    tol = 0.05 if fp8 else 0.03
    name = "wan_ti2v_executor_tiny" + ("_fp8" if fp8 else "")
    with torch.no_grad():
        got = ex(**inp)
        want = oracle(**{k: v.float() for k, v in inp.items()})
    r = _per_frame_cmp(name, got, want, tol)
    r["ok"] = r["ok"] and tuple(got.shape) == tuple(inp["x"].shape)
    sig = torch.tensor([[1.0, 0.8], [0.6, 0.5]], device=_dev())
    x, t, c = ex._prep(inp["x"], inp["timesteps"], inp["context"])
    worst = 0.0
    for it in range(4):                                 # eager, capture, replay, replay
        x.mul_(0.9)
        t[:, 1:].sub_(100.0)                            # new per-frame timesteps, same buffer
        t[1, 0] = 50.0 * it                             # the image frame's timestep changes too
        nxt = ex.denoise_step(x, t, c, sig).clone()
        with torch.no_grad():
            v = oracle(x.float(), t.float(), context=c.float())
        want2 = x.float() + (sig[:, 1] - sig[:, 0])[:, None, None, None, None] * v
        r2 = _per_frame_cmp(name + "_euler", nxt, want2, tol)
        worst = max(worst, r2["mean_rel"])
        r["ok"] = r["ok"] and r2["ok"]
    r["euler_worst_mean_rel"] = worst
    r["graphs"] = sorted(ex._graphs.state(k) for k in list(ex._graphs._graphs))
    r["ok"] = r["ok"] and "graph" in r["graphs"]
    r["launches"] = ex.launches_per_step
    return r


@check
def wan_ti2v_executor_tiny():
    return _wan_ti2v_case(False)


@check
def wan_ti2v_executor_tiny_fp8():
    return _wan_ti2v_case(True)


@check
def attention_two_kv():
    """Two-source attention ``softmax(q K1^T) V1 + softmax(q K2^T) V2`` (WAN2.1 text + CLIP image cross-attention)
    through the strided views the executor passes (q from a [B, L, H*128] buffer, K/V from [B, L, 2*H*128] buffers),
    including 1- and 2-key tail tiles (257 / 514 image tokens) and a text length that is not a multiple of 128."""
    res = {"name": "attention_two_kv", "ok": True}
    for (B, H, Lq, L1, L2) in ((1, 2, 260, 512, 257), (2, 4, 1000, 512, 514), (1, 40, 3600, 512, 257),
                               (2, 2, 300, 77, 257)):
        dim = H * 128
        qb = _rand(B, Lq, dim, seed=1)
        kv1, kv2 = _rand(B, L1, 2 * dim, seed=2), _rand(B, L2, 2 * dim, seed=3)
        heads = lambda t, w, n: t.view(B, t.shape[1], n, H, 128)[:, :, w].permute(0, 2, 1, 3)  # noqa: E731
        q, k1, v1, k2, v2 = heads(qb, 0, 1), heads(kv1, 0, 2), heads(kv1, 1, 2), heads(kv2, 0, 2), heads(kv2, 1, 2)
        want = (F.scaled_dot_product_attention(q.float(), k1.float(), v1.float())
                + F.scaled_dot_product_attention(q.float(), k2.float(), v2.float()))
        want = want.transpose(1, 2).reshape(B, Lq, dim)
        out = torch.zeros(B, Lq, dim, dtype=torch.bfloat16, device=_dev())
        ops.attention(q, k1, v1, out=out, kv2=(k2, v2))
        r = _cmp("attention_two_kv", out, want, 0.02)
        tag = f"{B}x{H}x{Lq}x{L1}x{L2}"
        res[tag + "_mean_rel"] = r["mean_rel"]
        res[tag + "_max_rel"] = r["max_rel"]
        res["ok"] = res["ok"] and r["ok"]
    # device time at the WAN2.1-I2V 720p shape: one two-source launch against two one-source launches (which would
    # still need an add to combine their outputs)
    B, H, Lq, L1, L2 = 1, 40, 14400, 512, 257
    dim = H * 128
    qb, kv1, kv2 = _rand(B, Lq, dim, seed=4), _rand(B, L1, 2 * dim, seed=5), _rand(B, L2, 2 * dim, seed=6)
    heads = lambda t, w, n: t.view(B, t.shape[1], n, H, 128)[:, :, w].permute(0, 2, 1, 3)  # noqa: E731
    q, k1, v1, k2, v2 = heads(qb, 0, 1), heads(kv1, 0, 2), heads(kv1, 1, 2), heads(kv2, 0, 2), heads(kv2, 1, 2)
    out, o1, o2 = (torch.empty(B, Lq, dim, dtype=torch.bfloat16, device=_dev()) for _ in range(3))
    runs = {"two_source_us": lambda: ops.attention(q, k1, v1, out=out, kv2=(k2, v2)),
            "two_launches_us": lambda: (ops.attention(q, k1, v1, out=o1), ops.attention(q, k2, v2, out=o2))}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for name, fn in list(runs.items()) * 2:          # alternated, the second pass is reported
        for _ in range(5):
            fn()
        e0.record()
        for _ in range(50):
            fn()
        e1.record()
        torch.cuda.synchronize()
        res[name] = round(e0.elapsed_time(e1) / 50 * 1000, 1)
    res["speed_shape"] = [B, H, Lq, L1, L2]
    res["gpu"] = torch.cuda.get_device_name()
    return res


@check
def gemm_gelu_erf():
    """``gelu_erf`` epilogue: exact erf GELU (nn.GELU(), WAN's CLIP image projection), 1280-wide like that projection."""
    a, w, b = _rand(2, 257, 1280), _rand(1280, 1280, scale=0.03), _rand(1280)
    out = torch.zeros(2, 257, 1280, dtype=torch.bfloat16, device=_dev())
    ops.gemm(a, w, "gelu_erf", out=out, bias=b)
    return _cmp("gemm_gelu_erf", out, F.gelu(_gemm_ref(a, w, b)), 0.012)


def _wan_clip_case(fp8: bool, flf2v: bool) -> dict:
    """Tiny WAN2.1 I2V (or FLF2V: 514 CLIP tokens + ``emb_pos``) executor against the fp32 oracle: ``forward`` with and
    without ``clip_fea``, then ``denoise_step`` eager, captured and replayed twice, and once more with ``clip_fea=None``."""
    import dataclasses
    from ..exec.wan_exec import WanClipExecutor
    from ..models import wan
    p = dataclasses.replace(wan.wan_tiny_params(), in_dim=36, clip_dim=128, clip_pos_tokens=514 if flf2v else 0)
    torch.manual_seed(5)
    m = wan.WanModel(p).to(device=_dev(), dtype=torch.bfloat16).eval()
    with torch.no_grad():
        for n_, p_ in m.named_parameters():
            if "norm" in n_ and n_.endswith("weight"):
                p_.add_(0.1 * torch.randn_like(p_))
    ex = WanClipExecutor(m, _dev(), cuda_graphs=True, fp8=fp8)
    oracle = wan.WanModel(p).to(device=_dev(), dtype=torch.float32).eval()
    oracle.load_state_dict({k: v.float() for k, v in m.state_dict().items()})
    inp = wan.clip_inputs(p, 2, frames=8, height=128, width=192, device=_dev(), dtype=torch.bfloat16, seed=6)
    tol = 0.05 if fp8 else 0.03
    name = ("wan_flf2v" if flf2v else "wan_clip") + "_executor_tiny" + ("_fp8" if fp8 else "")
    f32 = lambda d: {k: (v.float() if v is not None else None) for k, v in d.items()}  # noqa: E731
    with torch.no_grad():
        got = ex(**inp)
        want = oracle(**f32(inp))
        got0 = ex(**dict(inp, clip_fea=None))
        want0 = oracle(**f32(dict(inp, clip_fea=None)))
    r = _cmp(name, got, want, tol)
    r0 = _cmp(name + "_no_clip", got0, want0, tol)
    r["no_clip_mean_rel"] = r0["mean_rel"]
    r["ok"] = r["ok"] and r0["ok"] and tuple(got.shape) == (2, 16) + tuple(inp["x"].shape[2:])
    sig = torch.tensor([[1.0, 0.8], [0.6, 0.5]], device=_dev())
    x, t, c, cf = ex._prep(inp["x"], inp["timesteps"], inp["context"], inp["clip_fea"])
    worst = 0.0
    for it in range(5):                                 # eager, capture, replay, replay; then without clip_fea
        x[:, :16].mul_(0.9)
        clip = cf if it < 4 else None
        nxt = ex.denoise_step(x, t, c, clip, sig).clone()
        with torch.no_grad():
            v = oracle(x.float(), t.float(), context=c.float(), clip_fea=clip.float() if clip is not None else None)
        want2 = x[:, :16].float() + (sig[:, 1] - sig[:, 0])[:, None, None, None, None] * v
        r2 = _cmp(name + "_euler", nxt, want2, tol)
        worst = max(worst, r2["mean_rel"])
        r["ok"] = r["ok"] and r2["ok"]
    r["euler_worst_mean_rel"] = worst
    r["graphs"] = sorted(ex._graphs.state(k) for k in list(ex._graphs._graphs))
    r["ok"] = r["ok"] and "graph" in r["graphs"]
    return r


@check
def wan_clip_executor_tiny():
    return _wan_clip_case(False, False)


@check
def wan_clip_executor_tiny_fp8():
    return _wan_clip_case(True, False)


@check
def wan_flf2v_executor_tiny():
    return _wan_clip_case(False, True)


@check
def wan_flf2v_executor_tiny_fp8():
    return _wan_clip_case(True, True)


@check
def gemm_2cta():
    """CTA-pair (cta_group::2) GEMM kernel, selected with force_bn=512: numerics on even / ragged shapes and a
    device-timed comparison with the one-CTA 128x256 kernel at a FLUX-like shape."""
    res = {"name": "gemm_2cta", "ok": True}
    for tag, (B, rows, K, N) in {"even": (2, 1024, 512, 768), "ragged": (3, 300, 320, 512), "one_tile": (1, 256, 64, 256)}.items():
        a, w, b = _rand(B, rows, K, seed=1), _rand(N, K, scale=0.05, seed=2), _rand(N, seed=3)
        out = torch.zeros(B, rows, N, dtype=torch.bfloat16, device=_dev())
        ops.gemm(a, w, "bias", out=out, bias=b, force_bn=512)
        r = _cmp(tag, out, _gemm_ref(a, w, b), 0.01)
        res[tag + "_mean_rel"] = r["mean_rel"]
        res["ok"] = res["ok"] and r["ok"]
    # gated residual epilogue on a strided activation view
    B, rows, K, N = 2, 640, 256, 512
    big = _rand(B, rows + 64, K, seed=4)
    a = big[:, 64:]
    w, b, g = _rand(N, K, scale=0.05, seed=5), _rand(N, seed=6), _rand(B, N, seed=7)
    resid = _rand(B, rows, N, seed=8)
    want = resid.float() + g[:, None].float() * _gemm_ref(a, w, b)
    out = resid.clone()
    ops.gemm(a, w, "gate_res", out=out, bias=b, residual=out, gate=g, force_bn=512)
    r = _cmp("gate_res", out, want, 0.012)
    res["gate_res_mean_rel"] = r["mean_rel"]
    res["ok"] = res["ok"] and r["ok"]
    # fused QKV (+ GELU'd MLP columns) epilogue: the pair kernel must reproduce the one-CTA kernel bit for bit
    B, L, H, D = 2, 384, 2, 128
    hid = H * D
    x, w, b = _rand(B, L, hid, seed=12), _rand(3 * hid + 512, hid, scale=0.06, seed=13), _rand(3 * hid + 512, seed=14)
    qs, ks = (1 + 0.1 * _rand(D).float()).bfloat16(), (1 + 0.1 * _rand(D, seed=3).float()).bfloat16()
    _, table = _rope_table(L, _dev())
    outs = []
    for bn in (256, 512):
        q = torch.zeros(B, H, L, D, dtype=torch.bfloat16, device=_dev())
        k, v = torch.zeros_like(q), torch.zeros_like(q)
        cat = torch.zeros(B, L, hid + 512, dtype=torch.bfloat16, device=_dev())
        ops.gemm(x, w, "qkv_rope", q=q, k=k, v=v, q_scale=qs, k_scale=ks, rope=table, seq_off=0, out=cat, mlp_col_off=hid,
                 bias=b, force_bn=bn)
        outs.append(torch.cat([q.flatten(), k.flatten(), v.flatten(), cat[..., hid:].flatten()]))
    res["qkv_rope_bit_identical"] = bool(torch.equal(outs[0], outs[1]))
    res["ok"] = res["ok"] and res["qkv_rope_bit_identical"]
    M, K, N = 18432, 3072, 9216
    a, w, b = _rand(M, K, seed=9), _rand(N, K, scale=0.02, seed=10), _rand(N, seed=11)
    out = torch.empty(M, N, dtype=torch.bfloat16, device=_dev())
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for tag, bn in (("one_cta", 256), ("two_cta", 512), ("one_cta_again", 256), ("two_cta_again", 512)):
        for _ in range(3):
            ops.gemm(a, w, "bias", out=out, bias=b, force_bn=bn)
        e0.record()
        for _ in range(20):
            ops.gemm(a, w, "bias", out=out, bias=b, force_bn=bn)
        e1.record()
        torch.cuda.synchronize()
        res[tag + "_tflops"] = round(2.0 * M * N * K * 20 / e0.elapsed_time(e1) / 1e9, 1)
    for tag, bn in (("gelu_one_cta", 256), ("gelu_two_cta", 512)):          # epilogue-heavy case
        for _ in range(3):
            ops.gemm(a, w, "gelu", out=out, bias=b, force_bn=bn)
        e0.record()
        for _ in range(20):
            ops.gemm(a, w, "gelu", out=out, bias=b, force_bn=bn)
        e1.record()
        torch.cuda.synchronize()
        res[tag + "_tflops"] = round(2.0 * M * N * K * 20 / e0.elapsed_time(e1) / 1e9, 1)
    return res


@check
def gemm_swiglu():
    """w1 / w3 of a SwiGLU FFN as one GEMM over row-interleaved weights, ``a * silu(g)`` in the epilogue."""
    M, K, H = 520, 256, 768
    a, w3, w1 = _rand(M, K), _rand(H, K, scale=0.08, seed=1), _rand(H, K, scale=0.08, seed=2)
    out = torch.empty(M, H, dtype=torch.bfloat16, device=_dev())
    ops.gemm(a, ops.interleave_glu(w3, w1), "swiglu", out=out)
    want = _gemm_ref(a, w3) * F.silu(_gemm_ref(a, w1))
    return _cmp("gemm_swiglu", out, want, 0.012)


@check
def rmsnorm_modulate_kernel():
    B, L, D = 2, 300, 3840
    x, w = _rand(B, L, D), 1.0 + _rand(D, scale=0.1, seed=3)
    sc, gt = _rand(B, 4 * D, scale=0.3, seed=4), _rand(B, 4 * D, seed=5)
    res = _rand(B, L + 7, D, seed=6)[:, 7:]                       # strided residual / output view
    xf = x.float()
    rms = xf * torch.rsqrt(xf.pow(2).mean(-1, keepdim=True) + 1e-5) * w.float()
    got1 = ops.rmsnorm_modulate(x, weight=w, scale=sc[:, D:2 * D], eps=1e-5)
    r1 = _cmp("rms_scale", got1, rms * (1 + sc[:, None, D:2 * D].float()), 0.01)
    want2 = res.float() + torch.tanh(gt[:, None, 2 * D:3 * D].float()) * rms
    ops.rmsnorm_modulate(x, out=res, weight=w, gate=gt[:, 2 * D:3 * D], residual=res, eps=1e-5)
    r2 = _cmp("rms_gate_res", res, want2, 0.01)
    got3 = ops.rmsnorm_modulate(_rand(3, 50, 2560, seed=8), weight=None, eps=1e-5)
    x3 = _rand(3, 50, 2560, seed=8).float()
    r3 = _cmp("rms_plain", got3, x3 * torch.rsqrt(x3.pow(2).mean(-1, keepdim=True) + 1e-5), 0.01)
    r1["gate_res_mean_rel"], r1["plain_mean_rel"] = r2["mean_rel"], r3["mean_rel"]
    r1["ok"] = r1["ok"] and r2["ok"] and r3["ok"]
    r1["name"] = "rmsnorm_modulate_kernel"
    return r1


@check
def zimage_executor_tiny():
    from ..exec.zimage_exec import ZImageExecutor
    from ..models import zimage
    p = zimage.zimage_tiny_params()
    torch.manual_seed(6)
    m = zimage.ZImageModel(p).to(device=_dev(), dtype=torch.bfloat16).eval()
    ex = ZImageExecutor(m, _dev())
    oracle = zimage.ZImageModel(p).to(device=_dev(), dtype=torch.float32).eval()
    oracle.load_state_dict({k: v.float() for k, v in m.state_dict().items()})
    inp = zimage.example_inputs(p, 2, 256, 384, cap_len=40, device=_dev(), dtype=torch.bfloat16)
    with torch.no_grad():
        got = ex(**inp)
        want = oracle(**{k: v.float() for k, v in inp.items()})
        eager = m(**inp)
    r = _cmp("zimage_executor_tiny", got, want, 0.03)
    r["eager_bf16_mean_rel"] = _cmp("eager", eager, want, 1.0)["mean_rel"]
    r["launches"] = ex.launches_per_step
    sig = torch.tensor([[1.0, 0.8], [0.6, 0.5]], device=_dev())
    x, t, c = ex._prep(inp["x"], inp["timesteps"], inp["context"])
    nxt = ex.denoise_step(x, t, c, sig).clone()
    want2 = inp["x"].float() + (sig[:, 1] - sig[:, 0])[:, None, None, None] * want
    r2 = _cmp("zimage_euler", nxt, want2, 0.03)
    r["euler_mean_rel"] = r2["mean_rel"]
    r["second_step_launches"] = ex.launches_per_step            # caption path cached
    r["ok"] = r["ok"] and r2["ok"]
    return r


@check
def vae_decoder_executor():
    from ..exec.vae_exec import VAEDecoderExecutor
    from ..models import vae
    torch.manual_seed(4)
    cfg = dict(z_channels=4, ch=64, ch_mult=[1, 2], num_res_blocks=1, out_ch=3)
    m = vae.VAEDecoder(**cfg).to(device=_dev(), dtype=torch.bfloat16).eval()
    ex = VAEDecoderExecutor(m, _dev())
    oracle = vae.VAEDecoder(**cfg).to(device=_dev(), dtype=torch.float32).eval()
    oracle.load_state_dict({k: v.float() for k, v in m.state_dict().items()})
    z = _rand(2, 4, 16, 24, scale=0.18)
    with torch.no_grad():
        got = ex.decode(z)
        want = oracle(z.float())
    return _cmp("vae_decoder_executor", got, want, 0.03)


# ------------------------------------------------------------------------------ MXFP8
@check
def gemm_mxfp8():
    """tcgen05 block-scaled fp8 GEMM vs (a) the exact product of the dequantised operands (tests the kernel, all
    three B-tile variants) and (b) the bf16-input fp32 reference (shows the quantisation error level)."""
    B, M, K, N = 2, 320, 1024, 768
    a, w, bias = _rand(B, M, K), _rand(N, K, scale=0.03), _rand(N)
    aq, sfa = ops.quantize_mxfp8(a)
    ad = ops.dequantize_mxfp8(aq, sfa)
    worst = None
    for tile in (128, 224, 256):
        wq, sfb = ops.quantize_mxfp8(w, tile)
        wd = ops.dequantize_mxfp8(wq, sfb, tile)[0]
        exact = F.gelu(ad @ wd.t() + bias.float(), approximate="tanh")
        # one CTA per tile | CTA pairs (256-row tiles, ragged M) | CTA pairs with split-N accumulators (256-wide only)
        for pair in ((0,) if tile == 128 else ((0, 1) if tile == 224 else (0, 1, 2))):
            out = torch.zeros(B, M, N, dtype=torch.bfloat16, device=_dev())
            ops.gemm_fp8(aq, sfa, wq, sfb, "gelu", tile, out=out, bias=bias, pair=pair)
            r = _cmp(f"gemm_mxfp8_t{tile}_pair{pair}", out, exact, 0.01)
            if worst is None or r["mean_rel"] > worst["mean_rel"] or not r["ok"]:
                worst = r
    full = F.gelu(a.float() @ w.float().t() + bias.float(), approximate="tanh")
    worst["vs_bf16_inputs_mean_rel"] = _cmp("q", out, full, 1.0)["mean_rel"]
    worst["quant_roundtrip_rel"] = ((ad - a.float()).abs().mean() / a.float().abs().mean()).item()
    worst["name"] = "gemm_mxfp8"
    return worst


@check
def gemm_mxfp8_row_range_operand():
    """A operand = a row range of a larger [B, L, K] MXFP8 buffer (how the txt / img proj GEMMs of a FLUX double block read
    the joint attention output): strided batch + `sfa_mtiles`, must equal the GEMM over a contiguous copy bit for bit."""
    B, L, K, N, r0 = 2, 640, 1024, 768, 128
    a, w, bias = _rand(B, L, K), _rand(N, K, scale=0.03), _rand(N)
    aq, sfa = ops.quantize_mxfp8(a)
    sub_q, sub_sf = ops.quantize_mxfp8(a[:, r0:].contiguous())
    ok, worst = True, 0.0
    for tile, pair in ((224, 0), (224, 1), (256, 1), (256, 2)):
        wq, sfb = ops.quantize_mxfp8(w, tile)
        want = torch.zeros(B, L - r0, N, dtype=torch.bfloat16, device=_dev())
        got = torch.zeros_like(want)
        ops.gemm_fp8(sub_q, sub_sf, wq, sfb, "bias", tile, out=want, bias=bias, pair=pair)
        ops.gemm_fp8(aq[:, r0:], sfa[(r0 // 128) * (K // 128) * 512:], wq, sfb, "bias", tile, out=got, bias=bias, pair=pair,
                     sfa_mtiles=L // 128)
        torch.cuda.synchronize()
        ok = ok and bool(torch.equal(got, want))
        worst = max(worst, (got.float() - want.float()).abs().max().item())
    return {"name": "gemm_mxfp8_row_range_operand", "ok": ok, "max_abs": worst}


@check
def gemm_mxfp8_flux_shape():
    M, K, N = 4608, 3072, 9216
    a, w = _rand(M, K), _rand(N, K, scale=0.02)
    aq, sfa = ops.quantize_mxfp8(a)
    res = {}
    r = None
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for tile, pair in ((224, 0), (224, 1), (256, 0), (256, 1), (256, 2), (128, 0)):
        wq, sfb = ops.quantize_mxfp8(w, tile)
        out = torch.empty(M, N, dtype=torch.bfloat16, device=_dev())
        ops.gemm_fp8(aq, sfa, wq, sfb, "bias", tile, out=out, pair=pair)
        if tile == 224:
            exact = ops.dequantize_mxfp8(aq, sfa)[0] @ ops.dequantize_mxfp8(wq, sfb, tile)[0].t()
            rr = _cmp(f"gemm_mxfp8_flux_shape_pair{pair}", out, exact, 0.01)
            if r is None or not rr["ok"]:
                r = rr
        for _ in range(3):
            ops.gemm_fp8(aq, sfa, wq, sfb, "bias", tile, out=out, pair=pair)
        e0.record()
        for _ in range(10):
            ops.gemm_fp8(aq, sfa, wq, sfb, "bias", tile, out=out, pair=pair)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 10
        res[f"tile{tile}{('', '_pair', '_pairsplit')[pair]}_tflops"] = round(2.0 * M * N * K / ms / 1e9, 1)
    o16 = torch.empty(M, N, dtype=torch.bfloat16, device=_dev())
    for _ in range(3):
        ops.gemm(a, w, "bias", out=o16)
    e0.record()
    for _ in range(10):
        ops.gemm(a, w, "bias", out=o16)
    e1.record()
    torch.cuda.synchronize()
    res["bf16_tflops"] = round(2.0 * M * N * K / (e0.elapsed_time(e1) / 10) / 1e9, 1)
    r.update(res)
    return r


@check
def flux_executor_fp8():
    """FLUX executor with MXFP8 block GEMMs vs the fp32 oracle (loose tolerance: e4m3 has 3 mantissa bits)."""
    from ..exec.flux_exec import FluxExecutor
    from ..models import flux
    p = flux.FluxParams(in_channels=64, out_channels=64, vec_in_dim=768, context_in_dim=512, hidden_size=512,
                        mlp_ratio=4.0, num_heads=4, depth=2, depth_single_blocks=2)
    torch.manual_seed(1)
    m = flux.Flux(p).to(device=_dev(), dtype=torch.bfloat16).eval()
    ex8 = FluxExecutor(m, _dev(), fp8=True)
    ex16 = FluxExecutor(m, _dev())
    oracle = flux.Flux(p).to(device=_dev(), dtype=torch.float32).eval()
    oracle.load_state_dict({k: v.float() for k, v in m.state_dict().items()})
    inp = flux.example_inputs(p, 2, 256, 256, txt_len=128, device=_dev(), dtype=torch.bfloat16, seed=3)
    with torch.no_grad():
        got8, got16 = ex8(**inp), ex16(**inp)
        want = oracle(**{k: v.float() for k, v in inp.items()})
    # stated tolerance of the fp8 engine: mean error <= 2 % of the fp32 oracle and <= 3x the bf16 executor's error
    r = _cmp("flux_executor_fp8", got8, want, 0.02)
    r["bf16_mean_rel"] = _cmp("bf16", got16, want, 1.0)["mean_rel"]
    r["n_fp8_weights"] = sum(1 for k in ex8.W if k.endswith(".q"))
    r["ok"] = r["ok"] and r["n_fp8_weights"] > 0 and r["mean_rel"] <= 3.0 * r["bf16_mean_rel"] + 1e-3
    return r


@check
def pack_cache_roundtrip():
    """Packed-weight checkpoint: save an fp8 FLUX executor, scramble it, restore it, same output."""
    import os
    import tempfile
    from ..exec import pack_cache
    from ..exec.flux_exec import FluxExecutor
    from ..models import flux
    p = flux.flux_tiny_params()
    torch.manual_seed(5)
    m = flux.Flux(p).to(device=_dev(), dtype=torch.bfloat16).eval()
    ex = FluxExecutor(m, _dev(), fp8=True)
    inp = flux.example_inputs(p, 1, 128, 128, txt_len=32, device=_dev(), dtype=torch.bfloat16)
    before = ex(**inp).clone()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "flux_tiny.pa")
        nbytes = pack_cache.save_packed(ex, path)
        for k, v in ex.W.items():
            if isinstance(v, torch.Tensor) and v.dtype == torch.bfloat16:
                v.zero_()
        broken = ex(**inp).clone()
        meta = pack_cache.load_packed_into(ex, path)
    after = ex(**inp)
    ok = bool(torch.equal(before, after)) and not bool(torch.equal(before, broken)) and meta["fp8"] is True
    return dict(name="pack_cache_roundtrip", ok=ok, bytes=nbytes, keys=meta["keys"])


# ------------------------------------------------------------------------------ round-2 additions
@check
def scatter_conv_in():
    """Fused scatter + conv_in kernel on one GPU (source pointers are local): NCHW latent -> 3x3 im2col -> tcgen05
    GEMM -> NHWC rows, the timestep sinusoid and the local copy of the shard, vs torch conv2d in fp32."""
    import torch.nn.functional as F
    from ..models import unet
    C_ = ops.require()
    n, Cc, H, W, N = 3, 4, 40, 56, 320                      # H*W = 2240: not a multiple of the 128-pixel tile
    x = _rand(n, Cc, H, W)
    w4, b = _rand(N, Cc, 3, 3, scale=0.2), _rand(N)
    t = torch.tensor([999.0, 500.0, 3.0], device=_dev(), dtype=torch.bfloat16)
    out = torch.zeros(n, H * W, N, dtype=torch.bfloat16, device=_dev())
    temb = torch.zeros(n, N, dtype=torch.bfloat16, device=_dev())
    xc = torch.zeros_like(x)
    C_.scatter_conv_in(ops.pack_conv_in_weight(w4), b, x.data_ptr(), t.data_ptr(), temb, xc, out, Cc, H, W, 1.0, 10000.0)
    want = F.conv2d(x.float(), w4.float(), b.float(), padding=1).permute(0, 2, 3, 1).reshape(n, H * W, N)
    r = _cmp("scatter_conv_in", out, want, 0.012)
    r2 = _cmp("temb", temb, unet.sinusoidal_embedding(t.float(), N), 0.01)
    r["temb_mean_rel"] = r2["mean_rel"]
    r["ok"] = r["ok"] and r2["ok"] and bool(torch.equal(xc, x))
    return r


@check
def unet_executor_graph_replay():
    """SDXL-class executor as ONE CUDA graph: call 1 eager, call 2 captures, call 3+ replay - the replays must track
    an input that changes in place, and a rewritten prompt must re-run the (eager) K/V precompute."""
    from ..exec.unet_exec import UNetExecutor
    from ..models import unet
    cfg = unet.mini_sdxl_config()
    torch.manual_seed(5)
    m = unet.UNetModel(**cfg).to(device=_dev(), dtype=torch.bfloat16).eval()
    ex = UNetExecutor(m, _dev(), cuda_graphs=True)
    inp = unet.example_inputs(cfg, 2, 256, 256, ctx_len=77, device=_dev(), dtype=torch.bfloat16)
    sig = torch.tensor([[14.6, 10.0], [14.6, 10.0]], device=_dev())
    ref, ref2 = UNetExecutor(m, _dev(), cuda_graphs=False), UNetExecutor(m, _dev(), cuda_graphs=False)
    ok, worst, floor, drift = True, 0.0, 0.0, 0.0
    prev = None
    for it in range(5):
        inp["x"].mul_(0.9)
        if it == 3:
            inp["context"].mul_(-1.0)                       # new prompt, same buffer
            for e_ in (ex, ref, ref2):
                e_.invalidate_conditioning()
        got = ex.denoise_step(inp["x"], inp["timesteps"], inp["context"], inp["y"], sig).clone()
        want = ref.denoise_step(inp["x"], inp["timesteps"], inp["context"], inp["y"], sig).clone()
        again = ref2.denoise_step(inp["x"], inp["timesteps"], inp["context"], inp["y"], sig).clone()
        torch.cuda.synchronize()
        scale = want.float().abs().mean().item() + 1e-6
        # every kernel on this path is deterministic (the cluster GroupNorm folds its partial sums in a fixed order), so
        # a graph replay must reproduce eager launches bit for bit; `drift` shows the inputs really changed between steps
        d = (got.float() - want.float()).abs().max().item() / scale
        nf = (again.float() - want.float()).abs().max().item() / scale
        if prev is not None:
            drift = max(drift, (want.float() - prev).abs().mean().item() / scale)
        prev = want.float()
        worst, floor = max(worst, d), max(floor, nf)
        ok = ok and d == 0.0 and nf == 0.0
    ok = ok and drift > 1e-3
    return dict(name="unet_executor_graph_replay", ok=bool(ok and len(ex._graphs) == 1 and ex._graphs.replays >= 3
                                                          and ex.fused_in),
                max_rel_graph_vs_eager=worst, max_rel_eager_vs_eager=floor, step_to_step_drift=drift,
                captured=len(ex._graphs), replays=ex._graphs.replays, fused_conv_in=bool(ex.fused_in),
                launches=ex.launches_per_step)


@check
def dit_executors_graph_replay():
    """WAN and Z-Image executors: eager -> capture -> replay give bit-identical results to eager launches while the
    latent changes in place and the conditioning is rewritten (eager K/V / caption precompute outside the graph)."""
    from ..exec.wan_exec import WanExecutor
    from ..exec.zimage_exec import ZImageExecutor
    from ..models import wan, zimage
    res, ok = {}, True
    torch.manual_seed(6)
    wp = wan.wan_tiny_params()
    wm = wan.WanModel(wp).to(device=_dev(), dtype=torch.bfloat16).eval()
    zp = zimage.zimage_tiny_params()
    zm = zimage.ZImageModel(zp).to(device=_dev(), dtype=torch.bfloat16).eval()
    cases = (("wan", WanExecutor, wm, wan.example_inputs(wp, 2, 4, 128, 128, device=_dev(), dtype=torch.bfloat16)),
             ("zimage", ZImageExecutor, zm, zimage.example_inputs(zp, 2, 256, 256, cap_len=32, device=_dev(),
                                                                   dtype=torch.bfloat16)))
    for name, cls, model, inp in cases:
        ex, ref = cls(model, _dev(), cuda_graphs=True), cls(model, _dev(), cuda_graphs=False)
        sig = torch.tensor([[1.0, 0.9]] * 2, device=_dev())
        worst = 0.0
        for it in range(5):
            inp["x"].mul_(0.9)
            if it == 3:
                inp["context"].mul_(-1.0)
                ex.invalidate_conditioning()
                ref.invalidate_conditioning()
            got = ex.denoise_step(inp["x"], inp["timesteps"], inp["context"], sig).clone()
            want = ref.denoise_step(inp["x"], inp["timesteps"], inp["context"], sig).clone()
            torch.cuda.synchronize()
            worst = max(worst, (got.float() - want.float()).abs().max().item())
        res[name] = dict(max_abs=worst, captured=len(ex._graphs), replays=ex._graphs.replays)
        ok = ok and worst == 0.0 and len(ex._graphs) == 1 and ex._graphs.replays >= 3
    return dict(name="dit_executors_graph_replay", ok=bool(ok), **res)


@check
def lookalike_models_get_native_executors():
    """A FLUX / UNet rebuilt out of FOREIGN classes (no ``params``, no ``pa_family`` - what a ComfyUI model looks like
    to us) must be recognised structurally, get the native executor and reproduce the fp32 oracle."""
    from .. import exec as native_exec
    from ..models import flux, unet
    from .lookalike import launder
    torch.manual_seed(7)
    p = flux.FluxParams(in_channels=64, out_channels=64, vec_in_dim=768, context_in_dim=512, hidden_size=512,
                        mlp_ratio=4.0, num_heads=4, depth=1, depth_single_blocks=2)
    m = flux.Flux(p).to(device=_dev(), dtype=torch.bfloat16).eval()
    oracle = flux.Flux(p).to(device=_dev(), dtype=torch.float32).eval()
    oracle.load_state_dict({k: v.float() for k, v in m.state_dict().items()})
    foreign = launder(m)
    build = native_exec.builder_for(foreign)
    if build is None or isinstance(foreign, flux.Flux) or hasattr(foreign, "params"):
        return dict(name="lookalike_models_get_native_executors", ok=False, why="foreign FLUX not recognised")
    ex = build(foreign, _dev())
    inp = flux.example_inputs(p, 2, 256, 256, txt_len=64, device=_dev(), dtype=torch.bfloat16)
    with torch.no_grad():
        r = _cmp("lookalike_flux", ex(**inp), oracle(**{k: v.float() for k, v in inp.items()}), 0.03)
    cfg = unet.mini_sdxl_config()
    um = unet.UNetModel(**cfg).to(device=_dev(), dtype=torch.bfloat16).eval()
    uo = unet.UNetModel(**cfg).to(device=_dev(), dtype=torch.float32).eval()
    uo.load_state_dict({k: v.float() for k, v in um.state_dict().items()})
    fu = launder(um)
    ub = native_exec.builder_for(fu)
    if ub is None:
        return dict(name="lookalike_models_get_native_executors", ok=False, why="foreign UNet not recognised")
    uex = ub(fu, _dev())
    ui = unet.example_inputs(cfg, 2, 256, 256, ctx_len=77, device=_dev(), dtype=torch.bfloat16)
    with torch.no_grad():
        r2 = _cmp("lookalike_unet", uex(**ui), uo(**{k: v.float() for k, v in ui.items()}), 0.03)
    r["unet_mean_rel"] = r2["mean_rel"]
    r["ok"] = r["ok"] and r2["ok"]
    return r


@check
def mxfp8_fused_quant_epilogues():
    """Producers that emit the NEXT GEMM's MXFP8 A operand themselves: GELU epilogue (224-wide tiles), the GELU'd MLP
    half of the single-block linear1 (drain-first QKV epilogue) and the attention epilogue.  The dequantised result
    must match the fp32 reference to e4m3 precision, and agree with quantising the bf16 output separately."""
    import torch.nn.functional as F
    C_ = ops.require()
    dev = _dev()
    B, rows, K, N = 2, 200, 512, 896
    a, w, bias = _rand(B, rows, K), _rand(N, K, scale=0.06), _rand(N)
    aq, sfa = ops.quantize_mxfp8(a)
    wq, wsf = ops.quantize_mxfp8(w, 224)
    out8 = torch.zeros(B, rows, N, dtype=torch.uint8, device=dev)
    sf8 = torch.zeros(B * ((rows + 127) // 128) * (N // 128) * 512, dtype=torch.uint8, device=dev)
    ops.gemm_fp8(aq, sfa, wq, wsf, "gelu", 224, bias=bias, out8=out8, sf8=sf8)
    ref = F.gelu(ops.dequantize_mxfp8(aq, sfa) @ ops.dequantize_mxfp8(wq, wsf, 224)[0].t() + bias.float(), approximate="tanh")
    r = _cmp("gelu_fp8out", ops.dequantize_mxfp8(out8, sf8), ref, 0.06, hard=16.0)
    # single-block linear1: 2 heads of qkv + 256 MLP columns, fp8 MLP half lands at column offset 256 of a [B, L, 512] buffer
    H, L = 2, 256
    hid = H * 128
    a1, w1 = _rand(B, L, hid), _rand(3 * hid + 256, hid, scale=0.08)
    b1 = _rand(3 * hid + 256)
    aq1, sfa1 = ops.quantize_mxfp8(a1)
    wq1, wsf1 = ops.quantize_mxfp8(w1, 256)
    q, k, v = (torch.zeros(B, H, L, 128, dtype=torch.bfloat16, device=dev) for _ in range(3))
    qs, ks = _rand(128) + 1.0, _rand(128) + 1.0
    cat8 = torch.zeros(B, L, hid + 256, dtype=torch.uint8, device=dev)
    cat8_sf = torch.zeros(B * (L // 128) * ((hid + 256) // 128) * 512, dtype=torch.uint8, device=dev)
    ops.gemm_fp8(aq1, sfa1, wq1, wsf1, "qkv_rope", 256, bias=b1, q=q, k=k, v=v, q_scale=qs, k_scale=ks,
                 rope=_rope_table(L, dev)[1], seq_off=0, out8=cat8, sf8=cat8_sf, out8_col_off=hid)
    y = ops.dequantize_mxfp8(aq1, sfa1) @ ops.dequantize_mxfp8(wq1, wsf1, 256)[0].t() + b1.float()
    r2 = _cmp("l1_mlp_fp8out", ops.dequantize_mxfp8(cat8, cat8_sf)[:, :, hid:], F.gelu(y[:, :, 3 * hid:], approximate="tanh"),
              0.06, hard=16.0)
    # attention with MX-quantised output into columns [0, hid) of the same buffer
    C_.attention_fp8out(q, k, v, cat8, cat8_sf, 128 ** -0.5)
    want = F.scaled_dot_product_attention(q.float(), k.float(), v.float()).permute(0, 2, 1, 3).reshape(B, L, hid)
    r3 = _cmp("attention_fp8out", ops.dequantize_mxfp8(cat8, cat8_sf)[:, :, :hid], want, 0.06, hard=16.0)
    # LayerNorm + modulate with MXFP8 output
    xl, sc, sh = _rand(B, 300, 768), _rand(B, 768, scale=0.3), _rand(B, 768, scale=0.3)
    q8 = torch.zeros(B, 300, 768, dtype=torch.uint8, device=dev)
    s8 = torch.zeros(B * 3 * 6 * 512, dtype=torch.uint8, device=dev)
    C_.layernorm_modulate_fp8(xl, q8, s8, sc, sh, 1e-6)
    lw = F.layer_norm(xl.float(), (768,), eps=1e-6) * (1 + sc.float()[:, None]) + sh.float()[:, None]
    r4 = _cmp("ln_mod_fp8out", ops.dequantize_mxfp8(q8, s8), lw, 0.06, hard=16.0)
    r["l1_mlp_mean_rel"], r["attention_mean_rel"], r["ln_mean_rel"] = r2["mean_rel"], r3["mean_rel"], r4["mean_rel"]
    r["ok"] = r["ok"] and r2["ok"] and r3["ok"] and r4["ok"] and max(r["mean_rel"], r2["mean_rel"], r3["mean_rel"],
                                                                   r4["mean_rel"]) < 0.035
    return r


@check
def groupnorm_cluster_shapes():
    """Cluster / DSMEM GroupNorm(+SiLU) kernel across the SDXL and VAE channel counts, ragged H*W, batch 1..16 (small
    batches split a sample's channels over several clusters), vs torch group_norm in fp32; plus its memory throughput at
    the SDXL 128x128x320 shape (algorithmic bytes = one read + one write)."""
    res, ok = {}, True
    for B, C, HW, G, silu in ((1, 320, 999, 32, True), (2, 640, 1024, 32, True), (3, 960, 517, 32, False),
                              (2, 1280, 256, 32, True), (1, 1920, 300, 32, True), (2, 2560, 64, 32, True),
                              (2, 128, 4099, 32, True), (5, 512, 700, 32, False), (16, 320, 640, 32, True)):
        x = _rand(B, HW, C, seed=C)
        g, b = _rand(C, seed=1) + 1.0, _rand(C, seed=2)
        out = ops.groupnorm_silu(x, g, b, G, 1e-5, silu)
        want = F.group_norm(x.float().permute(0, 2, 1), G, g.float(), b.float(), 1e-5)
        want = (F.silu(want) if silu else want).permute(0, 2, 1)
        r = _cmp(f"gn_{B}x{HW}x{C}", out, want, 0.012)
        res[f"{B}x{HW}x{C}"] = round(r["mean_rel"], 5)
        ok = ok and r["ok"]
    x = _rand(16, 16384, 320)
    g, b = _rand(320) + 1.0, _rand(320)
    out = torch.empty_like(x)
    for _ in range(3):
        ops.groupnorm_silu(x, g, b, 32, 1e-5, True, out=out)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        ops.groupnorm_silu(x, g, b, 32, 1e-5, True, out=out)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 10
    return dict(name="groupnorm_cluster_shapes", ok=bool(ok), mean_rel=res, sdxl_16x16384x320_ms=round(ms, 4),
                algorithmic_gbs=round(2 * x.numel() * 2 / ms / 1e6, 1))


@check
def wan_zimage_executors_fp8():
    """WAN and Z-Image executors with MXFP8 block GEMMs (qkv via the drain-first 256-wide tiles for Z-Image, SwiGLU on
    256-wide tiles, everything else on double-buffered 224-wide tiles) vs the fp32 oracle and vs their bf16 executors."""
    from ..exec.wan_exec import WanExecutor
    from ..exec.zimage_exec import ZImageExecutor
    from ..models import wan, zimage
    res, ok = {}, True
    torch.manual_seed(8)
    wp = wan.wan_tiny_params()
    zp = zimage.zimage_tiny_params()
    cases = (("wan", WanExecutor, wan.WanModel, wp, wan.example_inputs(wp, 2, 8, 128, 192, device=_dev(), dtype=torch.bfloat16)),
             ("zimage", ZImageExecutor, zimage.ZImageModel, zp,
              zimage.example_inputs(zp, 2, 256, 256, cap_len=32, device=_dev(), dtype=torch.bfloat16)))
    for name, cls, mcls, params, inp in cases:
        m = mcls(params).to(device=_dev(), dtype=torch.bfloat16).eval()
        oracle = mcls(params).to(device=_dev(), dtype=torch.float32).eval()
        oracle.load_state_dict({k: v.float() for k, v in m.state_dict().items()})
        ex8, ex16 = cls(m, _dev(), fp8=True), cls(m, _dev())
        with torch.no_grad():
            got8, got16 = ex8(**inp), ex16(**inp)
            want = oracle(**{k: v.float() for k, v in inp.items()})
        r8, r16 = _cmp(name + "_fp8", got8, want, 0.03), _cmp(name + "_bf16", got16, want, 1.0)
        nq = sum(1 for k in ex8.W if k.endswith(".q"))
        res[name] = dict(fp8_mean_rel=r8["mean_rel"], bf16_mean_rel=r16["mean_rel"], fp8_max_rel=r8["max_rel"], n_fp8_weights=nq)
        ok = ok and r8["ok"] and nq > 0 and r8["mean_rel"] <= 3.0 * r16["mean_rel"] + 2e-3
    return dict(name="wan_zimage_executors_fp8", ok=bool(ok), **res)


@check
def cross_attention_cluster_kv():
    """Small-KV cross-attention kernel (CTA pairs sharing one multicast K/V tile): SDXL shapes (77 keys, head_dim 64,
    strided q/k/v views of fused projections), a ragged query length and key counts on both sides of the 64-row halves,
    vs SDPA in fp32; and its time against the general kernel at the SDXL 1024-query shape."""
    import os
    res, ok = {}, True
    for B, H, Lq, Lk in ((2, 20, 1024, 77), (1, 10, 4096, 77), (3, 5, 333, 40), (2, 4, 256, 128), (1, 2, 128, 64)):
        inner = H * 64
        qf = _rand(B, Lq, inner, seed=Lq)
        kvf = _rand(B, Lk, 2 * inner, seed=Lk)
        q = qf.view(B, Lq, H, 64).permute(0, 2, 1, 3)
        kv5 = kvf.view(B, Lk, 2, H, 64)
        k, v = kv5[:, :, 0].permute(0, 2, 1, 3), kv5[:, :, 1].permute(0, 2, 1, 3)
        got = ops.attention(q, k, v, variant=5)
        want = F.scaled_dot_product_attention(q.float(), k.float(), v.float()).permute(0, 2, 1, 3).reshape(B, Lq, inner)
        r = _cmp(f"xattn_{B}x{H}x{Lq}x{Lk}", got, want, 0.02)
        res[f"{B}x{H}x{Lq}x{Lk}"] = round(r["mean_rel"], 5)
        ok = ok and r["ok"]
    B, H, Lq, Lk = 16, 20, 1024, 77
    q = _rand(B, H, Lq, 64)
    k, v = _rand(B, H, Lk, 64, seed=1), _rand(B, H, Lk, 64, seed=2)
    out = torch.empty(B, Lq, H * 64, dtype=torch.bfloat16, device=_dev())
    times = {}
    for name, variant in (("cluster", 5), ("general", 4)):
        for _ in range(5):
            ops.attention(q, k, v, out=out, variant=variant)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(20):
            ops.attention(q, k, v, out=out, variant=variant)
        e1.record()
        torch.cuda.synchronize()
        times[name] = round(e0.elapsed_time(e1) / 20 * 1e3, 2)
    return dict(name="cross_attention_cluster_kv", ok=bool(ok), mean_rel=res, us_sdxl_16x20x1024x77=times)
