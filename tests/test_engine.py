"""Engine behaviour + differential tests against the unmodified reference on CPU
(SURVEY.md §4 items 1-2, Appendix A)."""
import copy
import gc
import os

import pytest
import torch
import torch.nn as nn

import comfyui_parallelanything_b200 as pa
from comfyui_parallelanything_b200.models import flux, unet
from comfyui_parallelanything_b200.parallel import pipeline as pp


class Toy(nn.Module):
    def __init__(self, d=16, n=4):
        super().__init__()
        self.hidden_size = d
        self.inp = nn.Linear(4, d)
        self.layers = nn.ModuleList([nn.Linear(d, d) for _ in range(n)])
        self.out = nn.Linear(d, 4)
        self.calls = []

    def forward(self, x, timesteps, context=None, y=None, **kw):
        self.calls.append(int(x.shape[0]))
        h = self.inp(x) + timesteps[:, None]
        if context is not None:
            h = h + context.mean(1)
        if y is not None:
            h = h + y.sum(-1, keepdim=True)
        for l in self.layers:
            h = torch.tanh(l(h))
        return self.out(h)


def chain_of(*pcts, dev="cpu"):
    c = None
    for p in pcts:
        c = pa.ParallelDevice().add_device(dev, p, c)[0]
    return c


def inputs(B, d=16):
    g = torch.Generator().manual_seed(B)
    return (torch.randn(B, 4, generator=g), torch.rand(B, generator=g),
            torch.randn(B, 3, d, generator=g), torch.randn(B, 5, generator=g))


@pytest.mark.parametrize("B", [1, 2, 3, 6, 21])
def test_matches_plain_module(B):
    m, plain = Toy(), Toy()
    plain.load_state_dict(m.state_dict())
    out, = pa.ParallelAnything().setup_parallel(m, chain_of(50, 50))
    assert out is m and m._true_parallel_active
    x, t, c, y = inputs(B)
    with torch.no_grad():
        got, want = m(x, t, context=c, y=y), plain(x, t, context=c, y=y)
    assert torch.allclose(got, want, atol=1e-6)
    pa.cleanup_parallel_model(m)


def test_differential_vs_reference():
    # weights, inputs, outputs and per-call batch sizes of the reference running this Toy on the same chain, stored
    # by baseline/make_golden.py
    golden = torch.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_differential.pt"),
                        weights_only=True)
    ours = Toy()
    ours.load_state_dict(golden["state_dict"])
    from comfyui_parallelanything_b200.utils.config import EngineConfig
    # small_batch="lead": the reference's "batch < n_devices -> lead device only" rule (ADP:1308); the default
    # ("spread") deliberately uses ``batch`` devices instead - covered by test_small_batch_spreads_over_devices
    pa.ParallelAnything().setup_parallel(ours, chain_of(40, 40, 15, 5), True, False,
                                         config=EngineConfig(small_batch="lead"))
    assert sorted(golden["cases"]) == [1, 3, 8, 21, 32]
    for B, theirs in golden["cases"].items():
        x, t, c, y = theirs["x"], theirs["t"], theirs["c"], theirs["y"]
        ours.calls.clear()
        with torch.no_grad():
            a = ours(x, t, context=c, y=y)
        assert torch.allclose(a, theirs["out"], atol=1e-6), B
        # same split decisions as the reference (cpu entries alias one replica)
        assert sorted(ours.calls) == theirs["calls"], (B, ours.calls, theirs["calls"])
    pa.cleanup_parallel_model(ours)


def test_mode_thresholds():
    from comfyui_parallelanything_b200.utils.config import EngineConfig
    m = Toy()
    pa.ParallelAnything().setup_parallel(m, chain_of(25, 25, 25, 25), config=EngineConfig(small_batch="lead"))
    x, t, c, y = inputs(3)
    m.calls.clear()
    with torch.no_grad():
        m(x, t, context=c)
    assert m.calls == [3]                      # reference rule (PA_SMALL_BATCH=lead): B < n_devices -> lead only
    x, t, c, y = inputs(4)
    m.calls.clear()
    with torch.no_grad():
        m(x, t, context=c)
    assert sorted(m.calls) == [1, 1, 1, 1]     # B == n -> DP (code behaviour, ADP:1308)
    pa.cleanup_parallel_model(m)
    m2 = Toy()
    pa.ParallelAnything().setup_parallel(m2, chain_of(50, 50), workload_split=False)
    m2.calls.clear()
    with torch.no_grad():
        m2(*inputs(8)[:2], context=None)
    assert m2.calls == [8]
    pa.cleanup_parallel_model(m2)


def test_cleanup_restores_everything():
    m = Toy()
    fwd_before = m.forward.__func__
    pa.ParallelAnything().setup_parallel(m, chain_of(50, 50))
    assert "forward" in m.__dict__
    pa.cleanup_parallel_model(m)
    assert "forward" not in m.__dict__ and m.forward.__func__ is fwd_before
    assert not any(k.startswith("_parallel") or k == "_true_parallel_active" for k in m.__dict__)
    assert all(isinstance(l, nn.Linear) for l in m.layers)
    # second setup never nests wrappers (the reference does, SURVEY A16)
    pa.ParallelAnything().setup_parallel(m, chain_of(50, 50))
    pa.ParallelAnything().setup_parallel(m, chain_of(50, 50))
    assert all(not isinstance(getattr(l, "local_block", None), pp.PipelineStage) for l in m.layers)
    pa.cleanup_parallel_model(m)


def test_finalizer_runs_on_owner_gc():
    class Patcher:
        def __init__(self, dm):
            self.model = type("BM", (), {})()
            self.model.diffusion_model = dm
            self.load_device = torch.device("cpu")
            self.patches = {}
    dm = Toy()
    p = Patcher(dm)
    out, = pa.ParallelAnything().setup_parallel(p, chain_of(50, 50))
    assert out is p and dm._true_parallel_active and p.load_device == torch.device("cpu")
    del p, out
    gc.collect()
    assert not getattr(dm, "_true_parallel_active", False)


def test_lora_patches_are_baked_before_clone():
    class Patcher:
        def __init__(self, dm):
            self.model = type("BM", (), {})()
            self.model.diffusion_model = dm
            self.load_device = torch.device("cpu")
            self.patches = {"w": 1}
            self.baked = False
        def patch_model(self, device_to=None):
            with torch.no_grad():
                self.model.diffusion_model.out.bias.add_(1.0)
            self.baked = True
    dm, plain = Toy(), Toy()
    plain.load_state_dict(dm.state_dict())
    p = Patcher(dm)
    pa.ParallelAnything().setup_parallel(p, chain_of(50, 50))
    assert p.baked
    x, t, c, y = inputs(4)
    with torch.no_grad():
        assert torch.allclose(dm(x, t, context=c), plain(x, t, context=c) + 1.0, atol=1e-6)
    # with LoRA even the home device runs on a frozen clone
    assert all(r is not dm for r in dm._parallel_replicas.values())
    pa.cleanup_parallel_model(dm)


def test_fault_injection_oom_paths(monkeypatch):
    m, plain = Toy(), Toy()
    plain.load_state_dict(m.state_dict())
    monkeypatch.setenv("PA_FAULT", "oom:1@step0")
    pa.ParallelAnything().setup_parallel(m, chain_of(50, 50))
    x, t, c, y = inputs(6)
    m.calls.clear()
    with torch.no_grad():
        got = m(x, t, context=c)               # worker 1 "OOMs" -> lead-only rerun (ADP:1435-1446)
    assert torch.allclose(got, plain(x, t, context=c), atol=1e-6)
    assert 6 in m.calls
    assert m._parallel_engine.metrics.counters.get("oom_fallbacks") == 1
    pa.cleanup_parallel_model(m)
    monkeypatch.setenv("PA_FAULT", "raise:0@step0")
    m3 = Toy()
    pa.ParallelAnything().setup_parallel(m3, chain_of(50, 50))
    with pytest.raises(RuntimeError, match="injected"):
        m3(x, t, context=c)
    pa.cleanup_parallel_model(m3)


def test_setup_oom_skips_device(monkeypatch):
    m = Toy()
    monkeypatch.setenv("PA_FAULT", "oom:cpu@setup")   # every clone target "OOMs" -> rollback
    out, = pa.ParallelAnything().setup_parallel(m, chain_of(50, 50))
    assert out is m and not getattr(m, "_true_parallel_active", False)


def test_pipeline_mode_flux_tiny_matches():
    torch.manual_seed(0)
    p = flux.flux_tiny_params()
    m = flux.Flux(p).eval()
    plain = copy.deepcopy(m)
    pa.ParallelAnything().setup_parallel(m, chain_of(50, 50))
    assert isinstance(m.double_blocks[0], pp.PipelineStage)
    inp = flux.example_inputs(p, 1, 64, 64, txt_len=8, dtype=torch.float32)
    with torch.no_grad():
        assert torch.allclose(m(**inp), plain(**inp), atol=1e-5)
    inp = flux.example_inputs(p, 4, 64, 64, txt_len=8, dtype=torch.float32)
    with torch.no_grad():
        assert torch.allclose(m(**inp), plain(**inp), atol=1e-5)
    pa.cleanup_parallel_model(m)


def test_baseline_config1_sd15_shape_two_cpu_replicas():
    """BASELINE.json config 1 plumbing (reduced width so it runs in seconds on CPU)."""
    cfg = unet.tiny_config()
    m = unet.UNetModel(**cfg).eval()
    plain = copy.deepcopy(m)
    pa.ParallelAnything().setup_parallel(m, chain_of(50, 50))
    inp = unet.example_inputs(cfg, 2, 64, 64, ctx_len=7)
    x, t, ctx = inp["x"], inp["timesteps"], inp["context"]
    with torch.no_grad():
        assert torch.allclose(m(x, t, context=ctx), plain(x, t, context=ctx), atol=1e-5)
    pa.cleanup_parallel_model(m)


def test_cfg_paired_split_keeps_pairs_together():
    from comfyui_parallelanything_b200.utils.config import EngineConfig
    m, plain = Toy(), Toy()
    plain.load_state_dict(m.state_dict())
    seen = []
    orig = Toy.forward

    def spy(self, x, timesteps, context=None, y=None, **kw):
        seen.append(x[:, 0].clone())
        return orig(self, x, timesteps, context=context, y=y, **kw)
    m.forward = spy.__get__(m, Toy)
    cfg = EngineConfig(pair_cfg=True)
    pa.ParallelAnything().setup_parallel(m, chain_of(50, 25, 25), config=cfg)
    B = 8                                            # 4 samples: cond rows 0..3, uncond rows 4..7
    x, t, c, y = inputs(B)
    x[:, 0] = torch.arange(B, dtype=torch.float32)   # tag rows with their index
    with torch.no_grad():
        got = m(x, t, context=c, y=y)
    assert torch.allclose(got, plain(x, t, context=c, y=y), atol=1e-6)
    chunks = sorted([s.tolist() for s in seen], key=lambda r: r[0])
    assert chunks == [[0.0, 1.0, 4.0, 5.0], [2.0, 6.0], [3.0, 7.0]], chunks
    assert m._parallel_engine.metrics.counters["cfg_paired_steps"] == 1
    pa.cleanup_parallel_model(m)


def test_zimage_layers_are_split_in_pipeline_mode_and_batch_split_matches():
    """Z_IMAGE is one of the reference's tested families (README); its blocks live in ``layers`` (ADP:1156)."""
    from comfyui_parallelanything_b200.models import zimage
    torch.manual_seed(0)
    p = zimage.zimage_tiny_params(dim=256, heads=2, layers=2)
    m = zimage.ZImageModel(p).eval()
    plain = copy.deepcopy(m)
    pa.ParallelAnything().setup_parallel(m, chain_of(50, 50))
    assert isinstance(m.layers[0], pp.PipelineStage)
    for batch in (1, 4):
        inp = zimage.example_inputs(p, batch, 64, 64, cap_len=8, dtype=torch.float32)
        with torch.no_grad():
            assert torch.allclose(m(**inp), plain(**inp), atol=1e-5)
    pa.cleanup_parallel_model(m)
    assert not isinstance(m.layers[0], pp.PipelineStage)


def test_small_batch_spreads_over_devices():
    """1 < batch < n_devices: the reference idles every device but the lead (ADP:1308); by default we hand one
    sample to each of the ``batch`` heaviest devices (chain order kept) and still return the plain module's result."""
    m, plain = Toy(), Toy()
    plain.load_state_dict(m.state_dict())
    pa.ParallelAnything().setup_parallel(m, chain_of(40, 40, 15, 5))
    x, t, c, y = inputs(3)
    m.calls.clear()
    with torch.no_grad():
        got, want = m(x, t, context=c, y=y), plain(x, t, context=c, y=y)
    assert torch.allclose(got, want, atol=1e-6)
    assert m.calls == [1, 1, 1]
    assert m._parallel_engine.metrics.counters.get("small_batch_spread_steps") == 1
    pa.cleanup_parallel_model(m)


def test_xpu_device_scope_matches_reference_branch(monkeypatch):
    """ADP:1398-1403: an XPU replica runs under ``torch.xpu.device(dev)`` with a synchronize before and after; cuda gets
    its device context only (ordering is done with streams / events), cpu nothing."""
    from comfyui_parallelanything_b200.parallel import workers
    calls = []

    class FakeCtx:
        def __init__(self, d):
            self.d = d

        def __enter__(self):
            calls.append(("enter", str(self.d)))

        def __exit__(self, *a):
            calls.append(("exit", str(self.d)))

    class FakeXpu:
        @staticmethod
        def device(d):
            return FakeCtx(d)

        @staticmethod
        def synchronize(d):
            calls.append(("sync", str(d)))

        @staticmethod
        def set_device(d):
            calls.append(("set", str(d)))

    monkeypatch.setattr(torch, "xpu", FakeXpu, raising=False)
    with workers.device_scope("xpu:1"):
        calls.append(("body", ""))
    assert calls == [("enter", "xpu:1"), ("sync", "xpu:1"), ("body", ""), ("sync", "xpu:1"), ("exit", "xpu:1")]
    calls.clear()
    workers.set_thread_device("xpu:0")
    assert calls == [("set", "xpu:0")]
    calls.clear()
    with workers.device_scope("cpu"):
        pass
    assert calls == []


def test_failed_sequence_parallel_step_falls_back_and_disables_itself():
    """A batch-1 step whose sequence-parallel path fails (stalled peer caught by the flag watchdog, failed capture, ...)
    must still return the right sample - recomputed by the layer-split / lead path - and must not be tried again."""
    m, plain = Toy(), Toy()
    plain.load_state_dict(m.state_dict())
    pa.ParallelAnything().setup_parallel(m, chain_of(50, 50))
    eng = m._parallel_engine

    class Broken:
        family = "fake"
        released = False

        def accepts(self, x, context):
            return True

        def check_polled(self):
            raise RuntimeError("sequence-parallel exchange timed out on GPU 1: 0xdead1001 (dead or stalled peer)")

        def release(self):
            Broken.released = True

    eng._ulysses = Broken()
    x, t, c, y = inputs(1)
    with torch.no_grad():
        got = m(x, t, context=c, y=y)
        assert torch.allclose(got, plain(x, t, context=c, y=y), atol=1e-6)
        assert eng._ulysses is None and Broken.released
        assert eng.metrics.counters.get("ulysses_fallbacks", 0) == 1
        got2 = m(x, t, context=c, y=y)                  # the next batch-1 step goes straight to the layer-split mode
        assert torch.allclose(got2, got, atol=1e-6)
    assert eng.metrics.counters.get("ulysses_fallbacks", 0) == 1
    pa.cleanup_parallel_model(m)
