"""WAN2.1 image-to-video with CLIP image conditioning through the ComfyUI-facing path: on one GPU the native replica
honours ``clip_fea``, prepares the image K/V once while it stays the same and again when it changes; on several GPUs
fused data parallelism, the batch-2 CFG split, batch-1 sequence parallelism and the SPMD engine carry ``clip_fea``.  Kernel and
executor checks run from utils/selfcheck.py (tests/test_gpu_kernels.py)."""
import copy
import dataclasses
import json
import os
import subprocess
import sys

import pytest
import torch

import comfyui_parallelanything_b200 as pa
from comfyui_parallelanything_b200.models import wan

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _rel(got, want):
    return (got.float() - want).abs().mean().item() / want.abs().mean().item()


@pytest.mark.parametrize("flf2v", [False, True])
def test_node_path_one_gpu_with_clip_fea(flf2v):
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    p = dataclasses.replace(wan.wan_tiny_params(), in_dim=36, clip_dim=128, clip_pos_tokens=514 if flf2v else 0)
    m = wan.WanModel(p).to(device=dev, dtype=torch.bfloat16).eval()
    oracle = copy.deepcopy(m).float()
    pa.ParallelAnything().setup_parallel(m, pa.ParallelDevice().add_device("cuda:0", 100.0, None)[0])
    eng = m._parallel_engine
    (rep,) = eng.replicas.values()
    assert getattr(rep, "pa_native", False) and type(rep).__name__ == "WanClipExecutor"
    preps = []
    orig = rep._prepare_ctx
    rep._prepare_ctx = lambda ws, *a: preps.append(orig(ws, *a)) or preps[-1]
    inp = wan.clip_inputs(p, 1, frames=8, height=64, width=96, device=dev, dtype=torch.bfloat16)
    with torch.no_grad():
        for _ in range(4):
            inp["x"][:, :16].mul_(0.97)
            got = m(inp["x"], inp["timesteps"], context=inp["context"], clip_fea=inp["clip_fea"]).clone()
        want = oracle(**{k: v.float() for k, v in inp.items()})
        assert _rel(got, want) < 0.03
        assert sum(1 for n in preps if n) == 1, preps         # constant clip_fea: image K/V prepared once
        other = torch.randn_like(inp["clip_fea"])
        got2 = m(inp["x"], inp["timesteps"], context=inp["context"], clip_fea=other).clone()
        want2 = oracle(**{k: v.float() for k, v in dict(inp, clip_fea=other).items()})
    assert sum(1 for n in preps if n) == 2
    assert _rel(got2, want2) < 0.03 and _rel(got2, want) > 0.01          # no stale image K/V


# ------------------------------------------------------------------ several GPUs


def _chain(devs):
    c = None
    for d in devs:
        c = pa.ParallelDevice().add_device(d, 100.0 / len(devs), c)[0]
    return c


def _clip_model(dev, flf2v=False, seed=0):
    torch.manual_seed(seed)
    p = dataclasses.replace(wan.wan_tiny_params(), in_dim=36, clip_dim=128, clip_pos_tokens=514 if flf2v else 0)
    m = wan.WanModel(p).to(device=dev, dtype=torch.bfloat16).eval()
    return p, m, copy.deepcopy(m).float()


def _through_nodes(devs, batch, calls=6, config=None):
    """setup_parallel on the tiny I2V + CLIP model; ``calls`` hooked forwards with the same context / clip_fea tensors
    and the noise channels changed in place, as a sampler does."""
    p, m, oracle = _clip_model(devs[0])
    pa.ParallelAnything().setup_parallel(m, _chain(devs), config=config)
    eng = m._parallel_engine
    assert all(type(r).__name__ == "WanClipExecutor" for r in eng.replicas.values())
    inp = wan.clip_inputs(p, batch, frames=8, height=64, width=96, device=devs[0], dtype=torch.bfloat16)
    with torch.no_grad():
        for _ in range(calls):
            inp["x"][:, :16].mul_(0.97)
            got = m(inp["x"], inp["timesteps"], context=inp["context"], clip_fea=inp["clip_fea"]).clone()
        want = oracle(**{k: v.float() for k, v in inp.items()})
    torch.cuda.synchronize()
    assert tuple(got.shape) == (batch, 16) + tuple(inp["x"].shape[2:])
    rel = _rel(got, want)
    pa.cleanup_parallel_model(m)
    return rel, eng


@pytest.mark.multigpu
def test_multi_gpu_fused_dp_clip():
    """Fused data parallelism: context and clip_fea are staged once, so the replicas' conditioning cache holds and the
    steps replay as native CUDA graph launches."""
    n = min(torch.cuda.device_count(), 4)
    rel, eng = _through_nodes([f"cuda:{i}" for i in range(n)], 2 * n + 1)
    assert rel < 0.03, rel
    assert any(r.get("fused") for r in eng.metrics.rows), "fused in-process path was not taken"
    assert eng.metrics.counters.get("native_graph_steps", 0) > 0, eng.metrics.counters
    assert eng.metrics.counters.get("cond_cache_hits", 0) > 0, eng.metrics.counters


@pytest.mark.multigpu
def test_multi_gpu_cfg_batch2_clip():
    """cond / uncond of one clip (batch 2): one sample per GPU, each with its own clip_fea row."""
    n = min(torch.cuda.device_count(), 4)
    rel, _ = _through_nodes([f"cuda:{i}" for i in range(n)], 2)
    assert rel < 0.03, rel


@pytest.mark.multigpu
@pytest.mark.parametrize("fp8", [False, True])
def test_batch1_sequence_parallel_clip(fp8):
    """Batch 1 on two GPUs: every GPU holds the full image K/V and attends with its own query tokens; a new latent every
    step, graphs replayed, result bit-identical to the lead replica alone."""
    from comfyui_parallelanything_b200.utils.config import EngineConfig
    devs = ["cuda:0", "cuda:1"]
    p, m, oracle = _clip_model(devs[0], flf2v=True)
    pa.ParallelAnything().setup_parallel(m, _chain(devs), config=EngineConfig(fp8=fp8, batch1_mode="ulysses"))
    eng = m._parallel_engine
    assert eng._ulysses is not None and eng._ulysses.family == "wan", "sequence-parallel WAN path was not set up"
    lead = eng.slots[0].replica
    base = wan.clip_inputs(p, 1, frames=8, height=64, width=64, device=devs[0], dtype=torch.bfloat16)
    rels = []
    with torch.no_grad():
        for it in range(5):
            inp = dict(base, x=base["x"].clone())
            inp["x"][:, :16].mul_(1.0 - 0.1 * it)
            got = m(inp["x"], inp["timesteps"], context=inp["context"], clip_fea=inp["clip_fea"])
            alone = lead(inp["x"], inp["timesteps"], context=inp["context"], clip_fea=inp["clip_fea"])
            want = oracle(**{k: v.float() for k, v in inp.items()})
            torch.cuda.synchronize()
            assert torch.equal(got, alone), (it, (got.float() - alone.float()).abs().max().item())
            rels.append(_rel(got, want))
    eng._ulysses.check_error()
    assert max(rels) < (0.05 if fp8 else 0.03), rels
    assert eng.metrics.counters.get("ulysses_steps", 0) == 5
    assert all(len(s.replica._graphs) >= 1 for s in eng.slots)
    pa.cleanup_parallel_model(m)


@pytest.mark.multigpu
def test_spmd_clip_fused_matches_single_gpu():
    n = min(torch.cuda.device_count(), 4)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}",
           "--master-addr", "127.0.0.1", "--master-port", "29543", os.path.join(ROOT, "tools", "spmd_check.py"),
           "wan_clip"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    lines = [l for l in r.stdout.splitlines() if l.startswith("PA_SPMD ")]
    assert lines, r.stdout[-2000:] + r.stderr[-2000:]
    res = json.loads(lines[-1][len("PA_SPMD "):])
    assert res["ok"] and res["world"] == n and res["family"] == "wan_clip", res
    for name, v in res["results"].items():
        assert v["mean_rel"] < 5e-3, (name, v)
