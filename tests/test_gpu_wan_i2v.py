"""WAN2.2 image-to-video (36-channel input, 16-channel output) through the ComfyUI-facing path and the SPMD engine:
native replicas, fused data-parallel, the batch-2 CFG split, batch-1 sequence parallelism and the one-process-per-GPU
engine.  The kernel and executor checks run from utils/selfcheck.py (tests/test_gpu_kernels.py)."""
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


def _chain(devs):
    c = None
    for d in devs:
        c = pa.ParallelDevice().add_device(d, 100.0 / len(devs), c)[0]
    return c


def _i2v_model(dev, seed=0):
    torch.manual_seed(seed)
    p = dataclasses.replace(wan.wan_tiny_params(), in_dim=36)
    m = wan.WanModel(p).to(device=dev, dtype=torch.bfloat16).eval()
    return p, m, copy.deepcopy(m).float()


def _rel(got, want):
    return (got.float() - want).abs().mean().item() / want.abs().mean().item()


def _through_nodes(devs, batch, calls=4, config=None):
    """setup_parallel on the tiny I2V model; ``calls`` hooked forwards with the noise channels changed in place."""
    p, m, oracle = _i2v_model(devs[0])
    pa.ParallelAnything().setup_parallel(m, _chain(devs), config=config)
    eng = m._parallel_engine
    assert all(getattr(r, "pa_native", False) for r in eng.replicas.values()), "expected native WAN I2V executors"
    inp = wan.i2v_inputs(p, batch, frames=8, height=64, width=96, device=devs[0], dtype=torch.bfloat16)
    with torch.no_grad():
        for _ in range(calls):
            inp["x"][:, :16].mul_(0.97)
            got = m(inp["x"], inp["timesteps"], context=inp["context"]).clone()
        want = oracle(**{k: v.float() for k, v in inp.items()})
    torch.cuda.synchronize()
    assert tuple(got.shape) == (batch, 16) + tuple(inp["x"].shape[2:])
    rel = _rel(got, want)
    pa.cleanup_parallel_model(m)
    return rel, eng


def test_single_gpu_native_i2v_through_nodes():
    rel, _ = _through_nodes(["cuda:0"], 2)
    assert rel < 0.03, rel


@pytest.mark.multigpu
def test_multi_gpu_fused_dp_i2v():
    n = min(torch.cuda.device_count(), 4)
    rel, eng = _through_nodes([f"cuda:{i}" for i in range(n)], 2 * n + 1)
    assert rel < 0.03, rel
    assert any(r.get("fused") for r in eng.metrics.rows), "fused in-process path was not taken"


@pytest.mark.multigpu
def test_multi_gpu_cfg_batch2_i2v():
    """cond / uncond of one clip (batch 2): one sample per GPU."""
    n = min(torch.cuda.device_count(), 4)
    rel, _ = _through_nodes([f"cuda:{i}" for i in range(n)], 2)
    assert rel < 0.03, rel


@pytest.mark.multigpu
@pytest.mark.parametrize("fp8", [False, True])
def test_batch1_sequence_parallel_i2v(fp8):
    """Batch 1 on two GPUs: the 36-channel clip is patchified whole and each GPU embeds its token slice; a new latent
    tensor every step, graphs replayed, result bit-identical to the lead replica alone."""
    from comfyui_parallelanything_b200.utils.config import EngineConfig
    devs = ["cuda:0", "cuda:1"]
    p, m, oracle = _i2v_model(devs[0])
    pa.ParallelAnything().setup_parallel(m, _chain(devs), config=EngineConfig(fp8=fp8, batch1_mode="ulysses"))
    eng = m._parallel_engine
    assert eng._ulysses is not None and eng._ulysses.family == "wan", "sequence-parallel WAN path was not set up"
    lead = eng.slots[0].replica
    base = wan.i2v_inputs(p, 1, frames=8, height=64, width=64, device=devs[0], dtype=torch.bfloat16)
    rels = []
    with torch.no_grad():
        for it in range(5):
            inp = {k: v.clone() for k, v in base.items()}
            inp["x"][:, :16].mul_(1.0 - 0.1 * it)
            got = m(inp["x"], inp["timesteps"], context=inp["context"])
            alone = lead(inp["x"], inp["timesteps"], context=inp["context"])
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
def test_spmd_i2v_fused_matches_single_gpu():
    n = min(torch.cuda.device_count(), 4)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}",
           "--master-addr", "127.0.0.1", "--master-port", "29541", os.path.join(ROOT, "tools", "spmd_check.py"),
           "wan_i2v"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    lines = [l for l in r.stdout.splitlines() if l.startswith("PA_SPMD ")]
    assert lines, r.stdout[-2000:] + r.stderr[-2000:]
    res = json.loads(lines[-1][len("PA_SPMD "):])
    assert res["ok"] and res["world"] == n and res["family"] == "wan_i2v", res
    for name, v in res["results"].items():
        assert v["mean_rel"] < 5e-3, (name, v)
