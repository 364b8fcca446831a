"""WAN2.2 TI2V (48 latent channels in and out, one timestep per latent frame) through the ComfyUI-facing path and the
SPMD engine: native replicas, fused data-parallel, the batch-2 CFG split, batch-1 sequence parallelism and the
one-process-per-GPU engine.  The kernel and executor checks run from utils/selfcheck.py (tests/test_gpu_kernels.py)."""
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


def _ti2v_model(dev, seed=0):
    torch.manual_seed(seed)
    p = dataclasses.replace(wan.wan_tiny_params(), in_dim=48, out_dim=48)
    m = wan.WanModel(p).to(device=dev, dtype=torch.bfloat16).eval()
    return p, m, copy.deepcopy(m).float()


def _rel(got, want):
    """Worst per-frame mean error: a per-sample modulation lookup is wrong on some frames only."""
    return max((got[:, :, f].float() - want[:, :, f]).abs().mean().item() / want[:, :, f].abs().mean().item()
               for f in range(want.shape[2]))


def _inputs(p, batch, dev, it=0):
    inp = wan.ti2v_inputs(p, batch, frames=9, height=256, width=320, device=dev, dtype=torch.bfloat16)
    inp["timesteps"][:, 1:] = 700.0 - 100.0 * it
    return inp


def _through_nodes(devs, batch, calls=4, config=None):
    """setup_parallel on the tiny TI2V model; ``calls`` hooked forwards with the latent and the per-frame timesteps
    changed in place."""
    p, m, oracle = _ti2v_model(devs[0])
    pa.ParallelAnything().setup_parallel(m, _chain(devs), config=config)
    eng = m._parallel_engine
    assert all(getattr(r, "pa_native", False) for r in eng.replicas.values()), "expected native WAN TI2V executors"
    inp = _inputs(p, batch, devs[0])
    with torch.no_grad():
        for it in range(calls):
            inp["x"].mul_(0.97)
            inp["timesteps"][:, 1:] = 700.0 - 100.0 * it
            got = m(inp["x"], inp["timesteps"], context=inp["context"]).clone()
        want = oracle(**{k: v.float() for k, v in inp.items()})
    torch.cuda.synchronize()
    assert tuple(got.shape) == tuple(inp["x"].shape)
    rel = _rel(got, want)
    pa.cleanup_parallel_model(m)
    return rel, eng


def test_single_gpu_native_ti2v_through_nodes():
    rel, _ = _through_nodes(["cuda:0"], 2)
    assert rel < 0.03, rel


@pytest.mark.multigpu
def test_multi_gpu_fused_dp_ti2v():
    """[B, T] timesteps split along the batch with the latent; the fused path stages them by shape and replays."""
    n = min(torch.cuda.device_count(), 4)
    rel, eng = _through_nodes([f"cuda:{i}" for i in range(n)], 2 * n + 1, calls=5)
    assert rel < 0.03, rel
    assert any(r.get("fused") for r in eng.metrics.rows), "fused in-process path was not taken"
    assert eng.metrics.counters.get("native_graph_steps", 0) > 0, eng.metrics.counters


@pytest.mark.multigpu
def test_multi_gpu_cfg_batch2_ti2v():
    """cond / uncond of one clip (batch 2): one sample per GPU."""
    n = min(torch.cuda.device_count(), 4)
    rel, _ = _through_nodes([f"cuda:{i}" for i in range(n)], 2)
    assert rel < 0.03, rel


@pytest.mark.multigpu
@pytest.mark.parametrize("fp8", [False, True])
def test_batch1_sequence_parallel_ti2v(fp8):
    """Batch 1 on two GPUs: L = 3 frames x 80 tokens = 240, so GPU 1's 120-token slice starts in the middle of frame 1
    and must read frame 1's and then frame 2's modulation vectors.  A new latent and new timesteps every step, graphs
    replayed, result bit-identical to the lead replica alone."""
    from comfyui_parallelanything_b200.utils.config import EngineConfig
    devs = ["cuda:0", "cuda:1"]
    p, m, oracle = _ti2v_model(devs[0])
    pa.ParallelAnything().setup_parallel(m, _chain(devs), config=EngineConfig(fp8=fp8, batch1_mode="ulysses"))
    eng = m._parallel_engine
    assert eng._ulysses is not None and eng._ulysses.family == "wan", "sequence-parallel WAN path was not set up"
    lead = eng.slots[0].replica
    rels = []
    with torch.no_grad():
        for it in range(5):
            inp = _inputs(p, 1, devs[0], it)
            inp["x"].mul_(1.0 - 0.1 * it)
            assert inp["x"].shape[2] * (inp["x"].shape[3] // 2) * (inp["x"].shape[4] // 2) == 240
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
def test_spmd_ti2v_fused_matches_single_gpu():
    n = min(torch.cuda.device_count(), 4)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}",
           "--master-addr", "127.0.0.1", "--master-port", "29543", os.path.join(ROOT, "tools", "spmd_check.py"),
           "wan_ti2v"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    lines = [l for l in r.stdout.splitlines() if l.startswith("PA_SPMD ")]
    assert lines, r.stdout[-2000:] + r.stderr[-2000:]
    res = json.loads(lines[-1][len("PA_SPMD "):])
    assert res["ok"] and res["world"] == n and res["family"] == "wan_ti2v", res
    for name, v in res["results"].items():
        assert v["mean_rel"] < 5e-3, (name, v)
