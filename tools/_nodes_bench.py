"""Shared `--api nodes` arm of tools/bench_{wan,zimage}.py: ONE process, the `Parallel Anything` node hooks the model's
forward, a sampler-like loop calls it with a NEW latent tensor every step and does the Euler update on the lead GPU
(batch 1 -> sequence-parallel over all GPUs of the chain).  Same JSON line as bench.py."""
from __future__ import annotations

import os
import time


def run(a, hb, model_name: str, build_model, host: dict, config: dict) -> int:
    """``build_model(lead_device) -> nn.Module``; ``host``: pinned inputs x / timesteps / context / sig (+ clip_fea for
    WAN2.1 I2V / FLF2V, passed on every call like the sampler's conditioning)."""
    hb.quiet_stdout()
    rank, world, _local = hb.dist_env()
    if hb.host_only_group(rank, world):
        return 0
    import torch
    import comfyui_parallelanything_b200 as pa
    lead = torch.device("cuda:0")
    torch.cuda.set_device(lead)
    torch.manual_seed(1234)
    t0 = time.perf_counter()
    model = build_model(lead)
    chain = None
    for i in range(a.gpus):
        chain = pa.ParallelDevice().add_device(f"cuda:{i}", 100.0 / a.gpus, chain)[0]
    if a.dtype == "fp8":
        os.environ["PA_FP8"] = "1"
    (model,) = pa.ParallelAnything().setup_parallel(model, chain, True, False, True, False)
    for i in range(a.gpus):
        torch.cuda.synchronize(i)
    setup_s = round(time.perf_counter() - t0, 2)
    eng = model._parallel_engine
    d = {k: v.to(lead) for k, v in host.items()}
    stage = {k: torch.empty_like(v, device=lead) for k, v in host.items()}
    result_host = torch.empty(tuple(host["x"].shape), dtype=torch.bfloat16).pin_memory()
    ones = (1,) * (host["x"].dim() - 1)

    def euler(x, e, sig):
        # image-to-video models see [noise | mask | image latent] and predict the noise channels only: the update covers
        # those, and the conditioning channels are concatenated back for the next call, as ComfyUI's sampler does
        nxt = x[:, :e.shape[1]] + (sig[:, 1] - sig[:, 0]).view(-1, *ones).to(x.dtype) * e
        return nxt if nxt.shape[1] == x.shape[1] else torch.cat([nxt, x[:, e.shape[1]:]], 1)

    cond = {k: d[k] for k in ("clip_fea",) if k in d}                  # step-invariant extra conditioning
    cond_e2e = {k: stage[k] for k in cond}
    state = {"x": d["x"]}

    def step_device():
        with torch.no_grad():
            x = state["x"]
            e = model(x, d["timesteps"], context=d["context"], **cond)
            state["x"] = euler(x, e, d["sig"])

    def step_e2e():
        with torch.no_grad():
            fresh = {k: torch.empty_like(v) for k, v in stage.items() if k in ("x", "timesteps")}
            for k in stage:
                (fresh.get(k, stage[k])).copy_(host[k], non_blocking=True)
            e = model(fresh["x"], fresh["timesteps"], context=stage["context"], **cond_e2e)
            result_host.copy_(euler(fresh["x"], e, stage["sig"]), non_blocking=True)

    def sync_all():
        for i in range(a.gpus):
            torch.cuda.synchronize(i)

    def timed_local(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        sync_all()
        return e0.elapsed_time(e1) / steps

    sampler = hb.ClockSampler()
    sampler.start()
    ms = timed_local(step_device, a.steps, max(a.warmup, 4))
    ms_e2e = timed_local(step_e2e, a.steps, max(3, a.warmup // 2))
    clocks = sampler.stop(a.gpus)
    extra = {}
    if a.gpus > 1:
        with torch.no_grad():
            got = model(d["x"], d["timesteps"], context=d["context"], **cond).clone()
            want = eng.slots[0].replica(d["x"], d["timesteps"], context=d["context"], **cond).clone()
        sync_all()
        extra["output_matches_n1"] = hb.rel_err(got, want)
    if getattr(eng, "_ulysses", None) is not None:
        eng._ulysses.check_error()
    desc = eng.describe() if hasattr(eng, "describe") else {}
    h2d = sum(v.numel() * v.element_size() for v in host.values())
    d2h = result_host.numel() * result_host.element_size()
    B = host["x"].shape[0]
    pa.cleanup_parallel_model(model)
    hb.host_only_release(world)
    cfg = dict(config)
    cfg["parallelism"] = f"one process, node API, {a.gpus} GPU(s)" + (
        ", sequence-parallel (Ulysses)" if B == 1 and a.gpus > 1 and desc.get("counters", {}).get("ulysses_steps") else "")
    hb.emit({"metric": hb.METRIC, "value": round(1000.0 / ms, 4), "unit": "steps/s", "n_gpus": a.gpus, "steps": a.steps,
             "warmup": a.warmup, "ms_per_step": round(ms, 3), "higher_is_better": True, "scaling": "strong",
             "vs_baseline": None, "sec_per_it": round(ms / 1000.0, 4), "dtype": a.dtype,
             "data": "synthetic, random-init weights", "impl": "ours", "api": "nodes", "clocks": clocks,
             "e2e": {"value": round(1000.0 / ms_e2e, 4), "unit": "steps/s", "ms_per_step": round(ms_e2e, 3),
                     "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
             "output_finite": bool(torch.isfinite(result_host.float()).all().item()),
             "setup": {"setup_s": setup_s}, "engine": desc, **extra, "config": cfg})
    return 0
