#!/usr/bin/env python
"""Headline benchmark: denoise-steps/sec of FLUX.1-dev (MM-DiT, 11.9 B params, random init),
1024x1024, global batch 8, bf16 compute, on N GPUs of one node (BASELINE.json config 3).

    python bench.py --gpus 1 --steps 5 --warmup 3                      # our engine
    python bench.py --impl reference --gpus 1 --steps 5 --warmup 3     # unmodified reference
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W         # N > 1 (both arms)

One "denoise step" = model forward on the whole batch + the sampler's Euler update
``x <- x + (sigma' - sigma) * v``.  Strong scaling: the global batch is fixed, ranks split it.

``value``  : device-timed steps/s (CUDA events, barrier + synchronize on both sides, max over ranks),
             inputs resident on the lead GPU.
``--api``  : ``spmd`` (default; one process per GPU, ``parallel/spmd.py``) or ``nodes`` (ONE process drives all N
             GPUs through the ComfyUI node API: ParallelDevice chain -> ParallelAnything.setup_parallel -> hooked
             ``model.forward`` with a NEW input tensor every step, as a sampler does).
``e2e``    : same metric through the public API with, inside the timed region of every step, the
             host(pinned)->device copy of that step's inputs and a device->host read of the result.
Both arms print one JSON line; the reference arm drives the UNMODIFIED reference
(baseline/_ref/any_device_parallel.py) wrapping the stock-torch FLUX definition from
``comfyui_parallelanything_b200.models.flux`` (the reference ships no model code of its own).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "denoise-steps/sec (device-timed, max over ranks)"
MODEL_NAME = "FLUX.1-dev DiT 1024x1024"


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self):
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self, n_gpus: int) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        try:
            self.proc.terminate()
            self.proc.wait(timeout=5)
        except Exception:
            pass
        sm, mx, reasons, power = [], [], set(), []
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                if int(f[0]) >= n_gpus:
                    continue
                sm.append(float(f[1]))
                mx.append(float(f[2]))
                power.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        busy = sorted(s for s, p in zip(sm, power) if p > 300) or sorted(sm)
        med = busy[len(busy) // 2] if busy else None
        return {"sm_mhz": med, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(power) if power else None}


# ----------------------------------------------------------------------------- helpers
def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", str(rank)))
    return rank, world, local


def synthetic_inputs(batch: int, pinned: bool):
    """Synthetic latents / conditioning of the named shape, created on the HOST."""
    import torch
    from comfyui_parallelanything_b200.models import flux
    p = flux.flux_dev_params()
    inp = flux.example_inputs(p, batch, 1024, 1024, txt_len=512, device="cpu", dtype=torch.bfloat16)
    sig = torch.tensor([[1.0, 0.96]] * batch, dtype=torch.float32)
    inp["sig"] = sig
    if pinned:
        inp = {k: v.pin_memory() for k, v in inp.items()}
    return p, inp


def max_over_ranks(ms: float, world: int):
    if world == 1:
        return ms
    import torch
    import torch.distributed as dist
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def barrier_sync(world: int):
    import torch
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    torch.cuda.synchronize()


def timed(fn, steps: int, warmup: int, world: int):
    """W untimed warm-up steps, then exactly K steps between CUDA events; returns ms/step (max over ranks)."""
    import torch
    for _ in range(warmup):
        fn()
    barrier_sync(world)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    barrier_sync(world)
    return max_over_ranks(e0.elapsed_time(e1), world) / steps


_REAL_STDOUT = sys.stdout


def emit(obj: dict):
    """The ONE JSON line goes to the real stdout; everything else (the reference's ``print`` chatter, our
    logger, NCCL's version banner written by C code to fd 1) is routed to stderr by ``quiet_stdout`` so the
    line stays machine-readable."""
    _REAL_STDOUT.write(json.dumps(obj) + "\n")
    _REAL_STDOUT.flush()


def quiet_stdout():
    global _REAL_STDOUT
    try:
        sys.stdout.flush()
        real_fd = os.dup(1)
        os.dup2(2, 1)                       # fd 1 -> stderr for C-level writers
        _REAL_STDOUT = os.fdopen(real_fd, "w")
    except OSError:
        pass
    sys.stdout = sys.stderr


# ----------------------------------------------------------------------------- shared
def bench_config(batch: int, n: int) -> dict:
    """Identical for both arms (the driver compares the dicts); free-text descriptions live in ``notes``."""
    return {"model": MODEL_NAME, "global_batch": batch, "seq_len": 4608, "parallelism": f"dp{n}", "params_b": 11.9,
            "l2": "no explicit flush: each step streams >= 12 GB of weights (>> 126 MB L2)"}


def make_line(args, impl, ms, ms_e2e, clocks, h2d, d2h, launches, finite, dtype, notes, extra=None) -> dict:
    value = 1000.0 / ms
    line = {"metric": METRIC, "value": round(value, 4), "unit": "steps/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms, 3), "sec_per_it": round(ms / 1e3, 4),
            "higher_is_better": True, "scaling": "strong",
            # BASELINE.md's only published numbers are Z-Image Turbo on an RTX 3090 (+V100): a different model on
            # different hardware, so there is no published number for this workload to divide by.
            "vs_baseline": None,
            "dtype": dtype, "data": "synthetic latents/conditioning of the named shape, random-init weights",
            "impl": impl, "clocks": clocks,
            "e2e": {"value": round(1000.0 / ms_e2e, 4), "unit": "steps/s", "ms_per_step": round(ms_e2e, 3),
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": launches, "output_finite": finite, "config": bench_config(args.batch, args.gpus),
            "notes": notes}
    if extra:
        line.update(extra)
    return line


def host_only_group(rank: int, world: int):
    """Ranks that must stay off the GPUs (reference arm, ``--api nodes``): a gloo group, no CUDA context, no NCCL
    communicator.  Rank != 0 sleeps in the final barrier and returns True (= caller should exit)."""
    if world <= 1:
        return False
    import datetime
    import torch.distributed as dist
    dist.init_process_group("gloo", timeout=datetime.timedelta(hours=3))
    if rank != 0:
        dist.barrier()
        dist.destroy_process_group()
        return True
    return False


def host_only_release(world: int):
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


def rel_err(a, b) -> dict:
    a, b = a.float(), b.float()
    d = (a - b).abs()
    return {"max_abs": float(d.max()), "mean_rel": float(d.mean() / (b.abs().mean() + 1e-12)),
            "max_rel_to_absmax": float(d.max() / (b.abs().max() + 1e-12))}


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, arrays: dict) -> None:
    """``--dump-outputs``: write each result as ``out_dir/<name>.npy`` in float32, so that two builds run with the same
    arguments can be compared output for output.  An array over its share of ``DUMP_BYTES`` is replaced by a fixed
    seeded sample of its flattened elements (the same positions for the same shape)."""
    if not out_dir:
        return
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    cap = DUMP_BYTES // (4 * len(arrays))
    for name, t in arrays.items():
        flat = t.detach().float().flatten().cpu()
        if flat.numel() > cap:
            idx = torch.randperm(flat.numel(), generator=torch.Generator().manual_seed(0))[:cap].sort().values
            flat = flat[idx]
        else:
            flat = flat.view(t.shape)
        np.save(os.path.join(out_dir, name + ".npy"), flat.numpy())


DTYPE_NAMES = {"bf16": "bf16", "fp8": "fp8 (MXFP8 block-scaled tcgen05 GEMMs for the block linears = 99.9% of the FLOPs; "
                                      "attention, norms, embedders bf16/fp32)"}


# ----------------------------------------------------------------------------- our arm (one process per GPU)
def measure_ours(args, dtype: str, rank: int, world: int, dev, host, params, with_clocks: bool) -> dict:
    """Build the executor (+ SPMD engine) for ``dtype``, time the device step and the end-to-end step, verify the
    multi-GPU result against the single-GPU executor, tear everything down.  Returns the measured fields."""
    import torch
    from comfyui_parallelanything_b200.exec.flux_exec import FluxExecutor
    from comfyui_parallelanything_b200.models import flux
    B = args.batch
    t_setup = time.perf_counter()
    setup = {}
    if world > 1 and args.replicate != "seed":
        # weights exist on rank 0 only; every other rank receives the PACKED executor weights device-to-device
        # (NVSwitch multicast kernel or NCCL broadcast) - the B200 answer to the reference's CPU-bounce clone loop
        from comfyui_parallelanything_b200.parallel import replicate_nvl
        torch.manual_seed(1234 if rank == 0 else 99)
        with torch.device(dev):
            model = flux.Flux(params, dtype=torch.bfloat16)
        ex = FluxExecutor(model, dev, fp8=(dtype == "fp8"), cuda_graphs=not args.no_graphs)
        del model
        torch.cuda.synchronize()
        setup = replicate_nvl.broadcast_executor(ex, src=0, method=args.replicate)
    else:
        torch.manual_seed(1234)                          # identical random-init weights on every rank
        with torch.device(dev):
            model = flux.Flux(params, dtype=torch.bfloat16)
        ex = FluxExecutor(model, dev, fp8=(dtype == "fp8"), cuda_graphs=not args.no_graphs)
        del model
    torch.cuda.empty_cache()
    torch.cuda.synchronize()
    setup["setup_s"] = round(time.perf_counter() - t_setup, 2)

    result_host = torch.empty(B, 16, 128, 128, dtype=torch.bfloat16).pin_memory()
    res = {"setup": setup}
    eng = None
    if world == 1:
        d = {k: v.to(dev) for k, v in host.items()}
        xs = ex._prep(d["x"], d["timesteps"], d["context"], d["y"], d["guidance"])
        stage = {k: torch.empty_like(v, device=dev) for k, v in host.items()}
        out_buf = torch.empty(B, 16, 128, 128, dtype=torch.bfloat16, device=dev)

        def step_device():
            ex.denoise_step(xs[0], xs[1], xs[2], xs[3], xs[4], d["sig"], out=out_buf)

        def step_e2e():
            for k in stage:
                stage[k].copy_(host[k], non_blocking=True)
            ex.denoise_step(stage["x"], stage["timesteps"], stage["context"], stage["y"], stage["guidance"],
                            stage["sig"], out=out_buf)
            result_host.copy_(out_buf, non_blocking=True)
        res["notes"] = {"parallelism": "one GPU, one CUDA graph per step",
                        "step": "model forward + Euler update (fused into the last GEMM epilogue)"}
    else:
        from comfyui_parallelanything_b200.parallel.spmd import SpmdFluxEngine
        eng = SpmdFluxEngine(ex, B, 1024, 1024, 512, backend=args.backend)
        if rank == 0:
            eng.stage_inputs(host["x"], host["timesteps"], host["context"], host["y"], host["guidance"], host["sig"])
        torch.cuda.synchronize()

        def step_device():
            eng.step()

        def step_e2e():
            if rank == 0:
                eng.stage_inputs(host["x"], host["timesteps"], host["context"], host["y"], host["guidance"],
                                 host["sig"])
            out = eng.step()
            if rank == 0:
                result_host.copy_(out, non_blocking=True)
        res["notes"] = {"parallelism": (f"one process per GPU ({args.backend}: in-kernel NVLink scatter/gather)"
                                        if args.backend == "fused" else "one process per GPU (NCCL send/recv baseline)"),
                        "step": "model forward + Euler update (fused into the last GEMM epilogue, peer stores to rank 0)"}

    sampler = ClockSampler()
    if rank == 0 and with_clocks:
        sampler.start()
    res["ms"] = timed(step_device, args.steps, args.warmup, world)
    res["ms_e2e"] = timed(step_e2e, args.steps, max(3, args.warmup // 2), world)
    res["clocks"] = sampler.stop(args.gpus) if (rank == 0 and with_clocks) else {}
    if world > 1:
        eng.check_error()
        res["launches"] = eng.comm_launches * args.steps
        # correctness of the multi-GPU result: one more SPMD step, then rank 0 recomputes the WHOLE batch on its own
        # single-GPU executor from the same staged inputs and compares with the gathered output.
        out = eng.step()
        barrier_sync(world)
        if rank == 0:
            got = out.clone()
            b = eng.buf
            want = ex.denoise_step(b["x"], b["t"], b["ctx"], b["y"], b["g"], b["sig"]).clone()
            torch.cuda.synchronize()
            res["output_matches_n1"] = rel_err(got, want)
            res["result"] = got
        barrier_sync(world)
    else:
        res["launches"] = ex.launches_per_step * args.steps
        res["result"] = out_buf.clone()
    res["finite"] = bool(torch.isfinite(result_host.float()).all().item()) if rank == 0 else True
    if eng is not None:
        eng.close()
    ex.release()
    del ex
    torch.cuda.empty_cache()
    return res


def run_ours(args) -> int:
    import torch
    rank, world, local = dist_env()
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    from comfyui_parallelanything_b200 import ops
    ops.require()
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    params, host = synthetic_inputs(args.batch, pinned=True)
    h2d = sum(v.numel() * v.element_size() for v in host.values())
    d2h = args.batch * 16 * 128 * 128 * 2
    main = measure_ours(args, args.dtype, rank, world, dev, host, params, with_clocks=True)
    extra = {"setup": main["setup"]}
    if "output_matches_n1" in main:
        extra["output_matches_n1"] = main["output_matches_n1"]
    if args.dtype == "fp8" and not args.no_bf16:
        # BASELINE config 3 names fp8, so the headline is the MXFP8 engine; the same workload in bf16 (the precision of
        # the reference arm) is measured in the same run so both comparisons can be read off one line.
        alt = measure_ours(args, "bf16", rank, world, dev, host, params, with_clocks=False)
        if rank == 0:
            extra["bf16"] = {"value": round(1000.0 / alt["ms"], 4), "unit": "steps/s", "ms_per_step": round(alt["ms"], 3),
                             "e2e_ms_per_step": round(alt["ms_e2e"], 3), "e2e_value": round(1000.0 / alt["ms_e2e"], 4)}
            extra["fp8_vs_bf16_output"] = rel_err(main["result"], alt["result"])
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()
    if rank == 0:
        dumps = {"x_next": main["result"]}
        if "bf16" in extra:
            dumps["bf16_x_next"] = alt["result"]
        dump_outputs(args.dump_outputs, dumps)
        emit(make_line(args, "ours", main["ms"], main["ms_e2e"], main["clocks"], h2d, d2h, main["launches"],
                       main["finite"], DTYPE_NAMES[args.dtype], main["notes"], extra))
    return 0


# ----------------------------------------------------------------------------- our arm, ONE process (node API)
def run_nodes(args) -> int:
    """What ComfyUI does: one process, the ParallelAnything node hooks ``model.forward``; a sampler calls it with a
    NEW latent tensor every step and does the Euler update itself on the lead GPU."""
    rank, world, local = dist_env()
    if host_only_group(rank, world):
        return 0
    import torch
    import comfyui_parallelanything_b200 as pa
    from comfyui_parallelanything_b200.models import flux
    from comfyui_parallelanything_b200.utils.config import EngineConfig
    lead = torch.device("cuda:0")
    torch.cuda.set_device(lead)
    B = args.batch
    params, host = synthetic_inputs(B, pinned=True)
    torch.manual_seed(1234)
    t_setup = time.perf_counter()
    with torch.device(lead):
        model = flux.Flux(params, dtype=torch.bfloat16).eval()
    chain = None
    for i in range(args.gpus):
        chain = pa.ParallelDevice().add_device(f"cuda:{i}", 100.0 / args.gpus, chain)[0]
    if args.dtype == "fp8":
        os.environ["PA_FP8"] = "1"
    (model,) = pa.ParallelAnything().setup_parallel(model, chain, True, False, True, False)
    for i in range(args.gpus):
        torch.cuda.synchronize(i)
    setup_s = round(time.perf_counter() - t_setup, 2)
    eng = model._parallel_engine
    d = {k: v.to(lead) for k, v in host.items()}
    stage = {k: torch.empty_like(v, device=lead) for k, v in host.items()}
    result_host = torch.empty(B, 16, 128, 128, dtype=torch.bfloat16).pin_memory()

    def euler(x, v, sig):
        return x + (sig[:, 1] - sig[:, 0]).view(-1, 1, 1, 1).to(x.dtype) * v

    state = {"x": d["x"]}

    def step_device():
        with torch.no_grad():
            x = state["x"]
            v = model(x, d["timesteps"], context=d["context"], y=d["y"], guidance=d["guidance"])
            state["x"] = euler(x, v, d["sig"])          # a NEW tensor every step, like a sampler loop

    def step_e2e():
        with torch.no_grad():
            fresh = {k: torch.empty_like(v) for k, v in stage.items() if k in ("x", "timesteps")}
            for k in stage:
                (fresh.get(k, stage[k])).copy_(host[k], non_blocking=True)
            x = fresh["x"]
            v = model(x, fresh["timesteps"], context=stage["context"], y=stage["y"], guidance=stage["guidance"])
            result_host.copy_(euler(x, v, stage["sig"]), non_blocking=True)

    h2d = sum(v.numel() * v.element_size() for v in host.values())
    d2h = result_host.numel() * result_host.element_size()
    sampler = ClockSampler()
    sampler.start()

    def sync_all():
        for i in range(args.gpus):
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

    ms = timed_local(step_device, args.steps, max(args.warmup, 4))
    ms_e2e = timed_local(step_e2e, args.steps, max(3, args.warmup // 2))
    clocks = sampler.stop(args.gpus)
    finite = bool(torch.isfinite(result_host.float()).all().item())
    extra = {"api": "nodes", "setup": {"setup_s": setup_s}, "engine": eng.describe() if hasattr(eng, "describe") else {}}
    if args.gpus > 1:
        # multi-GPU result vs the lead replica alone on the same inputs
        with torch.no_grad():
            got = model(d["x"], d["timesteps"], context=d["context"], y=d["y"], guidance=d["guidance"]).clone()
            lead_rep = eng.slots[0].replica
            want = lead_rep(d["x"], d["timesteps"], context=d["context"], y=d["y"], guidance=d["guidance"]).clone()
        sync_all()
        extra["output_matches_n1"] = rel_err(got, want)
    launches = sum(getattr(s.replica, "launches_per_step", 0) for s in eng.slots) * args.steps
    dump_outputs(args.dump_outputs, {"x_next": result_host})
    pa.cleanup_parallel_model(model)
    host_only_release(world)
    notes = {"parallelism": "ONE process, ComfyUI node API: native sm_100a replicas, in-kernel NVLink scatter/gather, "
                            "one CUDA graph per GPU replayed by native host threads",
             "step": "hooked model.forward on a new latent tensor each step + torch Euler update on the lead GPU"}
    emit(make_line(args, "ours", ms, ms_e2e, clocks, h2d, d2h, launches, finite, DTYPE_NAMES[args.dtype], notes, extra))
    return 0


# ----------------------------------------------------------------------------- reference arm
def run_reference(args) -> int:
    rank, world, local = dist_env()
    try:
        from baseline import ref_loader
        ref = ref_loader.load()
    except Exception as e:  # ReferenceUnavailable or import trouble
        if rank == 0:
            emit({"impl": "reference", "unavailable": str(e)[:300]})
        return 0
    # The reference is ONE process that drives all N GPUs from its own threads (ADP:1361-1433).  The other torchrun
    # ranks therefore stay off the GPUs entirely: no CUDA context, no NCCL communicator, no barrier kernel spinning
    # on a device the reference's replicas run on.  They sleep in a host-only (gloo) barrier until rank 0 is done.
    if host_only_group(rank, world):
        return 0
    import torch
    from comfyui_parallelanything_b200.models import flux
    B = args.batch
    params, host = synthetic_inputs(B, pinned=True)
    torch.manual_seed(1234)
    lead = torch.device("cuda", 0)
    torch.cuda.set_device(lead)
    # The reference rebuilds replicas with ``model_class(**config)`` (ADP:622) and copies weights INTO
    # them (ADP:656), so a replica gets the process' default dtype: run this arm with bf16 as the
    # default dtype (as a bf16 ComfyUI model would construct itself), otherwise clones would be fp32.
    torch.set_default_dtype(torch.bfloat16)
    with torch.device(lead):
        model = flux.Flux(params, dtype=torch.bfloat16).eval()
    # The reference rebuilds every replica on the host with ``model_class(**config)`` and then overwrites all
    # of its weights (ADP:622, 640-656); random-initialising 11.9 B parameters on the CPU per replica only
    # burns minutes of setup, so the (about to be overwritten) initialisation is skipped.  Timed steps are
    # unaffected.
    torch.nn.Linear.reset_parameters = lambda self: None
    chain = None
    pct = 100.0 / args.gpus
    t_setup = time.perf_counter()
    for i in range(args.gpus):
        chain = ref.ParallelDevice().add_device(f"cuda:{i}", pct, chain)[0]
    (model,) = ref.ParallelAnything().setup_parallel(model, chain, True, False, True, False)
    # The reference clones through ``source_model.cpu()`` in place (ADP:600-605) and leaves the original
    # (= the replica it re-uses for the lead device) stranded on the host; in ComfyUI the model manager
    # puts the MODEL back on ``load_device`` before sampling and the reference repairs it itself on the
    # next setup (ADP:932-961).  The harness plays that role: only tensors that are on the CPU are moved
    # (a blanket ``model.to(lead)`` would also drag the other replicas' blocks along, because the
    # reference registers them as submodules of the lead model through ``ParallelBlock``).
    with torch.no_grad():
        for t_ in list(model.parameters()) + list(model.buffers()):
            if t_.device.type == "cpu":
                t_.data = t_.data.to(lead)
    for i in range(args.gpus):
        torch.cuda.synchronize(i)
    setup_s = round(time.perf_counter() - t_setup, 2)
    d = {k: v.to(lead) for k, v in host.items()}
    stage = {k: torch.empty_like(v, device=lead) for k, v in host.items()}
    result_host = torch.empty(B, 16, 128, 128, dtype=torch.bfloat16).pin_memory()

    def euler(x, v, sig):
        return x + (sig[:, 1] - sig[:, 0]).view(-1, 1, 1, 1).to(x.dtype) * v

    def step_device():
        with torch.no_grad():
            v = model(d["x"], d["timesteps"], context=d["context"], y=d["y"], guidance=d["guidance"])
            return euler(d["x"], v, d["sig"])

    def step_e2e():
        for k in stage:
            stage[k].copy_(host[k], non_blocking=True)
        with torch.no_grad():
            v = model(stage["x"], stage["timesteps"], context=stage["context"], y=stage["y"],
                      guidance=stage["guidance"])
            result_host.copy_(euler(stage["x"], v, stage["sig"]), non_blocking=True)
    h2d = sum(v.numel() * v.element_size() for v in host.values())
    d2h = result_host.numel() * result_host.element_size()

    sampler = ClockSampler()
    sampler.start()
    # world=1 for the timing helpers: the whole reference lives in this process; its forward returns only after
    # every replica's output has been copied to the lead GPU with blocking ``.to`` calls (ADP:1408), so CUDA
    # events on the lead stream bracket all N GPUs' work.
    ms = timed(step_device, args.steps, args.warmup, 1)
    ms_e2e = timed(step_e2e, args.steps, max(3, args.warmup // 2), 1)
    clocks = sampler.stop(args.gpus)
    finite = bool(torch.isfinite(result_host.float()).all().item())
    dump_outputs(args.dump_outputs, {"x_next": result_host})
    host_only_release(world)
    notes = {"parallelism": f"reference threads x{args.gpus} (single process, stock torch kernels); idle torchrun ranks "
                            "hold no CUDA context",
             "step": "model forward (reference hook) + torch Euler update on the lead GPU"}
    emit(make_line(args, "reference", ms, ms_e2e, clocks, h2d, d2h, 0, finite, "bf16", notes,
                   {"setup": {"setup_s": setup_s}}))
    return 0


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--api", default="spmd", choices=["spmd", "nodes"],
                    help="spmd: one process per GPU (torchrun); nodes: ONE process drives all GPUs through the node API")
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--backend", default=os.environ.get("PA_BACKEND", "fused"), choices=["fused", "nccl"])
    ap.add_argument("--replicate", default="seed", choices=["seed", "nvls", "nccl"],
                    help="N>1: how ranks != 0 get their weights: same RNG seed (default), NVSwitch multicast kernel, "
                         "or NCCL broadcast of the packed executor weights from rank 0")
    ap.add_argument("--no-graphs", action="store_true", help="launch every kernel eagerly instead of replaying a CUDA graph")
    ap.add_argument("--dtype", default=os.environ.get("PA_BENCH_DTYPE", "fp8"), choices=["bf16", "fp8"],
                    help="fp8 (default; BASELINE config 3 names fp8) = MXFP8 block-scaled GEMMs for the block linears; "
                         "the bf16 number of the same workload is measured in the same run and reported under 'bf16'")
    ap.add_argument("--no-bf16", action="store_true", help="with --dtype fp8: skip the additional bf16 measurement")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the result of the last timed step (the next latent) as DIR/x_next.npy in float32; "
                         "when --dtype fp8 also measures bf16, that run's result as DIR/bf16_x_next.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    quiet_stdout()
    if args.impl == "reference":
        return run_reference(args)
    if args.api == "nodes":
        return run_nodes(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
