#!/usr/bin/env python
"""Secondary benchmark: WAN2.2-A14B-sized video DiT (14.3 B params, random init), 720p x 16 frames (latent
[16, 4, 90, 160] -> 14 400 tokens per sample), batch 8, bf16 - BASELINE.json config 4.  Same protocol and JSON line as
bench.py (one step = forward + Euler update; device-timed, max over ranks; e2e with per-step H2D/D2H).  ``--i2v`` runs
WAN2.2-I2V-A14B instead: the same layer stack on a 36-channel input ([noise 16 | mask 4 | image latent 16]).  ``--clip``
runs WAN2.1-I2V-14B (that input plus 257 CLIP image tokens and an image cross-attention in every block), ``--flf2v``
WAN2.1-FLF2V-14B (514 CLIP tokens of the first and last frame).  ``--ti2v`` runs WAN2.2-TI2V-5B at its own size:
1280 x 704 x 121 frames, a 48-channel [31, 44, 80] latent of the WAN2.2 VAE (27 280 tokens per sample), with one
timestep per latent frame (image-to-video mode; ``--sample-timesteps``: one per sample, text-to-video mode).

    python tools/bench_wan.py --gpus 1 [--impl reference] [--batch 8] [--i2v | --clip | --flf2v | --ti2v]
    python -m torch.distributed.run --nproc-per-node 8 ... tools/bench_wan.py --gpus 8
"""
from __future__ import annotations

import argparse
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench as hb  # noqa: E402  (helpers: ClockSampler, timed, emit, dist_env, ...)

MODEL_NAME = "WAN2.2-A14B video DiT 720p x 16 frames"
I2V_MODEL_NAME = "WAN2.2-I2V-A14B video DiT 720p x 16 frames"
CLIP_MODEL_NAME = "WAN2.1-I2V-14B video DiT 720p x 16 frames (257 CLIP tokens)"
FLF2V_MODEL_NAME = "WAN2.1-FLF2V-14B video DiT 720p x 16 frames (514 CLIP tokens)"
TI2V_MODEL_NAME = "WAN2.2-TI2V-5B video DiT 1280x704 x 121 frames"


def model_name(a) -> str:
    if a.ti2v:
        return TI2V_MODEL_NAME + (" (one timestep per sample)" if a.sample_timesteps else " (per-frame timesteps)")
    return FLF2V_MODEL_NAME if a.flf2v else CLIP_MODEL_NAME if a.clip else I2V_MODEL_NAME if a.i2v else MODEL_NAME


def geometry(a) -> tuple:
    """(pixel frames, height, width) of the workload."""
    return (121, 704, 1280) if a.ti2v else (16, 720, 1280)


def host_inputs(B, cap_len, a):
    import torch
    from comfyui_parallelanything_b200.models import wan
    if a.flf2v or a.clip:
        cfg, make = (wan.wan21_flf2v_14b_params() if a.flf2v else wan.wan21_i2v_14b_params()), wan.clip_inputs
    elif a.i2v:
        cfg, make = wan.wan22_i2v_a14b_params(), wan.i2v_inputs
    elif a.ti2v:
        cfg, make = wan.wan22_ti2v_5b_params(), wan.ti2v_inputs
    else:
        cfg, make = wan.wan22_a14b_params(), wan.example_inputs
    frames, height, width = geometry(a)
    inp = make(cfg, B, frames=frames, height=height, width=width, device="cpu", dtype=torch.bfloat16)
    if a.ti2v and a.sample_timesteps:
        inp["timesteps"] = inp["timesteps"][:, 1].contiguous()
    inp["sig"] = torch.tensor([[1.0, 0.875]] * B, dtype=torch.float32)
    return cfg, {k: v.pin_memory() for k, v in inp.items()}


def run_nodes(a) -> int:
    """One process through the node API (tools/_nodes_bench.py); batch 1 = the video workload: sequence-parallel."""
    import torch
    import _nodes_bench
    from comfyui_parallelanything_b200.models import wan
    cfg, host = host_inputs(a.batch, a.cap_len, a)
    name = model_name(a)

    def build(lead):
        with torch.device(lead):
            return wan.WanModel(cfg, dtype=torch.bfloat16).eval()

    return _nodes_bench.run(a, hb, name, build, host,
                            {"model": name, "global_batch": a.batch, "text_len": a.cap_len, "baseline_config": 4})


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "fp8"], help="fp8 = MXFP8 block GEMMs in the native executor")
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--cap-len", type=int, default=512)
    ap.add_argument("--api", default="spmd", choices=["spmd", "nodes"],
                    help="nodes = ONE process through the ComfyUI node API, new latent tensor every step (batch 1 -> "
                         "sequence-parallel over all GPUs)")
    ap.add_argument("--i2v", action="store_true", help="WAN2.2-I2V-A14B (36-channel input) instead of T2V")
    ap.add_argument("--clip", action="store_true", help="WAN2.1-I2V-14B (36-channel input + CLIP image cross-attention)")
    ap.add_argument("--flf2v", action="store_true", help="WAN2.1-FLF2V-14B (as --clip, 514 CLIP tokens)")
    ap.add_argument("--ti2v", action="store_true",
                    help="WAN2.2-TI2V-5B (48 channels in and out) at 1280x704 x 121 frames, per-frame timesteps")
    ap.add_argument("--sample-timesteps", action="store_true",
                    help="with --ti2v: one timestep per sample (text-to-video mode) instead of one per latent frame")
    a = ap.parse_args()
    if a.api == "nodes":
        return run_nodes(a)
    hb.quiet_stdout()
    import torch
    rank, world, local = hb.dist_env()
    B = a.batch
    pcts = [100.0 / a.gpus] * a.gpus
    tworld = world
    if a.impl == "reference":
        # the reference is one process driving all GPUs: the other torchrun ranks stay off the GPUs (host-only gloo
        # barrier, no CUDA context / NCCL kernels on the devices its replicas run on) - see bench.py
        if hb.host_only_group(rank, world):
            return 0
        tworld = 1
    torch.cuda.set_device(local if a.impl == "ours" else 0)
    dev = torch.device("cuda", local)
    if world > 1 and a.impl == "ours":
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    from comfyui_parallelanything_b200.models import wan
    cfg, host = host_inputs(B, a.cap_len, a)
    clip = "clip_fea" in host
    out_shape = (B, cfg.out_dim) + tuple(host["x"].shape[2:])
    result_host = torch.empty(out_shape, dtype=torch.bfloat16).pin_memory()
    h2d = sum(v.numel() * v.element_size() for v in host.values())
    d2h = result_host.numel() * result_host.element_size()
    launches = 0
    eng = None
    if a.impl == "ours":
        from comfyui_parallelanything_b200.exec.wan_exec import WanClipExecutor, WanExecutor
        torch.manual_seed(1234)
        with torch.device(dev):
            model = wan.WanModel(cfg, dtype=torch.bfloat16).eval()
        ex = (WanClipExecutor if clip else WanExecutor)(model, dev, cuda_graphs=True, fp8=(a.dtype == "fp8"))
        del model
        torch.cuda.empty_cache()
        if world == 1:
            d = {k: v.to(dev) for k, v in host.items()}
            stage = {k: torch.empty_like(v, device=dev) for k, v in host.items()}
            out_buf = torch.empty(out_shape, dtype=torch.bfloat16, device=dev)

            cond = ("context", "clip_fea") if clip else ("context",)

            def step_device():
                ex.denoise_step(d["x"], d["timesteps"], *(d[k] for k in cond), d["sig"], out=out_buf)

            def step_e2e():
                for k in stage:
                    stage[k].copy_(host[k], non_blocking=True)
                ex.invalidate_conditioning()        # the staged conditioning is re-sent every step: recompute it
                ex.denoise_step(stage["x"], stage["timesteps"], *(stage[k] for k in cond), stage["sig"], out=out_buf)
                result_host.copy_(out_buf, non_blocking=True)
        else:
            from comfyui_parallelanything_b200.parallel.spmd import SpmdWanEngine
            _, height, width = geometry(a)
            eng = SpmdWanEngine(ex, B, host["x"].shape[2], height, width, a.cap_len, weights=pcts,
                                clip_tokens=host["clip_fea"].shape[1] if clip else 0,
                                frame_timesteps=host["timesteps"].dim() == 2)
            order = [host[k] for k in ("x", "timesteps", "context", "sig") + (("clip_fea",) if clip else ())]
            if rank == 0:
                eng.stage_inputs(*order)
            torch.cuda.synchronize()

            def step_device():
                eng.step()

            def step_e2e():
                if rank == 0:
                    eng.stage_inputs(*order)
                eng.new_conditioning()
                out = eng.step()
                if rank == 0:
                    result_host.copy_(out, non_blocking=True)
        par = f"dp{world} split {eng.sizes if eng else [B]} (fused in-kernel NVLink scatter/gather)"
    else:
        from baseline import ref_loader
        try:
            ref = ref_loader.load()
        except Exception as e:
            if rank == 0:
                hb.emit({"impl": "reference", "unavailable": str(e)[:300]})
            return 0
        if rank == 0:
            lead = torch.device("cuda", 0)
            torch.set_default_dtype(torch.bfloat16)
            torch.manual_seed(1234)
            with torch.device(lead):
                model = wan.WanModel(cfg, dtype=torch.bfloat16).eval()
            torch.nn.Linear.reset_parameters = lambda self: None      # clones are overwritten anyway (see bench.py)
            chain = None
            for i in range(a.gpus):
                chain = ref.ParallelDevice().add_device(f"cuda:{i}", float(pcts[i]), chain)[0]
            (model,) = ref.ParallelAnything().setup_parallel(model, chain, True, False, True, False)
            with torch.no_grad():
                for t_ in list(model.parameters()) + list(model.buffers()):
                    if t_.device.type == "cpu":
                        t_.data = t_.data.to(lead)
            d = {k: v.to(lead) for k, v in host.items()}
            stage = {k: torch.empty_like(v, device=lead) for k, v in host.items()}

            def euler(x, e, sig):       # I2V: the update covers the predicted noise channels of x
                return x[:, :e.shape[1]] + (sig[:, 1] - sig[:, 0]).view(-1, 1, 1, 1, 1).to(x.dtype) * e

            kw = {"clip_fea": d["clip_fea"]} if clip else {}
            kw_e2e = {"clip_fea": stage["clip_fea"]} if clip else {}

            def step_device():
                with torch.no_grad():
                    e = model(d["x"], d["timesteps"], context=d["context"], **kw)
                    return euler(d["x"], e, d["sig"])

            def step_e2e():
                for k in stage:
                    stage[k].copy_(host[k], non_blocking=True)
                with torch.no_grad():
                    e = model(stage["x"], stage["timesteps"], context=stage["context"], **kw_e2e)
                    result_host.copy_(euler(stage["x"], e, stage["sig"]), non_blocking=True)
        else:
            def step_device():
                return None
            step_e2e = step_device
        par = f"reference threads x{a.gpus} pct {pcts}"
    sampler = hb.ClockSampler()
    if rank == 0:
        sampler.start()
    ms = hb.timed(step_device, a.steps, a.warmup, tworld)
    ms_e2e = hb.timed(step_e2e, a.steps, max(3, a.warmup // 2), tworld)
    clocks = sampler.stop(a.gpus) if rank == 0 else {}
    if eng is not None:
        eng.check_error()
        eng.close()
    if a.impl == "reference":
        hb.host_only_release(world)
    elif world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()
    if rank == 0:
        hb.emit({"metric": hb.METRIC, "value": round(1000.0 / ms, 4), "unit": "steps/s", "n_gpus": a.gpus, "steps": a.steps,
                 "warmup": a.warmup, "ms_per_step": round(ms, 3), "higher_is_better": True, "scaling": "strong",
                 "vs_baseline": None, "sec_per_it": round(ms / 1000.0, 4), "dtype": (a.dtype if a.impl == "ours" else "bf16"), "data": "synthetic, random-init weights", "impl": a.impl,
                 "clocks": clocks,
                 "e2e": {"value": round(1000.0 / ms_e2e, 4), "unit": "steps/s", "ms_per_step": round(ms_e2e, 3),
                         "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
                 "output_finite": bool(torch.isfinite(result_host.float()).all().item()),
                 "config": {"model": model_name(a), "global_batch": B, "text_len": a.cap_len, "baseline_config": 4, "parallelism": par}})
    return 0


if __name__ == "__main__":
    sys.exit(main())
