#!/usr/bin/env python
"""Multi-GPU correctness of the SPMD engine (run under torchrun, N >= 2):
fused (in-kernel NVLink scatter/gather, TMA over peer memory) vs the single-GPU executor result vs
the NCCL baseline, on a small FLUX config.  Rank 0 prints one JSON line."""
from __future__ import annotations

import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main() -> int:
    import torch
    import torch.distributed as dist
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    family = sys.argv[1] if len(sys.argv) > 1 else "flux"
    if family == "bcast":
        return bcast_check(rank, world, dev)
    if family != "flux":
        return other_family(family, rank, world, dev)
    from comfyui_parallelanything_b200.exec.flux_exec import FluxExecutor
    from comfyui_parallelanything_b200.models import flux
    from comfyui_parallelanything_b200.parallel.spmd import SpmdFluxEngine
    p = flux.FluxParams(in_channels=64, out_channels=64, vec_in_dim=768, context_in_dim=512, hidden_size=512,
                        mlp_ratio=4.0, num_heads=4, depth=2, depth_single_blocks=2)
    torch.manual_seed(5)
    model = flux.Flux(p).to(device=dev, dtype=torch.bfloat16).eval()
    ex = FluxExecutor(model, dev, cuda_graphs=True)
    B, H, W, Lt = 5 if world == 2 else 2 * world + 1, 256, 384, 77
    inp = flux.example_inputs(p, B, H, W, txt_len=Lt, device=dev, dtype=torch.bfloat16, seed=11)
    sig = torch.tensor([[1.0 - 0.1 * i, 0.8 - 0.1 * i] for i in range(B)], device=dev)
    res = {}
    x, t, c, y, g = ex._prep(inp["x"], inp["timesteps"], inp["context"], inp["y"], inp["guidance"])
    want = ex.denoise_step(x, t, c, y, g, sig).clone()          # whole batch on every rank (reference result)
    for backend, tma_peer in (("fused", "1"), ("fused", "0"), ("nccl", "0")):
        os.environ["PA_TMA_PEER"] = tma_peer
        weights = [60, 40][:world] if world == 2 else None
        eng = SpmdFluxEngine(ex, B, H, W, Lt, weights=weights, backend=backend)
        for it in range(4):                                     # several epochs: flag reuse; eager, capture, replay x2
            if rank == 0:
                eng.stage_inputs(inp["x"], inp["timesteps"], inp["context"], inp["y"], inp["guidance"], sig)
            out = eng.step()
        torch.cuda.synchronize()
        eng.check_error()
        if rank == 0:
            d = (out.float() - want.float()).abs()
            res[f"{backend}_tma{tma_peer}"] = dict(max_abs=d.max().item(), mean_rel=d.mean().item() / want.float().abs().mean().item(),
                                                  sizes=eng.sizes)
        eng.close()
    if rank == 0:
        ok = all(v["mean_rel"] < 5e-3 for v in res.values())
        print("PA_SPMD " + json.dumps(dict(world=world, ok=ok, results=res)), flush=True)
    dist.destroy_process_group()
    return 0


def bcast_check(rank, world, dev) -> int:
    """Weight replication for the one-process-per-GPU layout: every rank packs an executor from DIFFERENT random
    weights, rank 0 broadcasts its packed table (NVSwitch multicast kernel, NCCL fallback), and afterwards every rank
    must hold rank 0's bytes (fp64 checksums + first/last bytes of every tensor compared across ranks)."""
    import torch
    import torch.distributed as dist
    from comfyui_parallelanything_b200.exec.flux_exec import FluxExecutor
    from comfyui_parallelanything_b200.exec.pack_cache import packed_table
    from comfyui_parallelanything_b200.models import flux
    from comfyui_parallelanything_b200.parallel import replicate_nvl
    p = flux.FluxParams(in_channels=64, out_channels=64, vec_in_dim=768, context_in_dim=512, hidden_size=1024,
                        mlp_ratio=4.0, num_heads=8, depth=2, depth_single_blocks=3)
    res = {}
    for method, fp8 in (("nvls", False), ("nvls", True), ("nccl", False)):
        torch.manual_seed(100 + rank)
        ex = FluxExecutor(flux.Flux(p).to(device=dev, dtype=torch.bfloat16).eval(), dev, fp8=fp8)
        rep = replicate_nvl.broadcast_executor(ex, src=0, method=method, slot_bytes=8 << 20)   # small slots: many hand-offs
        sums = []
        for k, v in sorted(packed_table(ex).items()):
            if isinstance(v, torch.Tensor) and v.is_cuda:
                b = v.reshape(-1).view(torch.uint8)
                sums.append(b.double().sum() + 3.0 * b[:64].double().sum() + 7.0 * b[-64:].double().sum())
        mine = torch.stack(sums)
        allv = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(allv, mine)
        same = all(bool(torch.equal(a, allv[0])) for a in allv)
        res[f"{method}{'_fp8' if fp8 else ''}"] = dict(identical=same, tensors=len(sums), **rep)
        del ex
    if rank == 0:
        ok = all(v["identical"] for v in res.values())
        print("PA_SPMD " + json.dumps(dict(family="bcast", world=world, ok=ok, results=res)), flush=True)
    dist.destroy_process_group()
    return 0


def other_family(family, rank, world, dev) -> int:
    """Same comparison for the SDXL-class UNet (``unet``), Z-Image (``zimage``) and the WAN video DiT engines: ``wan``
    (text-to-video, 16 latent channels), ``wan_i2v`` (image-to-video: 36 input channels, 16 output channels),
    ``wan_clip`` (WAN2.1 image-to-video: ``wan_i2v`` plus CLIP image features staged as the ``"clip"`` input) and
    ``wan_ti2v`` (WAN2.2 TI2V: 48 channels in and out, one timestep per latent frame staged as ``"t"`` [B, T])."""
    import torch
    import torch.distributed as dist
    from comfyui_parallelanything_b200.parallel import spmd
    B = 5 if world == 2 else 2 * world + 1
    sig = torch.tensor([[1.0 - 0.1 * i, 0.8 - 0.1 * i] for i in range(B)], device=dev)
    if family == "unet":
        from comfyui_parallelanything_b200.exec.unet_exec import UNetExecutor
        from comfyui_parallelanything_b200.models import unet
        cfg = unet.mini_sdxl_config()
        torch.manual_seed(3)
        ex = UNetExecutor(unet.UNetModel(**cfg).to(device=dev, dtype=torch.bfloat16).eval(), dev, cuda_graphs=True)
        inp = unet.example_inputs(cfg, B, 256, 384, ctx_len=77, device=dev, dtype=torch.bfloat16)
        order = [inp["x"], inp["timesteps"], inp["context"], inp["y"], sig]
        want = ex.denoise_step(*order).clone()
        make = lambda backend, w: spmd.SpmdUNetEngine(ex, B, 256, 384, 77, weights=w, backend=backend)  # noqa: E731
    elif family == "zimage":
        from comfyui_parallelanything_b200.exec.zimage_exec import ZImageExecutor
        from comfyui_parallelanything_b200.models import zimage
        p = zimage.zimage_tiny_params()
        torch.manual_seed(4)
        ex = ZImageExecutor(zimage.ZImageModel(p).to(device=dev, dtype=torch.bfloat16).eval(), dev, cuda_graphs=True)
        inp = zimage.example_inputs(p, B, 256, 384, cap_len=40, device=dev, dtype=torch.bfloat16)
        x, t, c = ex._prep(inp["x"], inp["timesteps"], inp["context"])
        order = [x, t, c, sig]
        want = ex.denoise_step(*order).clone()
        make = lambda backend, w: spmd.SpmdZImageEngine(ex, B, 256, 384, 40, weights=w, backend=backend)  # noqa: E731
    else:
        import dataclasses
        from comfyui_parallelanything_b200.exec.wan_exec import WanClipExecutor, WanExecutor
        from comfyui_parallelanything_b200.models import wan
        p = wan.wan_tiny_params()
        make_inputs = wan.example_inputs
        if family == "wan_i2v":
            p, make_inputs = dataclasses.replace(p, in_dim=36), wan.i2v_inputs
        elif family == "wan_clip":
            p, make_inputs = dataclasses.replace(p, in_dim=36, clip_dim=128), wan.clip_inputs
        elif family == "wan_ti2v":
            p, make_inputs = dataclasses.replace(p, in_dim=48, out_dim=48), wan.ti2v_inputs
        torch.manual_seed(2)
        cls = WanClipExecutor if family == "wan_clip" else WanExecutor
        ex = cls(wan.WanModel(p).to(device=dev, dtype=torch.bfloat16).eval(), dev, cuda_graphs=True)
        frames, height, width = (9, 256, 384) if family == "wan_ti2v" else (8, 128, 192)   # TI2V: 16x VAE
        inp = make_inputs(p, B, frames=frames, height=height, width=width, device=dev, dtype=torch.bfloat16)
        if family == "wan_ti2v":
            inp["timesteps"][:, 1:] = torch.linspace(300.0, 900.0, B, device=dev)[:, None].to(torch.bfloat16)
        if family == "wan_clip":
            x, t, c, cf = ex._prep(inp["x"], inp["timesteps"], inp["context"], inp["clip_fea"])
            want = ex.denoise_step(x, t, c, cf, sig).clone()
            order = [x, t, c, sig, cf]                  # the engine's input order: "clip" follows "sig"
        else:
            x, t, c = ex._prep(inp["x"], inp["timesteps"], inp["context"])
            order = [x, t, c, sig]
            want = ex.denoise_step(*order).clone()
        li = cf.shape[1] if family == "wan_clip" else 0
        make = lambda backend, w: spmd.SpmdWanEngine(  # noqa: E731
            ex, B, x.shape[2], height, width, c.shape[1], weights=w, backend=backend, clip_tokens=li,
            frame_timesteps=family == "wan_ti2v")
    res = {}
    for backend, tma_peer in (("fused", "1"), ("fused", "0"), ("nccl", "0")):
        os.environ["PA_TMA_PEER"] = tma_peer
        eng = make(backend, [60, 40][:world] if world == 2 else None)
        for it in range(4):
            if rank == 0:
                eng.stage_inputs(*order)
            out = eng.step()
        torch.cuda.synchronize()
        eng.check_error()
        if rank == 0:
            d = (out.float() - want.float()).abs()
            res[f"{backend}_tma{tma_peer}"] = dict(max_abs=d.max().item(),
                                                  mean_rel=d.mean().item() / want.float().abs().mean().item(), sizes=eng.sizes)
        eng.close()
    if rank == 0:
        ok = all(v["mean_rel"] < 5e-3 for v in res.values())
        print("PA_SPMD " + json.dumps(dict(family=family, world=world, ok=ok, results=res)), flush=True)
    dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
