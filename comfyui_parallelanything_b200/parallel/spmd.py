"""One-process-per-GPU engine (``torchrun``): replicas on every rank, batch owned by rank 0.

The reference moves shards with ``torch.split`` + N blocking ``.to(dev)`` copies from N Python
threads and gathers with N blocking ``.to(lead)`` + ``torch.cat``
(/root/reference/any_device_parallel.py:1348-1356, 1372-1378, 1408, 1433).  Here:

  * every rank allocates one *symmetric* buffer (raw ``cudaMalloc``, exported with CUDA IPC and
    mapped by all peers — ``SymmetricHeap``); ``torch.distributed`` (NCCL) is used only for
    bootstrap (handle exchange, barriers) and as the ``backend="nccl"`` baseline;
  * **scatter**: rank r's first kernel reads its shard of ``x`` / ``t`` / conditioning straight
    out of rank 0's buffer over NVLink (peer loads inside the patchify / embed kernels) after
    acquiring a flag word that rank 0 releases once the step's inputs are in place;
  * **gather**: the last GEMM's epilogue (unpatchify + Euler update) stores rank r's rows of
    ``x_{t-1}`` directly at their final offset in rank 0's output buffer and releases a
    per-rank flag; rank 0 acquires all flags — no copy kernels, no cat, no host sync;
  * flag waits are bounded (watchdog) so a dead peer cannot hang the GPU.
"""
from __future__ import annotations

import os
from typing import Dict, List, Optional, Sequence

import torch
import torch.distributed as dist

from .. import chain as chain_mod
from .. import ops
from ..utils import log

_ALIGN = 1024


class SymmetricHeap:
    """Same-size raw device buffer on every rank, peer-mapped everywhere (CUDA IPC)."""

    def __init__(self, nbytes: int, group=None):
        C = ops.require()
        self.C = C
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        self.dev = torch.cuda.current_device()
        self.nbytes = (nbytes + _ALIGN - 1) // _ALIGN * _ALIGN
        self.local_ptr = C.dev_malloc(self.dev, self.nbytes, True)
        handle = C.ipc_get_handle(self.local_ptr)
        handles: List[Optional[bytes]] = [None] * self.world
        dist.all_gather_object(handles, (self.dev, handle), group=group)
        self.ptrs: List[int] = []
        self._opened: List[int] = []
        for r, (pdev, h) in enumerate(handles):
            if r == self.rank:
                self.ptrs.append(self.local_ptr)
            else:
                p = C.ipc_open_handle(self.dev, h)
                self._opened.append(p)
                self.ptrs.append(p)
        self.local = C.tensor_from_ptr(self.local_ptr, self.nbytes, self.dev)
        self._cursor = 0
        dist.barrier(group=group)

    def carve(self, nbytes: int) -> int:
        off = self._cursor
        self._cursor = (off + nbytes + 255) // 256 * 256
        if self._cursor > self.nbytes:
            raise MemoryError("symmetric heap exhausted")
        return off

    def view(self, off: int, shape: Sequence[int], dtype: torch.dtype) -> torch.Tensor:
        n = 1
        for s in shape:
            n *= s
        nb = n * torch.empty((), dtype=dtype).element_size()
        return self.local[off:off + nb].view(dtype).view(*shape)

    def peer_ptr(self, rank: int, off: int) -> int:
        return self.ptrs[rank] + off

    def close(self) -> None:
        for p in self._opened:
            try:
                self.C.ipc_close_handle(p)
            except Exception:
                pass
        self._opened = []
        if self.local_ptr:
            self.local = None
            self.C.dev_free(self.local_ptr)
            self.local_ptr = 0


class SpmdFluxEngine:
    """SPMD denoise-step engine for the FLUX family.  Every rank calls ``step`` each iteration;
    only rank 0 passes real inputs (pinned host or device tensors), the others pass ``None``."""

    FLAG_INPUTS = 0          # slot written by rank 0 on every peer: "inputs of epoch e are ready"
    FLAG_DONE0 = 8           # slots 8.. on rank 0: "rank r finished epoch e"

    def __init__(self, executor, global_batch: int, height: int, width: int, txt_len: int,
                 weights: Optional[Sequence[float]] = None, split_mode: str = "compat", backend: str = "fused",
                 timeout_ms: int = 20000):
        self.ex = executor
        self.rank, self.world = dist.get_rank(), dist.get_world_size()
        self.dev = torch.device("cuda", torch.cuda.current_device())
        self.backend = backend
        f = self._pixels_per_latent()
        self.B, self.H, self.W, self.Lt = global_batch, height // f, width // f, txt_len
        self.C = self._latent_channels()
        w = list(weights) if weights is not None else [1.0 / self.world] * self.world
        self.sizes = chain_mod.split_sizes(global_batch, chain_mod.normalize_weights(w), split_mode)
        self.offs = chain_mod.offsets(self.sizes)
        self.n_local, self.off_local = self.sizes[self.rank], self.offs[self.rank]
        B = global_batch
        bf = torch.bfloat16
        self.spec = self._make_spec(B)      # name -> (shape, dtype) of rank 0's staging area
        total = 4096
        for shape, dt in self.spec.values():
            n = 1
            for s in shape:
                n *= s
            total += (n * torch.empty((), dtype=dt).element_size() + 255) // 256 * 256
        self.heap = SymmetricHeap(total)
        self.off: Dict[str, int] = {"flags": self.heap.carve(256)}
        for name, (shape, dt) in self.spec.items():
            n = 1
            for s in shape:
                n *= s
            self.off[name] = self.heap.carve(n * torch.empty((), dtype=dt).element_size())
        self.flags = self.heap.view(self.off["flags"], (64,), torch.int32)
        self.buf = {k: self.heap.view(self.off[k], *self.spec[k]) for k in self.spec}
        self.err = torch.zeros(1, dtype=torch.int32, device=self.dev)
        self.peer_flag_table = torch.tensor([self.heap.peer_ptr(r, self.off["flags"]) for r in range(self.world)],
                                            dtype=torch.int64, device=self.dev)
        self.lead_flag_table = torch.tensor([self.heap.peer_ptr(0, self.off["flags"])], dtype=torch.int64,
                                            device=self.dev)
        self.timeout_cycles = int(timeout_ms * 1.9e6)
        self.epoch = 0
        # local shard buffers (inputs are pulled from rank 0 into these)
        n = max(self.n_local, 1)
        self.loc = {k: torch.empty((n,) + tuple(shape[1:]), dtype=dt, device=self.dev)
                    for k, (shape, dt) in self.spec.items() if k != "out"}
        self.input_names = tuple(k for k in self.spec if k != "out")
        self.comm_launches = 0
        self.tma_peer = os.environ.get("PA_TMA_PEER", "1") != "0"
        log.info("SPMD rank %d/%d: samples [%d, %d) of %d, backend=%s", self.rank, self.world, self.off_local,
                 self.off_local + self.n_local, B, backend)

    # -------------------------------------------------------------- family hooks (FLUX defaults)
    def _pixels_per_latent(self) -> int:
        """Spatial compression of the family's VAE (pixel size / latent size)."""
        return 8

    def _latent_channels(self) -> int:
        return self.ex.params.in_channels // 4

    def _make_spec(self, B: int) -> dict:
        p, bf = self.ex.params, torch.bfloat16
        return {"x": ((B, self.C, self.H, self.W), bf), "t": ((B,), bf), "ctx": ((B, self.Lt, p.context_in_dim), bf),
                "y": ((B, p.vec_in_dim), bf), "g": ((B,), bf), "sig": ((B, 2), torch.float32),
                "out": ((B, self.C, self.H, self.W), bf)}

    def _launch(self, loc: dict, fused: bool) -> None:
        """Run the replica on this rank's shard.  ``fused``: pull x/t/g inside the first kernel from rank 0 and
        store the result rows into rank 0's output buffer from the last kernel's epilogue."""
        if fused:
            self.ex.denoise_step(loc["x"], loc["t"], loc["ctx"], loc["y"], loc["g"], loc["sig"],
                                 out_ptr=self.heap.peer_ptr(0, self.off["out"]), out_sample_off=self.off_local,
                                 x_src_ptr=self._src("x", self._row_bytes("x")), t_src_ptr=self._src("t", 2),
                                 g_src_ptr=self._src("g", 2))
            return None
        return self.ex.denoise_step(loc["x"], loc["t"], loc["ctx"], loc["y"], loc["g"], loc["sig"])

    #: inputs that the replica's GEMMs may read straight from rank 0's HBM through TMA descriptors
    tma_peer_inputs = ("ctx", "y")
    #: inputs the first kernel pulls itself (never copied separately on the fused path)
    kernel_pulled_inputs = ("x", "t", "g")

    # -------------------------------------------------------------- helpers
    def _src(self, name: str, row_bytes: int) -> int:
        return self.heap.peer_ptr(0, self.off[name]) + self.off_local * row_bytes

    def _row_bytes(self, name: str) -> int:
        """Bytes of one sample of the staged input ``name``."""
        shape, dt = self.spec[name]
        row = 1
        for s_ in shape[1:]:
            row *= s_
        return row * torch.empty((), dtype=dt).element_size()

    def _peer_view(self, name: str) -> torch.Tensor:
        """This rank's shard of rank 0's staging tensor as a (peer-mapped) torch view."""
        shape, dt = self.spec[name]
        row_bytes = self._row_bytes(name)
        t = self.heap.C.tensor_from_ptr(self._src(name, row_bytes), row_bytes * self.n_local, self.dev.index)
        return t.view(dt).view(self.n_local, *shape[1:])

    def _pull(self, name: str) -> None:
        """Shard of a small tensor: peer -> local with a device-side copy (cudaMemcpyAsync P2P)."""
        dst = self.loc[name][:self.n_local]
        row_bytes = dst[0].numel() * dst.element_size() if dst.dim() > 1 else dst.element_size()
        self.heap.C.memcpy_async(dst.data_ptr(), self._src(name, row_bytes), row_bytes * self.n_local, 4,
                                 torch.cuda.current_stream().cuda_stream)

    def stage_inputs(self, *tensors, **named) -> int:
        """rank 0: copy this step's inputs (pinned host or device tensors) into the symmetric
        staging area (positional order = ``self.input_names``).  Returns the number of bytes copied."""
        nbytes = 0
        items = list(zip(self.input_names, tensors)) + list(named.items())
        for name, src in items:
            self.buf[name].copy_(src, non_blocking=True)
            nbytes += self.buf[name].numel() * self.buf[name].element_size()
        return nbytes

    # -------------------------------------------------------------- one denoise step
    def step(self, staged: bool = True) -> torch.Tensor:
        """All ranks.  Rank 0 must have called ``stage_inputs`` (same stream) before.  Returns rank
        0's output buffer (valid on rank 0 once the stream reaches this point)."""
        C = self.heap.C
        self.epoch += 1
        e = self.epoch
        n = 0
        if self.backend == "nccl":
            return self._step_nccl()
        if self.rank == 0:
            C.signal_flags(self.peer_flag_table, self.world, self.FLAG_INPUTS, e)
            n += 1
        C.wait_flags(self.flags, self.FLAG_INPUTS, 1, e, self.timeout_cycles, self.err)
        n += 1
        if self.n_local > 0:
            if self.rank == 0:
                # fresh non-owning views (version counter 0): executors key their cached conditioning work on
                # (pointer, shape, version); a slice of ``self.buf`` would bump its version on every ``stage_inputs``
                loc = {k: self._peer_view(k) for k in self.input_names}
            else:
                loc = {k: v[:self.n_local] for k, v in self.loc.items()}
                for name in self.input_names:
                    if name in self.kernel_pulled_inputs:
                        continue
                    if self.tma_peer and name in self.tma_peer_inputs:
                        # consumed by TMA directly from the lead's HBM (A operand of a GEMM over NVLink)
                        loc[name] = self._peer_view(name)
                    else:
                        self._pull(name)
                        n += 1
            # fused scatter: the first kernel loads this rank's latent shard directly from rank 0's buffer over
            # NVLink; fused gather: the last kernel stores x_{t-1} rows at their final offset in rank 0's
            # output buffer.
            self._launch(loc, fused=True)
            n += self.ex.launches_per_step
        C.signal_flags(self.lead_flag_table, 1, self.FLAG_DONE0 + self.rank, e)
        n += 1
        if self.rank == 0:
            C.wait_flags(self.flags, self.FLAG_DONE0, self.world, e, self.timeout_cycles, self.err)
            n += 1
        self.comm_launches = n
        return self.buf["out"]

    def _step_nccl(self) -> torch.Tensor:
        """Baseline: NCCL point-to-point scatter/gather around the same executor (what "just call
        the library" costs; not the product path)."""
        loc = {}
        for k in self.input_names:
            if self.rank == 0:
                for r in range(1, self.world):
                    if self.sizes[r]:
                        dist.send(self.buf[k][self.offs[r]:self.offs[r] + self.sizes[r]], dst=r)
                loc[k] = self.buf[k][:self.sizes[0]]
            else:
                loc[k] = self.loc[k][:self.n_local]
                if self.n_local:
                    dist.recv(loc[k], src=0)
        out = None
        if self.n_local:
            out = self._launch(loc, fused=False)
        if self.rank == 0:
            if out is not None:
                self.buf["out"][:self.sizes[0]].copy_(out)
            for r in range(1, self.world):
                if self.sizes[r]:
                    dist.recv(self.buf["out"][self.offs[r]:self.offs[r] + self.sizes[r]], src=r)
        elif out is not None:
            dist.send(out, dst=0)
        self.comm_launches = self.ex.launches_per_step
        return self.buf["out"]

    def new_conditioning(self) -> None:
        """Collective by convention (every rank calls it): the conditioning staged next differs from the previous
        one although it lives in the same heap buffer, so executors must drop what they cached from it (text
        embeddings, cross-attention K/V, refined caption tokens)."""
        inv = getattr(self.ex, "invalidate_conditioning", None)
        if inv is not None:
            inv()

    def check_error(self) -> None:
        v = int(self.err.item()) & 0xFFFFFFFF
        if v:
            raise RuntimeError(f"flag wait timed out on rank {self.rank}: 0x{v:08x} (dead or stalled peer)")

    def close(self) -> None:
        torch.cuda.synchronize()
        dist.barrier()
        self.buf, self.flags = {}, None
        self.heap.close()


def broadcast_executor_weights(executor, src: int = 0, group=None, bucket_bytes: int = 256 << 20) -> int:
    """Weight replication over NVLink for the one-process-per-GPU layout (SURVEY K9): rank ``src`` holds the
    packed weights, every other rank receives them device-to-device through NCCL broadcasts (NVSwitch
    multicast / NVLS when NCCL enables it) in ``bucket_bytes`` buckets — no host bounce, unlike the
    reference's ``source.cpu()`` + per-key H2D clone (/root/reference/any_device_parallel.py:600-663).
    Returns the number of bytes received/sent."""
    tensors = [t for t in _executor_tensors(executor) if isinstance(t, torch.Tensor) and t.is_cuda]
    total, bucket, size = 0, [], 0

    def flush():
        nonlocal bucket, size, total
        if not bucket:
            return
        flat = torch.cat([t.reshape(-1).view(torch.uint8) for t in bucket]) if len(bucket) > 1 \
            else bucket[0].reshape(-1).view(torch.uint8)
        dist.broadcast(flat, src=src, group=group)
        if dist.get_rank(group) != src and len(bucket) > 1:
            off = 0
            for t in bucket:
                n = t.numel() * t.element_size()
                t.reshape(-1).view(torch.uint8).copy_(flat[off:off + n])
                off += n
        total += flat.numel()
        bucket, size = [], 0

    for t in tensors:
        n = t.numel() * t.element_size()
        if n >= bucket_bytes:                 # big tensors go alone, in place (no staging copy)
            flush()
            dist.broadcast(t, src=src, group=group)
            total += n
            continue
        bucket.append(t)
        size += n
        if size >= bucket_bytes:
            flush()
    flush()
    return total


def _executor_tensors(executor):
    w = getattr(executor, "W", None)
    if isinstance(w, dict):
        for k in sorted(w):
            yield w[k]
        return
    seen = set()

    def walk(o):
        if isinstance(o, torch.Tensor):
            if id(o) not in seen:
                seen.add(id(o))
                yield o
        elif isinstance(o, (list, tuple)):
            for v in o:
                yield from walk(v)
        elif isinstance(o, dict):
            for k in sorted(o, key=str):
                yield from walk(o[k])
        elif hasattr(o, "__dict__") and not isinstance(o, (torch.nn.Module, type)):
            yield from walk(vars(o))
    for name in sorted(vars(executor)):
        if not name.startswith("_"):
            yield from walk(getattr(executor, name))


class SpmdUNetEngine(SpmdFluxEngine):
    """SDXL-class UNet replicas (``exec/unet_exec.py``): x is pulled by the NCHW->NHWC input kernel from rank
    0's buffer (peer loads), the gather kernel (eps -> Euler -> NCHW) stores into rank 0's output buffer."""

    tma_peer_inputs = ("ctx", "y")
    kernel_pulled_inputs = ("x", "t")

    def _latent_channels(self) -> int:
        return self.ex.in_ch

    def _make_spec(self, B: int) -> dict:
        bf = torch.bfloat16
        m = self.ex
        spec = {"x": ((B, self.C, self.H, self.W), bf), "t": ((B,), bf), "ctx": ((B, self.Lt, m.ctx_dim), bf)}
        if m.adm is not None:
            spec["y"] = ((B, m.adm), bf)
        spec["sig"] = ((B, 2), torch.float32)
        spec["out"] = ((B, m.out_ch, self.H, self.W), bf)
        return spec

    def _launch(self, loc: dict, fused: bool):
        y = loc.get("y")
        if fused:
            if getattr(self.ex, "fused_in", False):
                # fused scatter + conv_in: the first kernel reads the latent shard AND the timesteps from rank 0's heap
                # and leaves the local NCHW copy (x_in of the Euler gather) in loc["x"] - no separate pull
                self.ex.denoise_step(loc["x"], loc["t"], loc["ctx"], y, loc["sig"],
                                     out_ptr=self.heap.peer_ptr(0, self.off["out"]), out_sample_off=self.off_local,
                                     x_src_ptr=self._src("x", self._row_bytes("x")), t_src_ptr=self._src("t", 2))
                return None
            if self.rank != 0:
                self._pull("x")
                self._pull("t")
            self.ex.denoise_step(loc["x"], loc["t"], loc["ctx"], y, loc["sig"],
                                 out_ptr=self.heap.peer_ptr(0, self.off["out"]), out_sample_off=self.off_local)
            return None
        return self.ex.denoise_step(loc["x"], loc["t"], loc["ctx"], y, loc["sig"])


class _SpmdTextDiTEngine(SpmdFluxEngine):
    """WAN / Z-Image replicas: the step inputs are latent, timestep and text features (no pooled vector, no guidance);
    latent and timestep are pulled by the fused patch-embed kernel from rank 0's heap, the text features are read
    through a TMA descriptor on the peer mapping."""

    tma_peer_inputs = ("ctx",)
    kernel_pulled_inputs = ("x", "t")

    def _launch(self, loc: dict, fused: bool):
        # WAN2.1 I2V / FLF2V: the CLIP image features follow the context
        cond = (loc["ctx"], loc["clip"]) if "clip" in loc else (loc["ctx"],)
        if fused:
            self.ex.denoise_step(loc["x"], loc["t"], *cond, loc["sig"],
                                 out_ptr=self.heap.peer_ptr(0, self.off["out"]), out_sample_off=self.off_local,
                                 x_src_ptr=self._src("x", self._row_bytes("x")),
                                 t_src_ptr=self._src("t", self._row_bytes("t")))
            return None
        return self.ex.denoise_step(loc["x"], loc["t"], *cond, loc["sig"])


class SpmdWanEngine(_SpmdTextDiTEngine):
    """WAN2.x video DiT replicas (``exec/wan_exec.py``).  ``height``/``width`` are pixel sizes, ``frames`` the
    number of LATENT frames; the video latent is staged as [B, in_dim, T, H/8, W/8] (16 channels for text-to-video, 36
    for image-to-video) and the result as [B, out_dim = 16, T, H/8, W/8].  WAN2.2 TI2V-5B (48 channels in and out) has
    a 16x VAE: [B, 48, T, H/16, W/16].  ``frame_timesteps``: ``"t"`` is [B, T], one timestep per latent frame (TI2V
    image-to-video), and the fused patch-embed kernel pulls T of them per sample.  Executors with CLIP image
    conditioning (WAN2.1 I2V / FLF2V) add a ``"clip"`` input [B, clip_tokens, clip_dim] after ``"sig"`` (default 257
    tokens, the model's ``clip_pos_tokens`` for FLF2V), read through a peer TMA descriptor like ``"ctx"``."""

    tma_peer_inputs = ("ctx", "clip")

    def __init__(self, executor, global_batch: int, frames: int, height: int, width: int, txt_len: int,
                 clip_tokens: int = 0, frame_timesteps: bool = False, **kw):
        self.T = frames
        self.Tt = frames if frame_timesteps else 1
        self.Li = 0
        if getattr(executor, "conditioning_kwargs", ()):
            self.Li = clip_tokens or executor.clip_pos_tokens or 257
        super().__init__(executor, global_batch, height, width, txt_len, **kw)

    def _pixels_per_latent(self) -> int:
        return 16 if self.ex.params.out_dim == 48 else 8          # WAN2.2 VAE (48 channels) / WAN2.1 VAE

    def _latent_channels(self) -> int:
        return self.ex.params.in_dim

    def _make_spec(self, B: int) -> dict:
        p, bf = self.ex.params, torch.bfloat16
        t = (B, self.Tt) if self.Tt > 1 else (B,)
        spec = {"x": ((B, self.C, self.T, self.H, self.W), bf), "t": (t, bf), "ctx": ((B, self.Lt, p.text_dim), bf),
                "sig": ((B, 2), torch.float32)}
        if self.Li:
            spec["clip"] = ((B, self.Li, p.clip_dim), bf)
        spec["out"] = ((B, p.out_dim, self.T, self.H, self.W), bf)
        return spec


class SpmdZImageEngine(_SpmdTextDiTEngine):
    """Z-Image / NextDiT replicas (``exec/zimage_exec.py``)."""

    def _latent_channels(self) -> int:
        return self.ex.params.in_channels

    def _make_spec(self, B: int) -> dict:
        p, bf = self.ex.params, torch.bfloat16
        shape = (B, self.C, self.H, self.W)
        return {"x": (shape, bf), "t": ((B,), bf), "ctx": ((B, self.Lt, p.cap_feat_dim), bf),
                "sig": ((B, 2), torch.float32), "out": (shape, bf)}
