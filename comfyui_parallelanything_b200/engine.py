"""In-process multi-device engine: replicate once, then split/run/gather per step.

This is the B200-first re-design of the reference's ``setup_parallel`` +
``parallel_forward`` closure (/root/reference/any_device_parallel.py:917-1471):

===========================  =====================================================
reference                    here
===========================  =====================================================
closure state + ``_parallel_*``  ``ParallelEngine`` object (same ``_parallel_*`` attrs are
attrs (ADP:1203-1208, 1452)      still published on the module for tooling parity)
ThreadPoolExecutor per call      persistent ``DeviceWorker`` threads (parallel/workers.py)
2x device sync per worker        stream/event ordering only, no host-blocking sync
blocking ``.to`` + ``torch.cat``   async P2P copies on side streams, peers write their rows
                                 at final offsets of a pre-allocated output (no cat)
context re-sent every step       conditioning cache keyed on tensor identity+version (K3)
CPU-bounce weight clone          D2D clone (utils/replicate.py)
===========================  =====================================================

When the wrapped module belongs to a model family with a native executor
(``comfyui_parallelanything_b200.exec``) and the device is a B200, the replica is
the hand-written sm_100a executor instead of the torch module; the engine logic is
identical.  The multi-process (one rank per GPU, in-kernel NVLink scatter/gather)
variant lives in ``parallel/spmd.py``.
"""
from __future__ import annotations

import threading
import time
import weakref
from typing import Any, Dict, List, Optional, Sequence, Tuple

import torch
import torch.nn as nn

from . import chain as chain_mod
from . import exec as native_exec
from .parallel import pipeline as pp
from .parallel import split as sp
from .parallel.workers import WorkerPool, device_scope
from .utils import dtypes, faults, log, memory, replicate
from .utils.config import EngineConfig

_PARALLEL_ATTRS = (
    "_true_parallel_active", "_parallel_devices", "_parallel_streams", "_parallel_weights",
    "_auto_vram_balance", "_parallel_purge_cache", "_parallel_purge_models", "_parallel_replicas",
    "_parallel_engine",
)


def _is_oom(e: BaseException) -> bool:
    return isinstance(e, torch.cuda.OutOfMemoryError) or "out of memory" in str(e).lower()


class _Slot:
    """One active chain entry."""
    __slots__ = ("index", "name", "device", "replica", "stream", "weight", "worker")

    def __init__(self, index: int, name: str, replica: nn.Module, stream, weight: float):
        self.index = index
        self.name = name
        self.device = torch.device(name)
        self.replica = replica
        self.stream = stream
        self.weight = weight
        self.worker = None


class ParallelEngine:
    def __init__(self, target_model: nn.Module, device_chain: Sequence, config: Optional[EngineConfig] = None):
        self.config = (config or EngineConfig()).validate()
        self.target = target_model
        self.entries = chain_mod.parse_chain(device_chain)
        self.slots: List[_Slot] = []
        self.replicas: Dict[str, nn.Module] = {}
        self.streams: Dict[str, Any] = {}
        self.pool = WorkerPool()
        self.metrics = log.Metrics()
        self.step = 0
        self._orig_forward = None
        self._cond_cache: Dict[Tuple, Any] = {}
        self._lock = threading.Lock()
        self._peer_ready = False
        self._io: Dict[Tuple, dict] = {}       # fixed staging buffers of the fused path, keyed on shapes + split
        self._native_src = None                # first native executor built from the module: source of the replication
        self._native_shells: List[Any] = []    # executors of the same geometry on other GPUs, filled over NVLink
        self.setup_report: Dict[str, Any] = {}
        self._host_exec = None                 # native per-GPU launcher threads (csrc/runtime HostExecutor)
        self._ulysses = None                   # sequence-parallel batch-1 path (exec/{flux,wan}_sp.py), native replicas only
        self.active = False

    # ------------------------------------------------------------------ setup
    @property
    def device_names(self) -> List[str]:
        return [s.name for s in self.slots]

    @property
    def weights(self) -> List[float]:
        return [s.weight for s in self.slots]

    @property
    def lead_device(self) -> torch.device:
        return self.slots[0].device

    def _merge_duplicate_cuda(self) -> None:
        seen: Dict[str, int] = {}
        merged: List[chain_mod.DeviceEntry] = []
        for e in self.entries:
            if e.device.startswith("cuda") and e.device in seen:
                j = seen[e.device]
                merged[j] = chain_mod.DeviceEntry(e.device, merged[j].percentage + e.percentage)
                log.warn("device %s listed twice; merged its percentages", e.device)
                continue
            seen.setdefault(e.device, len(merged))
            merged.append(e)
        self.entries = merged

    def setup(self, has_lora: bool = False, original_device: Optional[torch.device] = None) -> bool:
        """Replicate onto every chain device.  Returns False (and leaves the model
        untouched) when nothing usable remains — same contract as ADP:1138-1150."""
        cfg = self.config
        self._merge_duplicate_cuda()
        names = [e.device for e in self.entries]
        bad = chain_mod.validate_devices(names)
        if bad is not None:
            log.error("Invalid device %r in chain; leaving model untouched", bad)
            return False
        weights = chain_mod.normalize_weights([e.percentage for e in self.entries])
        log.info("Using devices: %s", names)
        log.info("Workload split: %s", [f"{w * 100:.1f}%" for w in weights])
        safe_attn = {n for n in names if not dtypes.check_sm80_support(n)}
        for n in sorted(safe_attn):
            log.info("%s is below SM 8.0: using plain attention on its replica", n)

        if original_device is None:
            original_device = memory.module_device(self.target) or torch.device("cpu")

        built: List[_Slot] = []
        try:
            for i, (name, w) in enumerate(zip(names, weights)):
                if name in self.replicas:                       # duplicate (cpu,cpu): alias one replica
                    built.append(_Slot(i, name, self.replicas[name], self.streams.get(name), w))
                    continue
                dev = torch.device(name)
                try:
                    same = (dev == original_device) or (dev.type == "cpu" and original_device.type == "cpu")
                    native = self._native_replica(dev, name, i)
                    if native is not None:
                        replica = native
                    elif same and not has_lora:
                        faults.check_setup(name, i)
                        replica = self.target
                        log.info("Reusing original model on %s", name)
                    else:
                        if dev.type == "cuda":
                            log.info("Cloning to %s (free VRAM %.0f MiB)", name, memory.get_free_vram(name))
                        replica = replicate.safe_model_clone(self.target, dev, safe_attention=name in safe_attn,
                                                             index=i)
                        if replica is self.target and has_lora:
                            # LoRA baked: even the home device gets its own frozen copy (ADP:1073-1086)
                            replica = replicate._finalize_replica(
                                replicate.clone_module_d2d(self.target, dev), dev, name in safe_attn)
                    stream = torch.cuda.Stream(device=dev) if dev.type == "cuda" else None
                except Exception as e:
                    if _is_oom(e):
                        log.warn("OOM while cloning to %s, skipping this device", name)
                        memory.aggressive_cleanup()
                        continue
                    raise
                self.replicas[name] = replica
                if stream is not None:
                    self.streams[name] = stream
                built.append(_Slot(i, name, replica, stream, w))
            if not built:
                raise RuntimeError("no device could hold a replica")
        except Exception as e:
            log.error("Parallel setup failed: %s", e)
            self._drop_replicas()
            return False

        if len(built) != len(names):                            # renormalise over survivors
            tot = sum(s.weight for s in built)
            for s in built:
                s.weight = s.weight / tot if tot > 0 else 1.0 / len(built)
            log.info("Surviving devices: %s", [s.name for s in built])
        for j, s in enumerate(built):
            s.index = j
            s.worker = self.pool.add(s.device, s.stream)
        self.slots = built

        shells = [sh for sh in self._native_shells if any(s.replica is sh for s in built)]
        if shells and self._native_src is not None:
            from .parallel import replicate_nvl
            try:
                rep = replicate_nvl.replicate_inprocess(self._native_src, shells, method=self.config.replicate)
            except Exception as e:
                log.error("Weight replication over NVLink failed: %s", e)
                self._drop_replicas()
                return False
            self.setup_report["replication"] = rep
            log.info("Replicated %.1f GB of packed weights to %d GPU(s) via %s in %.3f s (%.0f GB/s)",
                     rep["bytes"] / 1e9, rep["receivers"], rep["method"], rep["seconds"], rep["gbps"])
        self._native_shells = []
        self._setup_native_runtime()
        if cfg.workload_split and len(built) > 1:
            log.info("Configuring pipeline (layer-split) plan for batch=1")
            pp.wrap_blocks(self.replicas[built[0].name], self.replicas, [s.name for s in built],
                           [s.weight for s in built])
        self.active = True
        return True

    def _setup_native_runtime(self) -> None:
        """Peer access between the lead and EVERY native replica (not only the first active set), and one native
        launcher thread per GPU that replays captured step graphs without the GIL."""
        native = [s for s in self.slots if getattr(s.replica, "pa_native", False) and s.device.type == "cuda"]
        if len(native) < 2 or self.slots[0] not in native:
            self._peer_ready = len(native) == len(self.slots) == 1
            return
        from . import ops
        C = ops.require()
        lead = self.lead_device.index
        try:
            ok = all(C.enable_peer_access(s.device.index, lead) and C.enable_peer_access(lead, s.device.index)
                     for s in native)
        except Exception as e:
            log.warn("peer access could not be enabled (%s); using copy-based scatter/gather", e)
            ok = False
        self._peer_ready = bool(ok) and len(native) == len(self.slots)
        if self._peer_ready and self.config.batch1_mode in ("auto", "ulysses") and self.config.workload_split:
            from .exec import sp_common
            try:
                self._ulysses, why = sp_common.build([s.replica for s in self.slots],
                                                     timeout_ms=self.config.flag_timeout_ms)
            except Exception as e:
                self._ulysses, why = None, str(e)
            if self._ulysses is not None:
                log.info("batch=1 will run sequence-parallel (Ulysses, %s) over %d GPUs", self._ulysses.family,
                         len(self.slots))
            elif self.config.batch1_mode == "ulysses":
                log.warn("PA_BATCH1=ulysses requested but %s; using the layer-split mode", why)
        if self._peer_ready and self.config.host_threads and self.config.cuda_graphs:
            try:
                self._host_exec = C.HostExecutor([s.device.index for s in self.slots])
            except Exception as e:
                log.warn("native launcher threads unavailable (%s); replaying graphs from Python workers", e)
                self._host_exec = None

    def describe(self) -> dict:
        """Small JSON-able summary (bench / logs)."""
        return {"devices": self.device_names, "native": [bool(getattr(s.replica, "pa_native", False)) for s in self.slots],
                "peer_fused": bool(self._peer_ready), "host_threads": self._host_exec is not None,
                "graphs": {s.name: len(getattr(s.replica, "_graphs", ())) for s in self.slots
                           if hasattr(getattr(s.replica, "_graphs", None), "__len__")},
                "counters": dict(self.metrics.counters), "setup": dict(self.setup_report)}

    def _native_replica(self, dev: torch.device, name: str, index: int):
        """B200 + known model family -> hand-written sm_100a executor packed straight from the
        source weights (device-to-device), instead of a torch replica."""
        if self.config.backend == "torch" or dev.type != "cuda":
            return None
        build = native_exec.builder_for(self.target)
        if build is None:
            return None
        from . import ops
        if not ops.native_ok(dev):
            if self.config.backend == "fused":
                raise RuntimeError(f"backend=fused requested but no native library/sm_100 device for {name}: "
                                   f"{ops.load_error()!r}")
            return None
        faults.check_setup(name, index)
        if self._native_src is not None and self.config.replicate != "rebuild":
            # The packed weights already exist on another GPU: allocate an executor of the same geometry here and fill
            # it device-to-device afterwards (NVSwitch multicast kernel, or peer copies) instead of re-packing /
            # re-quantising from the torch module once per device (reference: CPU bounce per device, ADP:600-663).
            from .parallel import replicate_nvl
            log.info("Allocating native %s replica on %s (free VRAM %.0f MiB); weights arrive over NVLink",
                     native_exec.family_of(self.target) or "?", name, memory.get_free_vram(name))
            shell = replicate_nvl.shell_like(self._native_src, dev)
            self._native_shells.append(shell)
            return shell
        log.info("Building native sm_100a %s executor on %s (free VRAM %.0f MiB)",
                 native_exec.family_of(self.target) or "?", name, memory.get_free_vram(name))
        ex = build(self.target, dev, cuda_graphs=self.config.cuda_graphs, fp8=self.config.fp8)
        self._native_src = ex
        return ex

    # ------------------------------------------------------------------ forward
    def _replica_call(self, replica: nn.Module, *a, **k):
        fn = replica
        if replica is self.target and self._orig_forward is not None:
            fn = self._orig_forward
        return fn(*a, **k)

    def _lead_only(self, x, timesteps, context, kwargs):
        lead = self.slots[0]
        with torch.no_grad():
            return self._replica_call(lead.replica, x, timesteps, context=context, **kwargs)

    def split_sizes(self, batch: int) -> List[int]:
        names, weights = self.device_names, self.weights
        if self.config.auto_vram_balance:
            return chain_mod.split_sizes_vram(batch, names, weights, self.config.split_mode)
        return chain_mod.split_sizes(batch, weights, self.config.split_mode)

    def forward(self, x, timesteps, context=None, **kwargs):
        """Replacement for ``diffusion_model.forward(x, timesteps, context=None, **kw)``."""
        step = self.step
        self.step += 1
        try:
            batch = sp.get_batch_size(x)
            n = len(self.slots)
            if batch == 1 and self.config.workload_split and self._ulysses is not None \
                    and self._can_ulysses(x, timesteps, context):
                try:
                    return self._forward_ulysses(step, x, timesteps, context, kwargs)
                except Exception as e:  # noqa: BLE001
                    if _is_oom(e):
                        raise
                    # a stalled / dead peer (flag watchdog), a failed capture, ...: this sample is recomputed on the lead
                    # replica below and the chain stays on the layer-split / lead path from now on
                    log.error("sequence-parallel batch-1 step failed (%s); disabling it for this model", e)
                    self.metrics.incr("ulysses_fallbacks")
                    try:
                        self._ulysses.release()
                    finally:
                        self._ulysses = None
            if batch == 1 and self.config.workload_split:
                with pp.pipeline_mode(True):
                    lead = self.slots[0]
                    return self._replica_call(lead.replica, x, timesteps, context=context, **kwargs)
            if not self.config.workload_split or (batch < n and self.config.small_batch == "lead"):
                return self._lead_only(x, timesteps, context, kwargs)
            if batch < n:
                # The reference runs the lead device alone here (ADP:1308).  With 8 GPUs and a batch of 4 that idles
                # seven of them, so instead the ``batch`` heaviest devices get one sample each (chain order kept).
                keep = sorted(sorted(range(n), key=lambda i: (-self.slots[i].weight, i))[:batch])
                active = [(self.slots[i], 1) for i in keep]
                self.metrics.incr("small_batch_spread_steps")
                return self._data_parallel(step, batch, active, x, timesteps, context, kwargs)
            if self.config.pair_cfg and batch % 2 == 0 and batch // 2 >= n:
                return self._forward_cfg_paired(step, batch, x, timesteps, context, kwargs)
            sizes = self.split_sizes(batch)
            active = [(s, z) for s, z in zip(self.slots, sizes) if z > 0]
            if not active:
                raise RuntimeError("No active devices available")
            if len(active) == 1:
                with torch.no_grad():
                    return self._replica_call(active[0][0].replica, x, timesteps, context=context, **kwargs)
            return self._data_parallel(step, batch, active, x, timesteps, context, kwargs)
        except RuntimeError as e:
            if _is_oom(e):
                log.warn("OOM in parallel forward, cleaning up and falling back to the lead device")
                memory.aggressive_cleanup()
                self.metrics.incr("oom_fallbacks")
                return self._lead_only(x, timesteps, context, kwargs)
            raise

    __call__ = forward

    def _forward_cfg_paired(self, step, batch, x, timesteps, context, kwargs):
        """CFG-aware split (SURVEY §2.3 "CFG parallel"): ComfyUI hands the sampler's cond and uncond halves as
        one 2B batch; the reference splits it blindly, so a sample's two halves usually land on different
        devices.  Here sample i and i + B/2 always travel together (so a replica can apply
        ``uncond + s*(cond - uncond)`` locally and ship half the bytes back)."""
        half = batch // 2
        pair_sizes = self.split_sizes(half)
        idx, sizes = [], []
        off = 0
        for z in pair_sizes:
            idx += list(range(off, off + z)) + list(range(half + off, half + off + z))
            sizes.append(2 * z)
            off += z
        dev = x.device if isinstance(x, torch.Tensor) else None
        perm = torch.tensor(idx, dtype=torch.long, device=dev)

        def pick(v):
            if isinstance(v, torch.Tensor) and v.dim() > 0 and v.shape[0] == batch:
                return v.index_select(0, perm.to(v.device))
            if isinstance(v, (list, tuple)):
                return type(v)(pick(t) for t in v)
            if isinstance(v, dict):
                return {k: pick(t) for k, t in v.items()}
            return v
        active = [(s, z) for s, z in zip(self.slots, sizes) if z > 0]
        if len(active) == 1:
            return self._lead_only(x, timesteps, context, kwargs)
        out_p = self._data_parallel(step, batch, active, pick(x), pick(timesteps), pick(context), pick(kwargs))
        inv = torch.empty_like(perm)
        inv[perm] = torch.arange(batch, device=perm.device)

        def unpick(v):
            if isinstance(v, torch.Tensor):
                return v.index_select(0, inv.to(v.device))
            if isinstance(v, (list, tuple)):
                return type(v)(unpick(t) for t in v)
            return v
        self.metrics.incr("cfg_paired_steps")
        return unpick(out_p)

    def _data_parallel(self, step: int, batch: int, active, x, timesteps, context, kwargs):
        act_sizes = [z for _, z in active]
        offs = chain_mod.offsets(act_sizes)
        x_chunks = sp.split_value(x, act_sizes)
        t_chunks = sp.split_value(timesteps, act_sizes)
        c_chunks = sp.split_value(context, act_sizes) if context is not None else [None] * len(active)
        k_chunks = sp.split_kwargs(kwargs, act_sizes, batch)
        lead_dev = self.lead_device
        lead_stream = torch.cuda.current_stream(lead_dev) if lead_dev.type == "cuda" else None
        if self._can_fuse(active, x):
            return self._data_parallel_fused(step, batch, active, offs, x, t_chunks, c_chunks, k_chunks, lead_stream)
        out_box: Dict[str, Any] = {"buf": None}
        results: List[Any] = [None] * len(active)
        t0 = time.perf_counter()

        def run(i: int):
            slot = active[i][0]
            dev = slot.device
            pp.set_pipeline_mode(False)
            faults.check_step(step, slot.name, slot.index)

            def body():
                x_in = sp.move_to_device(x_chunks[i], dev, non_blocking=True)
                t_in = sp.move_to_device(t_chunks[i], dev, non_blocking=True)
                c_in = self._cached_move(("ctx", i), c_chunks[i], dev)
                k_in = {k: sp.move_to_device(v, dev, non_blocking=True) for k, v in k_chunks[i].items()}
                with torch.no_grad():
                    out = self._replica_call(slot.replica, x_in, t_in, context=c_in, **k_in)
                # gather: write rows at their final offset on the lead device (no cat)
                with self._lock:
                    if out_box["buf"] is None:
                        # Allocate from the LEAD stream's pool: every writer is ordered after ``lead_stream`` (peers
                        # copy on it, the lead's own side stream waited on it), so a block the allocator hands back
                        # cannot still be in use by work that is only ordered on some replica's side stream.
                        if lead_stream is not None:
                            with torch.cuda.stream(lead_stream):
                                out_box["buf"] = sp.output_like(out, batch, lead_dev)
                        else:
                            out_box["buf"] = sp.output_like(out, batch, lead_dev)
                buf = out_box["buf"]
                if buf is None:                     # non-tensor outputs: fall back to concat
                    return sp.move_to_device(out, lead_dev)
                if lead_stream is not None and dev == lead_dev and slot.stream is not None:
                    _record_stream(buf, slot.stream)    # the lead replica writes its rows on its side stream
                sp.write_rows(buf, out, offs[i])
                return None

            if dev.type == "cuda":
                with torch.cuda.device(dev):
                    # ``torch.cuda.stream(s)`` also makes s.device current: enter the lead-stream context FIRST and
                    # the replica's own stream LAST so the replica's forward runs with ITS device current (model
                    # code that says ``device="cuda"`` / ``torch.cuda.current_stream()`` must land on ``dev``),
                    # exactly as the reference guarantees with set_device + cuda.device(dev) (ADP:1370, 1386).
                    ctxs = []
                    if lead_stream is not None and lead_dev != dev:
                        ctxs.append(torch.cuda.stream(lead_stream))
                    if slot.stream is not None:
                        ctxs.append(torch.cuda.stream(slot.stream))
                    ctxs.append(torch.cuda.device(dev))
                    with _nested(ctxs):
                        if slot.stream is not None and lead_stream is not None and lead_dev == dev:
                            slot.stream.wait_stream(lead_stream)
                        r = body()
                        if slot.stream is not None and lead_stream is not None and lead_dev == dev:
                            lead_stream.wait_stream(slot.stream)
                        return r
            if dev.type == "xpu":
                with device_scope(dev):                 # torch.xpu.device(dev) + sync before/after (ADP:1398-1403)
                    return body()
            return body()

        futures = [active[i][0].worker.submit(lambda i=i: run(i)) for i in range(len(active))]
        errors: List[Tuple[str, BaseException]] = []
        for i, f in enumerate(futures):
            try:
                results[i] = f.result()
            except BaseException as e:  # noqa: BLE001 - reported below
                errors.append((active[i][0].name, e))
        if errors:
            for name, e in errors:
                log.error("on %s: %s", name, e)
            raise errors[0][1]
        self.metrics.record(step=step, host_ms=(time.perf_counter() - t0) * 1e3, batch=batch, sizes=act_sizes)
        if out_box["buf"] is not None:
            return out_box["buf"]
        if any(r is None for r in results):
            missing = [active[i][0].name for i, r in enumerate(results) if r is None]
            raise RuntimeError(f"Missing results from devices: {missing}")
        return sp.concatenate_results(results, dim=0)

    # ---- native executors, one process: scatter/gather happen inside the replicas' kernels --------------
    def _can_fuse(self, active, x) -> bool:
        if self.config.backend in ("torch", "nccl") or not isinstance(x, torch.Tensor):
            return False
        if x.device != self.lead_device or x.device.type != "cuda" or not x.is_floating_point():
            return False
        if not all(getattr(s.replica, "pa_native", False) and hasattr(s.replica, "forward_shard") for s, _ in active):
            return False
        return self._peer_ready

    def _io_block(self, active, x, t_chunks, c_chunks, k_chunks) -> dict:
        """Fixed device buffers for one (shape, split) configuration.  A sampler hands the hooked forward a NEW latent
        tensor every step (and ComfyUI re-concatenates cond/uncond conditioning every step), while a captured CUDA
        graph bakes in every pointer: so the step's inputs are staged into these buffers (tiny async copies that also
        do the dtype conversion) and the replicas' kernels only ever see stable addresses."""
        def sig(v):
            return (tuple(v.shape), str(v.dtype)) if isinstance(v, torch.Tensor) else None
        key = (tuple(x.shape), tuple((s.index, z) for s, z in active), tuple(sig(t) for t in t_chunks),
               tuple(sig(c) for c in c_chunks), tuple(tuple(sorted((k, sig(v)) for k, v in kc.items())) for kc in k_chunks))
        io = self._io.get(key)
        if io is not None:
            return io
        lead = self.lead_device
        bf = torch.bfloat16
        rep0 = active[0][0].replica
        out_shape = rep0.out_shape(tuple(x.shape)) if hasattr(rep0, "out_shape") else tuple(x.shape)
        io = {"x": torch.empty(tuple(x.shape), dtype=bf, device=lead), "out": torch.empty(out_shape, dtype=bf, device=lead),
              "slots": []}
        for i, (slot, _z) in enumerate(active):
            dev = slot.device

            def stage(v):
                if isinstance(v, torch.Tensor) and v.is_floating_point():
                    return torch.empty(tuple(v.shape), dtype=bf, device=dev)
                return None
            io["slots"].append({"t": stage(t_chunks[i]), "ctx": stage(c_chunks[i]), "ctx_src": None,
                                "kw": {k: stage(v) for k, v in k_chunks[i].items()}})
        if len(self._io) >= 8:                      # a session walking through many shapes must not pin them all
            self._io.pop(next(iter(self._io)))
        self._io[key] = io
        return io

    def _stage_conditioning(self, st: dict, name: str, buf: torch.Tensor, src: torch.Tensor) -> torch.Tensor:
        """Copy the step-invariant conditioning ``src`` into its staging buffer only when it changed (another tensor, or
        written in place since), so the replica's conditioning cache and its captured graph stay valid across steps."""
        # a split chunk is a fresh view object every step: identify it by the tensor it was split from (the sampler's
        # conditioning, which stays the same object) plus where and how large the chunk is
        base = src._base if src._base is not None else src
        ident = (id(base), base.data_ptr(), base._version, src.data_ptr(), tuple(src.shape))
        key = "ctx_src" if name == "ctx" else name + "_src"
        if not self.config.cache_conditioning or st.get(key) is None or st[key][0] != ident:
            buf.copy_(src, non_blocking=True)           # conditioning changed (or first step)
            st[key] = (ident, base)                     # keep the source alive: id/ptr stay unique
        else:
            self.metrics.incr("cond_cache_hits")
        return buf

    def _data_parallel_fused(self, step, batch, active, offs, x, t_chunks, c_chunks, k_chunks, lead_stream):
        """Every replica's FIRST kernel loads its latent shard from the lead GPU's staging buffer (NVLink peer loads)
        and its LAST kernel stores its output rows at their final offset in the lead GPU's output buffer; the host only
        orders streams (no cat, no device-wide sync).  Steps after the second replay ONE CUDA graph per GPU, launched
        by native host threads (no GIL, no Python in the per-GPU path)."""
        io = self._io_block(active, x, t_chunks, c_chunks, k_chunks)
        xs, out = io["x"], io["out"]
        sample_bytes = xs[0].numel() * xs.element_size()
        t0 = time.perf_counter()
        xs.copy_(x, non_blocking=True)                                   # lead stream; also converts fp16/fp32 -> bf16

        # Small per-replica inputs are staged from THIS thread before any replica starts: a cross-device copy orders
        # itself after the source device's current stream, so issued from a worker it can queue behind the lead
        # replica's whole step (measured: 2 GPUs overlapped only ~70 %).
        calls = []
        for i, (slot, size) in enumerate(active):
            dev, st = slot.device, io["slots"][i]
            with torch.cuda.device(dev), torch.cuda.stream(slot.stream):
                slot.stream.wait_stream(lead_stream)
                t_in = t_chunks[i]
                if st["t"] is not None:
                    st["t"].copy_(t_in, non_blocking=True)
                    t_in = st["t"]
                c_in = c_chunks[i]
                if st["ctx"] is not None:
                    c_in = self._stage_conditioning(st, "ctx", st["ctx"], c_in)
                k_in = {}
                cond_kw = getattr(slot.replica, "conditioning_kwargs", ())
                for k, v in k_chunks[i].items():
                    buf = st["kw"].get(k)
                    if buf is not None and k in cond_kw:
                        k_in[k] = self._stage_conditioning(st, "kw:" + k, buf, v)
                    elif buf is not None:
                        buf.copy_(v, non_blocking=True)
                        k_in[k] = buf
                    else:
                        k_in[k] = sp.move_to_device(v, dev, non_blocking=True)
            shape = (size,) + tuple(xs.shape[1:])
            calls.append((slot, (xs.data_ptr() + offs[i] * sample_bytes, shape, t_in, c_in, out.data_ptr(), offs[i]), k_in))

        # ---- replay path: every replica already holds a captured graph for exactly these buffers
        launched = False
        if self._host_exec is not None:
            handles = []
            for slot, args, k_in in calls:
                fn = getattr(slot.replica, "shard_graph_handle", None)
                h = fn(*args, **k_in) if fn is not None else 0
                if not h:
                    handles = None
                    break
                handles.append(h)
            if handles is not None:
                for (slot, _a, _k), h in zip(calls, handles):
                    faults.check_step(step, slot.name, slot.index)
                    self._host_exec.launch_graph(slot.index, h, slot.stream.cuda_stream)
                self._host_exec.sync()                  # launches are enqueued (GIL released); no device sync
                for slot, _a, _k in calls:
                    lead_stream.wait_stream(slot.stream)
                self.metrics.incr("native_graph_steps")
                launched = True

        if not launched:
            def run(i: int):
                slot, args, k_in = calls[i]
                pp.set_pipeline_mode(False)
                faults.check_step(step, slot.name, slot.index)
                with torch.cuda.device(slot.device), torch.cuda.stream(slot.stream):
                    slot.replica.forward_shard(*args, **k_in)
                    lead_stream.wait_stream(slot.stream)
                return None

            futures = [calls[i][0].worker.submit(lambda i=i: run(i)) for i in range(len(calls))]
            errors = []
            for i, f in enumerate(futures):
                try:
                    f.result()
                except BaseException as e:  # noqa: BLE001
                    errors.append((calls[i][0].name, e))
            if errors:
                for name, e in errors:
                    log.error("on %s: %s", name, e)
                raise errors[0][1]
        self.metrics.record(step=step, host_ms=(time.perf_counter() - t0) * 1e3, batch=batch,
                            sizes=[z for _, z in active], fused=True, native_launch=launched)
        # the sampler may keep every step's result alive: hand back a copy, the fixed buffer is rewritten next step
        res = out.clone()
        return res if x.dtype == res.dtype else res.to(x.dtype)

    # ---- batch == 1: sequence-parallel (Ulysses) over all native FLUX / WAN replicas -------------------------------
    def _can_ulysses(self, x, timesteps, context) -> bool:
        if not (isinstance(x, torch.Tensor) and isinstance(context, torch.Tensor) and isinstance(timesteps, torch.Tensor)):
            return False
        if x.device != self.lead_device or not x.is_floating_point():
            return False
        return bool(self._ulysses.accepts(x, context))

    def _forward_ulysses(self, step, x, timesteps, context, kwargs):
        """One sample, every GPU of the chain: token-sliced linear layers, head-sliced attention, peer-pull all-to-all
        (exec/flux_sp.py, exec/wan_sp.py).  Inputs are staged into fixed buffers (a sampler passes fresh tensors), each GPU's share of
        the step is one CUDA graph; the velocity rows land in the lead GPU's output buffer through the fused gather."""
        sp = self._ulysses
        sp.check_polled()                  # error words of the PREVIOUS step (copied to pinned memory at its end)
        lead_dev = self.lead_device
        lead_stream = torch.cuda.current_stream(lead_dev)
        bf = torch.bfloat16
        key = sp.io_key(x, timesteps, context, kwargs)
        io = self._io.get(key)
        if io is None:
            io = {"x": torch.empty(tuple(x.shape), dtype=bf, device=lead_dev),
                  "out": torch.empty(sp.out_shape(x), dtype=bf, device=lead_dev),
                  "slots": [sp.slot_buffers(slot.device, x, timesteps, context, kwargs) for slot in self.slots]}
            if len(self._io) >= 8:
                self._io.pop(next(iter(self._io)))
            self._io[key] = io
        t0 = time.perf_counter()
        xs, out = io["x"], io["out"]
        xs.copy_(x, non_blocking=True)
        wss = sp.workspace(*sp.geometry(x, timesteps, context, kwargs))
        for g, (slot, st) in enumerate(zip(self.slots, io["slots"])):
            with torch.cuda.device(slot.device), torch.cuda.stream(slot.stream), torch.no_grad():
                slot.stream.wait_stream(lead_stream)
                sp.stage(st, timesteps, context, kwargs, self.config.cache_conditioning)
                sp.pre_step(g, wss, st)          # conditioning-only precomputes stay outside the step graph
        gkey = ("sp",) + key[1:]

        def body(g):
            sp.run_rank(g, wss, xs.data_ptr(), io["slots"][g], out.data_ptr())

        caches = [s.replica._graphs for s in self.slots]
        states = [c.state(gkey) for c in caches]
        if gkey not in sp.warmed:
            # very first step of this shape: load every kernel on every GPU without cross-GPU waits (FluxUlysses.warm_up),
            # one GPU after the other from this thread, then start the real (concurrent) step
            for g, slot in enumerate(self.slots):
                with torch.cuda.device(slot.device), torch.cuda.stream(slot.stream), torch.no_grad():
                    sp.warm_up(g, wss, xs.data_ptr(), io["slots"][g], out.data_ptr())
            for slot in self.slots:
                torch.cuda.synchronize(slot.device)
            sp.warmed.add(gkey)
        if all(st_ == "seen" for st_ in states) and all(c.enabled for c in caches):
            # second step: capture EVERY GPU's graph before any of them runs.  The step's kernels wait on the other GPUs'
            # flags, and torch's capture prologue (device synchronise + empty_cache -> cudaFree, which synchronises all
            # devices) would dead-lock against a peer that already replays its graph (see GraphCache.capture_only).
            for dsync in self.slots:
                torch.cuda.synchronize(dsync.device)
            for g, slot in enumerate(self.slots):
                with torch.cuda.device(slot.device), torch.cuda.stream(slot.stream), torch.no_grad():
                    caches[g].capture_only(gkey, lambda g=g: body(g))
            states = [c.state(gkey) for c in caches]
        all_graph = all(st_ == "graph" for st_ in states)
        launched = False
        if all_graph and self._host_exec is not None:
            handles = [c.exec_handle(gkey) for c in caches]
            if all(handles):
                for s, h in zip(self.slots, handles):
                    self._host_exec.launch_graph(s.index, h, s.stream.cuda_stream)
                self._host_exec.sync()
                for s in self.slots:
                    lead_stream.wait_stream(s.stream)
                self.metrics.incr("native_graph_steps")
                launched = True
        if not launched:
            def run(g: int):
                slot = self.slots[g]
                pp.set_pipeline_mode(False)
                faults.check_step(step, slot.name, slot.index)
                with torch.cuda.device(slot.device), torch.cuda.stream(slot.stream), torch.no_grad():
                    if all_graph:
                        caches[g].replay(gkey)
                    elif states[g] in ("new", "seen") and caches[g].enabled and not all_graph:
                        # eager pass on every GPU at once (marks the key as seen); mixed states stay eager
                        body(g)
                        if caches[g].state(gkey) == "new":
                            caches[g]._graphs[gkey] = "seen"
                    else:
                        body(g)
                    lead_stream.wait_stream(slot.stream)
            futures = [self.slots[g].worker.submit(lambda g=g: run(g)) for g in range(len(self.slots))]
            errors = []
            for g, f in enumerate(futures):
                try:
                    f.result()
                except BaseException as e:  # noqa: BLE001
                    errors.append((self.slots[g].name, e))
            if errors:
                for name, e in errors:
                    log.error("on %s: %s", name, e)
                raise errors[0][1]
        for g, slot in enumerate(self.slots):
            with torch.cuda.device(slot.device), torch.cuda.stream(slot.stream):
                sp.poll_async(g)           # 4-byte D2H per GPU, looked at by the next step (no host sync here)
        self.metrics.incr("ulysses_steps")
        self.metrics.record(step=step, host_ms=(time.perf_counter() - t0) * 1e3, batch=1, sizes=[1], ulysses=True,
                            native_launch=launched)
        res = out.clone()
        return res if x.dtype == res.dtype else res.to(x.dtype)

    def _cached_move(self, key, value, dev):
        """Conditioning is constant across the steps of one sampling run; re-use the
        device copy while the source tensor object/version is unchanged (SURVEY K3)."""
        if value is None or not self.config.cache_conditioning or not isinstance(value, torch.Tensor):
            return sp.move_to_device(value, dev, non_blocking=True)
        if value.device == dev:
            return value
        sig = (key, str(dev), value.data_ptr(), tuple(value.shape), value.dtype, value._version,
               tuple(value.stride()))
        with self._lock:
            hit = self._cond_cache.get((key, str(dev)))
        if hit is not None and hit[0] == sig:
            self.metrics.incr("cond_cache_hits")
            return hit[1]
        moved = sp.move_to_device(value, dev, non_blocking=True)
        with self._lock:
            self._cond_cache[(key, str(dev))] = (sig, moved, value)   # keep src alive: ptr stays unique
        return moved

    # ------------------------------------------------------------------ teardown
    def _drop_replicas(self) -> None:
        for name, r in list(self.replicas.items()):
            if r is self.target:
                continue
            try:
                if hasattr(r, "release"):
                    r.release()
                    continue
                memory.clear_model_caches(r, quiet=True)
                r.to("meta") if hasattr(r, "to") else None   # free device memory without a D2H copy
            except Exception:
                try:
                    r.cpu()
                except Exception:
                    pass
        self.replicas.clear()
        self.streams.clear()

    def cleanup(self) -> None:
        if not self.active and not self.replicas:
            return
        log.info("Cleaning up parallel model...")
        self.active = False
        for r in self.replicas.values():
            try:
                pp.unwrap_blocks(r)
            except Exception:
                pass
        self.pool.shutdown()
        if self._host_exec is not None:
            try:
                self._host_exec.shutdown()
            except Exception:
                pass
            self._host_exec = None
        self._io.clear()
        if self._ulysses is not None:
            self._ulysses.release()
            self._ulysses = None
        self._cond_cache.clear()
        self._drop_replicas()
        self.slots = []
        if self.config.purge_models:
            mm = memory.comfy_mm()
            if mm is not None:
                try:
                    log.info("Purging models from VRAM...")
                    mm.unload_all_models()
                except Exception as e:
                    log.warn("could not unload models: %s", e)
        if self.config.purge_cache:
            memory.aggressive_cleanup()


def _record_stream(value, stream) -> None:
    if isinstance(value, torch.Tensor):
        if value.is_cuda:
            value.record_stream(stream)
    elif isinstance(value, (list, tuple)):
        for v in value:
            _record_stream(v, stream)


class _nested:
    def __init__(self, ctxs):
        self.ctxs = ctxs

    def __enter__(self):
        for c in self.ctxs:
            c.__enter__()
        return self

    def __exit__(self, *exc):
        for c in reversed(self.ctxs):
            c.__exit__(*exc)
        return False


# ---------------------------------------------------------------------- module hook

def cleanup_parallel_model(model_ref) -> None:
    """Undo ``install`` (ADP:211-282): restore forward, free replicas, drop attrs,
    unwrap pipeline stages (the reference forgets this), optional purges."""
    model = model_ref() if isinstance(model_ref, weakref.ref) else model_ref
    if model is None or not getattr(model, "_true_parallel_active", False):
        return
    eng: Optional[ParallelEngine] = getattr(model, "_parallel_engine", None)
    if "forward" in model.__dict__:
        try:
            del model.__dict__["forward"]         # falls back to the class forward
        except Exception:
            pass
    orig = model.__dict__.pop("_original_forward", None)
    if orig is not None and getattr(orig, "__self__", None) is not model:
        model.forward = orig                      # an instance-level forward existed before us
    if eng is not None:
        eng.cleanup()
    try:
        pp.unwrap_blocks(model)
    except Exception:
        pass
    for a in _PARALLEL_ATTRS:
        if a in model.__dict__:
            try:
                delattr(model, a)
            except Exception:
                pass


def install(engine: ParallelEngine, owner: Any = None) -> None:
    """Patch ``engine.target.forward`` and publish the reference's ``_parallel_*`` attrs."""
    import types

    tm = engine.target
    engine._orig_forward = tm.forward

    def parallel_forward(self, x, timesteps, context=None, **kwargs):
        return engine.forward(x, timesteps, context=context, **kwargs)

    object.__setattr__(tm, "_original_forward", engine._orig_forward)
    object.__setattr__(tm, "forward", types.MethodType(parallel_forward, tm))
    for k, v in (("_true_parallel_active", True), ("_parallel_replicas", engine.replicas),
                 ("_parallel_devices", engine.device_names), ("_parallel_streams", engine.streams),
                 ("_parallel_weights", engine.weights), ("_auto_vram_balance", engine.config.auto_vram_balance),
                 ("_parallel_purge_cache", engine.config.purge_cache),
                 ("_parallel_purge_models", engine.config.purge_models), ("_parallel_engine", engine)):
        object.__setattr__(tm, k, v)
    if owner is not None:
        try:
            weakref.finalize(owner, cleanup_parallel_model, weakref.ref(tm))
        except TypeError:
            pass
