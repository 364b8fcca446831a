"""Shared plumbing of the sequence-parallel (Ulysses) batch-1 paths (``flux_sp.py``, ``wan_sp.py``, ``zimage_sp.py``).

One object wires the N native executors of a chain (one per GPU, same process): per-GPU flag arrays, device-resident
epoch counters and error words, descriptor tables for the peer-pull all-to-all kernel (csrc/comm/sp_a2a.cu), the
exchange itself and the dry warm-up pass.  The model-specific subclasses provide the geometry (``accepts`` / ``geometry``
/ ``workspace``), the staged per-GPU inputs (``slot_buffers`` / ``stage``) and one GPU's share of a step (``run_rank``).

Replaces the reference's batch == 1 mode (/root/reference/any_device_parallel.py:24-87, 1295-1305: one sample walks the
blocks sequentially across devices) with a mode in which every GPU works on the sample at the same time.
"""
from __future__ import annotations

import struct
from typing import Dict, List, Optional

import torch

from .. import ops


def attention_variant(hpg: int, L: int) -> Optional[int]:
    """Attention kernel for ``hpg`` heads per GPU over ``L`` tokens.  With few heads the ping-pong kernel (two 128-row
    query tiles per CTA) would leave most SMs idle: below ~3/4 of a wave, the one-tile-per-CTA kernel (variant 1)
    doubles the CTA count and halves the attention latency.  None: the default kernel."""
    return 1 if hpg * ((L + 255) // 256) < 110 else None


class UlyssesBase:
    family = "?"

    def __init__(self, executors: List, timeout_ms: int = 20000):
        self.ex = list(executors)
        self.n = len(executors)
        self.C = ops.require()
        C = self.C
        devs = [e.device for e in self.ex]
        for a in devs:
            for b in devs:
                if a != b and not C.enable_peer_access(a.index, b.index):
                    raise RuntimeError(f"no peer access {a} -> {b}")
        self.timeout_cycles = int(timeout_ms * 1.9e6)
        self.flags = [torch.zeros(C.SP_MAX_SLOTS * C.SP_MAX_RANKS, dtype=torch.int32, device=d) for d in devs]
        self.epoch = [torch.ones(1, dtype=torch.int32, device=d) for d in devs]
        self.err = [torch.zeros(1, dtype=torch.int32, device=d) for d in devs]
        self.flag_tab = [torch.tensor([f.data_ptr() for f in self.flags], dtype=torch.int64, device=d) for d in devs]
        self.err_host = torch.zeros(self.n, dtype=torch.int32).pin_memory()      # polled copies of the error words
        self._ws: Dict[tuple, list] = {}
        self._dry = False
        self.warmed = set()

    # ------------------------------------------------------------------ engine-facing protocol
    def accepts(self, x, context) -> bool:
        raise NotImplementedError

    def geometry(self, x, timesteps, context, kwargs=None) -> tuple:
        raise NotImplementedError

    def out_shape(self, x) -> tuple:
        """Shape of the step's output for the latent ``x`` (WAN image-to-video: fewer channels than its input)."""
        return tuple(x.shape)

    def workspace(self, *geometry) -> list:
        raise NotImplementedError

    def slot_buffers(self, device, x, timesteps, context, kwargs) -> dict:
        """Fixed per-GPU staging buffers for the step inputs other than the latent (a sampler passes fresh tensors)."""
        bf = torch.bfloat16
        return {"t": torch.empty(1, dtype=bf, device=device),
                "ctx": torch.empty(tuple(context.shape), dtype=bf, device=device), "ctx_src": None}

    def stage(self, st: dict, timesteps, context, kwargs, cache_conditioning: bool) -> None:
        """Copy this step's inputs into one GPU's staging buffers (called on that GPU's stream).  The ``"t"`` buffer's
        shape says how many timesteps are staged: one, or one per latent frame (WAN2.2 TI2V)."""
        t = st["t"]
        t.copy_(timesteps.reshape(-1)[:t.numel()].view(t.shape), non_blocking=True)
        ident = (id(context), context.data_ptr(), context._version)
        if not cache_conditioning or st["ctx_src"] is None or st["ctx_src"][0] != ident:
            st["ctx"].copy_(context, non_blocking=True)
            st["ctx_src"] = (ident, context)

    def io_key(self, x, timesteps, context, kwargs) -> tuple:
        return ("sp", tuple(x.shape), tuple(context.shape))

    def pre_step(self, g: int, wss, st: dict) -> None:
        """Eager work that must not live in the step graph (conditioning-only precomputes); default none."""

    def run_rank(self, g: int, wss, x_ptr: int, st: dict, out_ptr: int) -> int:
        raise NotImplementedError

    def warm_up(self, g: int, wss, x_ptr: int, st: dict, out_ptr: int) -> None:
        """First use on a GPU: run the step's launches ONCE without any cross-GPU wait.  The first launch of a kernel on a
        device loads its module / sets function attributes, and those driver calls can block on OTHER devices' running
        kernels - a peer already spinning on this GPU's flag would then dead-lock it until the flag watchdog fires."""
        self._dry = True
        try:
            self.run_rank(g, wss, x_ptr, st, out_ptr)
        finally:
            self._dry = False

    # ------------------------------------------------------------------ exchange
    def _table(self, rows, device) -> torch.Tensor:
        """(src, dst, src_pitch, dst_pitch, rows, row_bytes) copy descriptors of one GPU's pull."""
        blob = b"".join(struct.pack("<QQqqii", s, d, sp, dp, r, rb) for s, d, sp, dp, r, rb in rows)
        assert len(blob) == len(rows) * self.C.SP_DESC_BYTES
        return torch.frombuffer(bytearray(blob), dtype=torch.uint8).to(device)

    def _exchange(self, g: int, ws, slot: int, which: str) -> None:
        C = self.C
        peers = 0 if self._dry else self.n        # dry pass: same launches, nobody signals / waits (see warm_up)
        C.sp_signal(self.flag_tab[g], peers, slot, g, self.epoch[g])
        # enough CTAs that ~all SMs hold a few (each thread keeps eight 16-byte peer loads in flight)
        blocks = max(4, min(64, 592 // ws["N_" + which]))
        C.sp_pull(ws["DESC_" + which], ws["N_" + which], blocks, self.flags[g], slot, peers,
                  self.epoch[g], self.timeout_cycles, self.err[g])

    def _end_step(self, g: int) -> None:
        if not self._dry:
            self.C.sp_epoch_inc(self.epoch[g])

    def poll_async(self, g: int) -> None:
        """Queue a copy of GPU g's error word to pinned host memory on the current stream (no synchronisation)."""
        self.err_host[g:g + 1].copy_(self.err[g], non_blocking=True)

    def check_polled(self) -> None:
        """Raise if a previous step's exchange hit the flag watchdog (values arrive with ``poll_async``)."""
        for g in range(self.n):
            v = int(self.err_host[g]) & 0xFFFFFFFF
            if v:
                raise RuntimeError(f"sequence-parallel exchange timed out on GPU {g}: 0x{v:08x} (dead or stalled peer)")

    def check_error(self) -> None:
        for g, e in enumerate(self.err):
            v = int(e.item()) & 0xFFFFFFFF
            if v:
                raise RuntimeError(f"sequence-parallel exchange timed out on GPU {g}: 0x{v:08x} (dead or stalled peer)")

    def release(self) -> None:
        self._ws.clear()


def build(executors, timeout_ms: int = 20000) -> "tuple[Optional[UlyssesBase], Optional[str]]":
    """(sequence-parallel driver, None) for a chain of native replicas, or (None, reason)."""
    fam = getattr(executors[0], "pa_family", None) if executors else None
    if fam == "flux":
        from . import flux_sp as mod
        cls = mod.FluxUlysses
    elif fam == "wan":
        from . import wan_sp as mod
        cls = mod.WanUlysses
    elif fam == "zimage":
        from . import zimage_sp as mod
        cls = mod.ZImageUlysses
    else:
        return None, "no sequence-parallel path for this model family"
    why = mod.supported(executors)
    if why:
        return None, why
    return cls(executors, timeout_ms=timeout_ms), None
