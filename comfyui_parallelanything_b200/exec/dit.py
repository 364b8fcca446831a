"""Host-side plumbing shared by the native DiT executors (FLUX, WAN, Z-Image).

The families differ in their weight packing, workspace geometry and kernel schedule (``_run``).  What surrounds the
schedule is the same for all of them and lives here: the workspace LRU, the step entry points with their CUDA-graph
keys, the eagerly cached conditioning path (``_prepare_ctx``, WAN and Z-Image), the modulation-table slices, the
fp32 RoPE-table layout and the head GEMM that unpatchifies, applies the Euler update and stores into a (peer) buffer.
"""
from __future__ import annotations

from typing import Dict, Optional, Tuple

import torch
import torch.nn as nn

from .. import ops
from . import cache_workspace, conditioning_sig, recognize, touch_workspace
from .graphs import GraphCache


def rope_layout(pe: torch.Tensor) -> torch.Tensor:
    """``EmbedND`` output [1, 1, L, 64, 2, 2] -> the fp32 [L, 64, 2] (cos, sin) table the QKV-RoPE epilogue and the
    ``rms_rope`` kernel read."""
    return torch.stack([pe[0, 0, :, :, 0, 0], pe[0, 0, :, :, 1, 0]], -1).float().contiguous()


def head_gather(a, w, b, C: int, Hl: int, Wl: int, out=None, out_ptr: Optional[int] = None, out_sample_off: int = 0,
                x_in=None, sigmas=None, tok_off: int = 0, xin_bstride: int = 0) -> None:
    """Head GEMM with the unpatchify epilogue: token rows -> [B, C, Hl, Wl] latent, written to ``out`` or through
    ``out_ptr`` (e.g. the lead GPU's buffer) at sample ``out_sample_off``.  With ``sigmas`` the epilogue applies the
    Euler update ``x_in + (sigma_next - sigma) * v``.  ``tok_off``: first token of ``a`` (a sequence-parallel slice).
    ``xin_bstride``: elements per sample of ``x_in`` when it is wider than the output (0: ``C*Hl*Wl``); the update then
    reads its first ``C`` channels."""
    kw = dict(bias=b, C=C, Hl=Hl, Wl=Wl, xout_sample_off=out_sample_off, tok_off=tok_off)
    if out_ptr is not None:
        kw["x_out_ptr"] = out_ptr
    else:
        kw["x_out"] = out
    if sigmas is not None:
        kw["sigmas"], kw["x_in"] = sigmas, x_in
        if xin_bstride:
            kw["xin_bstride"] = xin_bstride
    ops.gemm(a, w, "euler_unpatch", **kw)


def _step_bf16(t: torch.Tensor, device) -> torch.Tensor:
    return t.to(device=device, dtype=torch.bfloat16).contiguous()


def _ptrs(tensors) -> tuple:
    return tuple(0 if t is None else t.data_ptr() for t in tensors)


class DiTExecutor(nn.Module):
    """Base of the DiT executors.  A family sets ``pa_family``, packs ``W`` and provides ``_new_workspace(*geometry)``
    (geometry = batch, the latent's spatial / temporal sizes, text length), ``rope`` and ``_run(ws, x_ptr, *inputs,
    out, ...)``.  ``inputs`` are timesteps and context, plus whatever ``_inputs`` adds (FLUX: ``y``, ``guidance``)."""

    pa_family = "?"
    pa_native = True
    fused_embed = True          # the first kernel pulls the latent itself and leaves a local copy in ``x``
    _prepare_ctx = None         # conditioning-only work (WAN, Z-Image): run eagerly, cached per workspace by ``ctx_sig``

    def __init__(self, model: nn.Module, device, cuda_graphs: bool):
        super().__init__()
        ops.require()
        self.device = torch.device(device)
        # hyper-parameters come from the module's STRUCTURE (weight shapes, ComfyUI attribute names), so a ComfyUI model
        # is packed exactly like the repository's own oracle class
        self.params = recognize.params_of(model, self.pa_family)
        self.cuda_graphs = cuda_graphs
        self._ws: Dict[Tuple, dict] = {}
        self._graphs = GraphCache(self.device, enabled=cuda_graphs)
        self.launches_per_step = 0

    # nn.Module plumbing so engine utilities (module_device, .to("meta") on cleanup) work
    def parameters(self, recurse: bool = True):  # type: ignore[override]
        return iter(())

    def release(self) -> None:
        self.W.clear()
        self._ws.clear()
        self._graphs.clear()

    def weight_bytes(self) -> int:
        return sum(t.numel() * t.element_size() for t in self.W.values() if isinstance(t, torch.Tensor))

    def invalidate_conditioning(self) -> None:
        """Forget the cached conditioning-only results (call when the prompt buffer is rewritten in place)."""
        for ws in self._ws.values():
            ws["ctx_sig"] = None

    # ------------------------------------------------------------------ workspaces
    def workspace(self, *geometry) -> dict:
        """Activation buffers for one geometry.  The least recently used one is dropped beyond ``WORKSPACE_LIMIT``,
        together with the captured graphs, which point into it."""
        ws = touch_workspace(self._ws, geometry)
        if ws is None:
            ws = cache_workspace(self._ws, geometry, self._new_workspace(*geometry), device=self.device,
                                 on_evict=lambda _k: self._graphs.clear())
        return ws

    def out_shape(self, shape) -> Tuple[int, ...]:
        """Shape of the model output for an input latent of ``shape`` (the same, unless a family says otherwise)."""
        return tuple(shape)

    @staticmethod
    def _geometry(shape, context) -> tuple:
        return (shape[0],) + tuple(shape[2:]) + (context.shape[1],)

    def _geometry_of(self, shape, inputs: tuple) -> tuple:
        """Workspace geometry of a step with latent ``shape`` and step inputs ``inputs`` (timesteps first)."""
        return self._geometry(shape, *self._conditioning(inputs))

    @staticmethod
    def _conditioning(inputs: tuple) -> tuple:
        """The step inputs that ``_geometry``, ``_prepare_ctx`` and ``_cond_sig`` take: the context (WAN with CLIP image
        conditioning adds ``clip_fea``)."""
        return inputs[1:2]

    @staticmethod
    def _cond_sig(context) -> tuple:
        """What ``_prepare_ctx`` stores in ``ws["ctx_sig"]`` for this conditioning."""
        return conditioning_sig(context)

    def _mod(self, ws, key, idx: int):
        """``idx``-th modulation vector of block ``key`` in the step's modulation table (each is as wide as ``X``)."""
        width = ws["X"].shape[-1]
        off = self.mod_off[key] + idx * width
        return ws["MOD"][:, off:off + width]

    # ------------------------------------------------------------------ step inputs
    def _inputs(self, B: int, timesteps, context) -> tuple:
        """The step inputs other than the latent, as bf16 on this executor's device."""
        return _step_bf16(timesteps, self.device), _step_bf16(context, self.device)

    def _prep(self, x, timesteps, context):
        return (_step_bf16(x, self.device),) + self._inputs(x.shape[0], timesteps, context)

    def _shard_args(self, x_src_ptr: int, shape, out_ptr: int, out_sample_off: int, *step_inputs):
        inputs = self._inputs(shape[0], *step_inputs)
        key = (("shard", tuple(shape), tuple(inputs[1].shape), x_src_ptr, out_ptr, out_sample_off) + _ptrs(inputs)
               + (tuple(inputs[0].shape),))
        return key, inputs

    # ------------------------------------------------------------------ step entry points
    def _forward(self, x, *step_inputs):
        with torch.cuda.device(self.device):
            x, *inputs = self._prep(x, *step_inputs)
            ws = self.workspace(*self._geometry_of(x.shape, inputs))
            out = torch.empty(self.out_shape(tuple(x.shape)), dtype=x.dtype, device=x.device)
            if self._prepare_ctx is not None:
                self._prepare_ctx(ws, *self._conditioning(inputs))
            self._run(ws, x.data_ptr(), *inputs, out)
            return out

    def _forward_shard(self, x_src_ptr: int, shape, out_ptr: int, out_sample_off: int, *step_inputs) -> None:
        with torch.cuda.device(self.device):
            key, inputs = self._shard_args(x_src_ptr, shape, out_ptr, out_sample_off, *step_inputs)
            ws = self.workspace(*self._geometry_of(shape, inputs))
            if self._prepare_ctx is not None:
                self._prepare_ctx(ws, *self._conditioning(inputs))
            self._graphs.run(key, lambda: self._run(ws, x_src_ptr, *inputs, None, out_ptr=out_ptr,
                                                    out_sample_off=out_sample_off))

    def _graph_handle(self, x_src_ptr: int, shape, out_ptr: int, out_sample_off: int, *step_inputs) -> int:
        with torch.cuda.device(self.device):
            key, inputs = self._shard_args(x_src_ptr, shape, out_ptr, out_sample_off, *step_inputs)
            if self._prepare_ctx is not None:
                ws = self.workspace(*self._geometry_of(shape, inputs))
                if ws["ctx_sig"] != self._cond_sig(*self._conditioning(inputs)):
                    return 0                # conditioning changed: take the Python path once (eager precompute)
        return self._graphs.exec_handle(key)

    def _denoise(self, x, inputs: tuple, sigmas, out, out_ptr, out_sample_off, x_src_ptr, t_src_ptr, **src_ptrs):
        """``src_ptrs``: peer pointers of family-specific per-sample inputs, passed on to ``_run`` (FLUX: ``g_ptr``)."""
        with torch.cuda.device(self.device):
            ws = self.workspace(*self._geometry_of(x.shape, inputs))
            if out is None and out_ptr is None:
                out = ws["OUT"]
            if self._prepare_ctx is not None:
                self._prepare_ctx(ws, *self._conditioning(inputs))

            def body():
                self._run(ws, x_src_ptr if x_src_ptr is not None else x.data_ptr(), *inputs, out, x_in=x, sigmas=sigmas,
                          out_ptr=out_ptr, out_sample_off=out_sample_off, t_ptr=t_src_ptr,
                          x_copy=x if (x_src_ptr is not None and self.fused_embed) else None, **src_ptrs)

            key = ((tuple(x.shape), tuple(inputs[1].shape), out_ptr or 0, out_sample_off, x_src_ptr or 0, t_src_ptr or 0)
                   + tuple(p or 0 for p in src_ptrs.values()) + _ptrs((x, sigmas, out) + tuple(inputs))
                   + (tuple(inputs[0].shape),))
            self._graphs.run(key, body)
            return out

    @torch.no_grad()
    def forward_shard(self, x_src_ptr: int, shape, timesteps, context, out_ptr: int, out_sample_off: int, **_ignored):
        """In-process multi-GPU path: pull this replica's latent shard from the lead GPU's tensor (peer
        pointer) inside the first kernel and store the velocity rows straight into the lead's output.
        The engine stages every tensor argument into fixed device buffers, so the key (= all baked pointers) repeats
        from step to step and the step replays as one CUDA graph."""
        self._forward_shard(x_src_ptr, shape, out_ptr, out_sample_off, timesteps, context)

    def shard_graph_handle(self, x_src_ptr: int, shape, timesteps, context, out_ptr: int, out_sample_off: int,
                           **_ignored) -> int:
        """``cudaGraphExec_t`` of the captured step for exactly these buffers (0 = not captured yet, or the conditioning
        changed): lets the engine hand the replay to a native host thread instead of calling ``forward_shard``."""
        return self._graph_handle(x_src_ptr, shape, out_ptr, out_sample_off, timesteps, context)

    @torch.no_grad()
    def denoise_step(self, x, timesteps, context, sigmas, out=None, out_ptr=None, out_sample_off=0,
                     x_src_ptr: Optional[int] = None, t_src_ptr: Optional[int] = None):
        """Model forward + Euler update ``x + (sigma_next - sigma) * v`` fused into the last GEMM's
        epilogue; the result may be stored straight into a peer GPU's buffer (``out_ptr``).
        ``x_src_ptr`` / ``t_src_ptr`` let the first kernel pull the latent shard and the timesteps from a peer mapping
        (then ``x`` is filled with a local copy as a side effect)."""
        return self._denoise(x, (timesteps, context), sigmas, out, out_ptr, out_sample_off, x_src_ptr, t_src_ptr)
