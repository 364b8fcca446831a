"""CUDA-graph cache shared by the native executors.

A denoise step is a static schedule of a few hundred to ~2 000 kernel launches over fixed buffers; replaying it as ONE
CUDA graph removes the per-launch host cost (what makes the reference's per-replica Python threads GIL-bound,
/root/reference/any_device_parallel.py:1390, 1414) and lets a native host thread (``csrc/runtime`` ``HostExecutor``) or a
GIL-free ``replay()`` drive each GPU.

Policy per key (= every pointer / shape the kernels bake in): 1st call eager (also warms lazily-built state), 2nd call
captured + replayed, later calls replayed.  A failed capture pins the key to eager.  Captures are serialised across
executors and use a per-executor capture stream (torch's default capture stream is a per-process singleton bound to the
first capturing device: capturing another GPU's step on it records nothing).
"""
from __future__ import annotations

import threading
from typing import Callable, Dict, Hashable, Optional

import torch

from ..utils import log

_CAPTURE_LOCK = threading.Lock()
_SEEN, _EAGER = "seen", "eager"


class GraphCache:
    def __init__(self, device, enabled: bool = True, limit: int = 32):
        self.device = torch.device(device)
        self.enabled = bool(enabled)
        self.limit = limit
        self._graphs: Dict[Hashable, object] = {}
        self._stream: Optional[torch.cuda.Stream] = None
        self.replays = 0
        self.captures = 0

    def __len__(self) -> int:
        return sum(1 for g in self._graphs.values() if not isinstance(g, str))

    def values(self):
        return self._graphs.values()

    def clear(self) -> None:
        self._graphs.clear()

    def captured(self, key) -> Optional["torch.cuda.CUDAGraph"]:
        g = self._graphs.get(key)
        return None if g is None or isinstance(g, str) else g

    def exec_handle(self, key) -> int:
        """Raw ``cudaGraphExec_t`` of a captured key (0 if not captured yet) for the native HostExecutor."""
        g = self.captured(key)
        if g is None:
            return 0
        try:
            return int(g.raw_cuda_graph_exec())
        except Exception:
            return 0

    def state(self, key) -> str:
        """'new' | 'seen' (ran eagerly once, next call captures) | 'eager' (capture failed) | 'graph'."""
        g = self._graphs.get(key)
        if g is None:
            return "new"
        return g if isinstance(g, str) else "graph"

    def capture_only(self, key, body: Callable[[], None]) -> bool:
        """Capture ``body`` for a key that already ran eagerly once, WITHOUT replaying it.  For step graphs whose kernels
        wait on other GPUs' flags (sequence-parallel exchanges): torch's capture prologue synchronises the device and
        empties the caching allocator (``cudaFree`` synchronises every device of the process), so capturing GPU B's graph
        while GPU A already replays a graph that spins on B's flags dead-locks until the flag watchdog fires.  The
        engine therefore captures all GPUs' graphs first, from one thread, and only then launches them."""
        if not self.enabled or self._graphs.get(key) != _SEEN:
            return self.captured(key) is not None
        return self._capture(key, body, eager_on_failure=False)

    def replay(self, key) -> None:
        g = self.captured(key)
        if g is None:
            raise KeyError("no captured graph for this key")
        g.replay()
        self.replays += 1

    def run(self, key, body: Callable[[], None]) -> None:
        if not self.enabled:
            body()
            return
        g = self._graphs.get(key)
        if g is None:
            body()
            if len(self._graphs) > self.limit:      # callers that pass fresh buffers every step never re-hit a key
                self._graphs = {k: v for k, v in self._graphs.items() if v != _SEEN}
            self._graphs[key] = _SEEN
        elif g == _SEEN:
            if self._capture(key, body, eager_on_failure=True):
                self.replay(key)
        elif g == _EAGER:
            body()
        else:
            g.replay()
            self.replays += 1

    def _capture(self, key, body: Callable[[], None], eager_on_failure: bool) -> bool:
        """Record ``body`` as the graph of ``key``.  A failed capture pins the key to eager and returns False, after
        running ``body`` eagerly once if ``eager_on_failure`` (never lose a step to a failed capture)."""
        # "thread_local" keeps other threads' CUDA calls legal while we record (the in-process engine drives one
        # executor per GPU from its own thread); the lock serialises captures, whose prologue synchronises.
        with _CAPTURE_LOCK:
            torch.cuda.synchronize(self.device)
            graph = torch.cuda.CUDAGraph()
            if self._stream is None:
                self._stream = torch.cuda.Stream(device=self.device)
            try:
                with torch.cuda.graph(graph, stream=self._stream, capture_error_mode="thread_local"):
                    body()
            except Exception as e:
                log.warn("CUDA graph capture failed on %s (%s); staying eager for this shape", self.device, e)
                torch.cuda.synchronize(self.device)
                self._graphs[key] = _EAGER
                if eager_on_failure:
                    body()
                return False
        self._graphs[key] = graph
        self.captures += 1
        return True
