"""Host-side state the C ABI leaves to its caller: the CUDA-graph plan cache behind the shape policy (DESIGN.md
section 1), the capture stream and grow-only workspaces.  torch only, so the policy is testable without a GPU."""
from collections import OrderedDict
from typing import Callable, Dict, Optional

import torch


class PlanCache:
    """``get(key, build)`` returns None until ``key`` has been seen ``graph_after`` times, then the record ``build()``
    made once.  At most ``max_plans`` records live, in LRU order; each evicted or cleared record goes to ``destroy``
    exactly once.  Only the ``64 * max_plans`` most recent keys keep their sightings (one-off shapes cannot grow it)."""

    def __init__(self, destroy: Callable[[object], None], graph_after: int, max_plans: int):
        self.destroy, self.graph_after, self.max_plans = destroy, graph_after, max_plans
        self._plans: "OrderedDict[tuple, object]" = OrderedDict()
        self._seen: "OrderedDict[tuple, int]" = OrderedDict()

    def __len__(self) -> int:
        return len(self._plans)

    def get(self, key: tuple, build: Callable[[], object]) -> Optional[object]:
        rec = self._plans.get(key)
        if rec is not None:
            self._plans.move_to_end(key)
            return rec
        seen = self._seen[key] = self._seen.pop(key, 0) + 1          # re-inserted: the most recent key is last
        while len(self._seen) > 64 * self.max_plans:
            self._seen.popitem(last=False)
        if seen < self.graph_after:
            return None
        rec = self._plans[key] = build()
        while len(self._plans) > self.max_plans:
            self.destroy(self._plans.popitem(last=False)[1])
        return rec

    def clear(self) -> None:
        while self._plans:
            self.destroy(self._plans.popitem(last=False)[1])

    def __del__(self):
        try:
            self.clear()
        except Exception:                  # interpreter shutdown: the library may be unloaded already
            pass


_capture_streams: Dict[int, torch.cuda.Stream] = {}


def capture(device: torch.device, create: Callable[[int], None]) -> None:
    """Runs ``create(stream)`` on the device's capture stream (the legacy default stream cannot capture), after the
    work queued on the current stream, and waits for it."""
    with torch.cuda.device(device):
        cs = _capture_streams.get(device.index or 0)
        if cs is None:
            cs = _capture_streams[device.index or 0] = torch.cuda.Stream(device=device)
        cs.wait_stream(torch.cuda.current_stream(device))
        create(cs.cuda_stream)
        cs.synchronize()


class WorkspacePool:
    """One grow-only byte buffer per (tag, device, stream).  The library carves a workspace's layout per call and calls
    on one stream run in order, so a buffer that is large enough serves every shape.  It regrows with 25 % + 1 KB slack."""

    def __init__(self):
        self._bufs: Dict[tuple, torch.Tensor] = {}

    def __len__(self) -> int:
        return len(self._bufs)

    def get(self, tag: str, nbytes: int, device: torch.device, stream: int) -> torch.Tensor:
        key = (tag, device.index or 0, stream)
        ws = self._bufs.get(key)
        if ws is None or ws.numel() < nbytes:
            ws = self._bufs[key] = torch.empty(nbytes + nbytes // 4 + 1024, dtype=torch.uint8, device=device)
        return ws
