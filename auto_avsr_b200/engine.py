"""Host-side driver of the C-ABI encoder: owns the prepared-weight buffer, per-(B,T) workspaces and CUDA-graph
plans.  torch is used for device memory and streams only; all arithmetic happens in libavsr_b200.so."""
from __future__ import annotations

import ctypes as C
import os
from typing import Dict, Optional, Tuple

import torch

from . import _cabi
from ._cache import PlanCache, WorkspacePool, capture
from ._cabi import EncoderConfig, LayerParams, LAYER_FIELDS, PREC_F16, PREC_FP32, PREC_TF32, check, lib

PRECISIONS = {"fp32": PREC_FP32, "tf32": PREC_TF32, "f16": PREC_F16}


def default_precision() -> str:
    return os.environ.get("AVSR_B200_PRECISION", "f16")


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _stream_handle(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def require_cuda(t: torch.Tensor, what: str) -> None:
    if not t.is_cuda:
        raise RuntimeError(
            f"{what}: tensor is on {t.device}; the B200 encoder path has no CPU fallback "
            "(move the module and its inputs to a CUDA device)")
    if t.dtype != torch.float32:
        raise TypeError(f"{what}: expected float32, got {t.dtype}")


class SaturationError(OverflowError):
    """The fp16 operand path left its range (+-65504) for these weights / inputs: use precision "tf32" or "fp32"."""


class EncoderEngine:
    """Runs ConformerEncoder.forward (eval) for one parameter set on one device.

    Shape policy (the reference's eval path feeds B=1 with a different T per utterance, lightning.py:72): a (B, T)
    shape runs on direct launches -- one grow-only workspace per (device, stream), no capture cost -- until it has been
    seen ``graph_after`` times; only then a CUDA-graph plan (own ~85 KB/frame workspace, ~190-node capture) is built for
    it.  ``plans`` keeps at most ``MAX_PLANS`` (env AVSR_B200_MAX_PLANS) in LRU order.  Fixed-shape loops (training
    buckets, bench) reach the graph after ``graph_after - 1`` calls; ``graph_after=1`` captures at first sight."""

    MAX_PLANS = int(os.environ.get("AVSR_B200_MAX_PLANS", "16"))
    GRAPH_AFTER = int(os.environ.get("AVSR_B200_GRAPH_AFTER", "3"))

    def __init__(self, d_model: int, n_heads: int, linear_units: int, num_blocks: int, cnn_kernel: int):
        self.cfg = EncoderConfig(d_model, n_heads, linear_units, num_blocks, cnn_kernel)
        need = lib.avsr_prepared_bytes(C.byref(self.cfg))
        if need == 0:
            check(_cabi.E_INVALID)
        self.prepared_bytes = need
        self._prepared: Dict[Tuple[int, int], torch.Tensor] = {}      # (device index, precision) -> buffer
        self._workspaces = WorkspacePool()
        self.plans = PlanCache(lambda rec: lib.avsr_plan_destroy(rec[0]), self.GRAPH_AFTER, self.MAX_PLANS)
        self._sat: Dict[int, torch.Tensor] = {}
        self.stats = {"direct": 0, "graph": 0, "plans_built": 0}

    @property
    def graph_after(self) -> int:
        return self.plans.graph_after

    @graph_after.setter
    def graph_after(self, n: int) -> None:
        self.plans.graph_after = n

    # ---- weights -------------------------------------------------------------------------------
    def invalidate(self) -> None:
        """Forget prepared weights (and the plans that bake their addresses)."""
        self.plans.clear()
        self._prepared.clear()

    def prepare(self, state, device: torch.device, precision: str) -> torch.Tensor:
        """state: reference-keyed tensors ('encoders.{l}.<suffix>', 'after_norm.*') living on `device`, or a
        callable returning them (only called when the prepared copy for (device, precision) is missing)."""
        key = (device.index or 0, PRECISIONS[precision])
        buf = self._prepared.get(key)
        if buf is not None:
            return buf
        if callable(state):
            state = state()
        L = self.cfg.num_blocks
        arr = (LayerParams * L)()
        keep = []
        for l in range(L):
            for field, suffix in LAYER_FIELDS:
                t = state[f"encoders.{l}.{suffix}"]
                require_cuda(t, suffix)
                if t.device != device:
                    raise RuntimeError(f"encoder parameter {suffix} (layer {l}) lives on {t.device} but the input is on "
                                       f"{device}: move the module with .to(device) first")
                t = t.detach().contiguous()
                keep.append(t)
                setattr(arr[l], field, t.data_ptr())
        aw = state["after_norm.weight"].detach().contiguous()
        ab = state["after_norm.bias"].detach().contiguous()
        buf = torch.empty(self.prepared_bytes, dtype=torch.uint8, device=device)
        with torch.cuda.device(device):
            check(lib.avsr_prepare_weights(C.byref(self.cfg), arr, aw.data_ptr(), ab.data_ptr(), buf.data_ptr(),
                                           self.prepared_bytes, PRECISIONS[precision], _stream_handle(device)))
        self._prepared[key] = buf
        return buf

    # ---- forward -------------------------------------------------------------------------------
    def forward(self, prepared: torch.Tensor, xs: torch.Tensor, lengths: Optional[torch.Tensor], precision: str,
                use_graph: bool = True, taps: Optional[torch.Tensor] = None, check_saturation: bool = False) -> torch.Tensor:
        require_cuda(xs, "xs")
        if xs.dim() != 3 or xs.size(2) != self.cfg.d_model:
            raise ValueError(f"xs must be (B, T, {self.cfg.d_model}), got {tuple(xs.shape)}")
        B, T, D = xs.shape
        device = xs.device
        xs = xs.contiguous()
        out = torch.empty_like(xs)
        if B == 0 or T == 0:
            return out
        if lengths is not None:
            if lengths.device != device or lengths.dtype != torch.int32 or lengths.numel() != B:
                raise ValueError("lengths must be an int32 tensor of B elements on the input's device")
            lengths = lengths.contiguous()
        prec = PRECISIONS[precision]
        with torch.cuda.device(device):
            st = _stream_handle(device)
            rec = None
            if use_graph and taps is None and not check_saturation:
                rec = self.plans.get((device.index or 0, B, T, prec, prepared.data_ptr(), st),
                                     lambda: self._build_plan(prepared, B, T, device, prec))
            if rec is not None:
                self.stats["graph"] += 1
                check(lib.avsr_plan_forward(rec[0], xs.data_ptr(), _ptr(lengths), out.data_ptr(), st))
            else:
                self.stats["direct"] += 1
                ws = self._workspaces.get("direct", int(lib.avsr_workspace_bytes(C.byref(self.cfg), B, T)), device, st)
                if check_saturation:
                    cnt = self._sat.get(device.index or 0)
                    if cnt is None:
                        cnt = self._sat[device.index or 0] = torch.zeros(1, dtype=torch.int64, device=device)
                    check(lib.avsr_encoder_forward_checked(C.byref(self.cfg), prepared.data_ptr(), xs.data_ptr(),
                                                           _ptr(lengths), B, T, out.data_ptr(), ws.data_ptr(),
                                                           ws.numel(), prec, cnt.data_ptr(), st))
                    n = int(cnt.item())                      # host sync: this is the diagnostic path
                    if n:
                        raise SaturationError(
                            f"{n} fp16 operand value(s) saturated at +-65504 (or NaN) in this forward: the f16 path "
                            "is outside its range for these weights / inputs -- use precision='tf32' or 'fp32'")
                elif taps is None:
                    check(lib.avsr_encoder_forward(C.byref(self.cfg), prepared.data_ptr(), xs.data_ptr(), _ptr(lengths),
                                                   B, T, out.data_ptr(), ws.data_ptr(), ws.numel(), prec, st))
                else:
                    check(lib.avsr_encoder_forward_taps(C.byref(self.cfg), prepared.data_ptr(), xs.data_ptr(),
                                                        _ptr(lengths), B, T, out.data_ptr(), taps.data_ptr(),
                                                        ws.data_ptr(), ws.numel(), prec, st))
        return out

    def _build_plan(self, prepared: torch.Tensor, B: int, T: int, device: torch.device, prec: int) -> tuple:
        """(plan, its workspace) for one shape.  The workspace is private to the plan, so to the stream in its key."""
        self.stats["plans_built"] += 1
        ws = torch.empty(int(lib.avsr_workspace_bytes(C.byref(self.cfg), B, T)), dtype=torch.uint8, device=device)
        plan = C.c_void_p()
        capture(device, lambda cs: check(lib.avsr_plan_create(C.byref(self.cfg), prepared.data_ptr(), B, T, ws.data_ptr(),
                                                               ws.numel(), prec, cs, C.byref(plan))))
        return plan, ws
