"""The steps either side of the encoder (SURVEY.md 8f #1) on prepared weights: ``proj_encoder`` in front
(e2e_asr_conformer.py:31,70), the CTC head ``ctc_lo`` + log_softmax behind (ctc.py:21,77-93).

``PreparedHead`` owns the library-side copy of the two projections' weights (operand storage, ctc_lo padded), rebuilt
only when a parameter changes.  ``features_to_log_probs`` is the fused inference call a Lightning-free replay of
``ModelModule.forward`` / ``test_step`` (lightning.py:58,69-72) makes: one C-ABI entry from front-end features to CTC
log-probabilities (and the encoder features the attention decoder / beam search consume)."""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional, Tuple

import torch

from ._cabi import EncoderConfig, check, lib
from ._cache import PlanCache, WorkspacePool, capture
from .engine import PRECISIONS, EncoderEngine, _ptr, _stream_handle, default_precision, require_cuda


class PreparedHead:
    def __init__(self, d_model: int, n_heads: int = 12, linear_units: int = 3072, num_blocks: int = 12, cnn_kernel: int = 31):
        self.cfg = EncoderConfig(d_model, n_heads, linear_units, num_blocks, cnn_kernel)
        self._buf: Dict[tuple, Tuple[tuple, torch.Tensor]] = {}
        self.workspaces = WorkspacePool()
        # plans of features_to_log_probs: (plan, workspace, enc_out, logp, argmax)
        self.plans = PlanCache(lambda rec: lib.avsr_plan_destroy(rec[0]), EncoderEngine.GRAPH_AFTER, EncoderEngine.MAX_PLANS)

    @staticmethod
    def _fp(*tensors) -> tuple:
        return tuple((t.data_ptr(), t._version, tuple(t.shape)) for t in tensors if t is not None)

    def prepare(self, proj: Optional[torch.nn.Linear], ctc_lo: Optional[torch.nn.Linear], device, precision: str,
                idim: Optional[int] = None, odim: Optional[int] = None):
        """-> (buffer, idim, odim).  Either projection may be None (its half of the buffer is left empty)."""
        idim = proj.in_features if proj is not None else (idim or 8)
        odim = ctc_lo.out_features if ctc_lo is not None else (odim or 1)
        params = [p for m in (proj, ctc_lo) if m is not None for p in (m.weight, m.bias)]
        for p in params:
            require_cuda(p, "head parameter")
            if p.device != device:
                raise RuntimeError(f"head parameter lives on {p.device}, input on {device}")
        key = (device.index or 0, PRECISIONS[precision], idim, odim, proj is not None, ctc_lo is not None)
        fp = self._fp(*params)
        hit = self._buf.get(key)
        if hit is not None and hit[0] == fp:
            return hit[1], idim, odim
        nbytes = int(lib.avsr_head_prepared_bytes(C.byref(self.cfg), idim, odim))
        buf = torch.empty(nbytes, dtype=torch.uint8, device=device)
        keep = [p.detach().contiguous() for p in params]
        pw, pb = (keep[0], keep[1]) if proj is not None else (None, None)
        cw, cb = (keep[-2], keep[-1]) if ctc_lo is not None else (None, None)
        with torch.cuda.device(device):
            check(lib.avsr_prepare_head(C.byref(self.cfg), idim, odim, _ptr(pw), _ptr(pb), _ptr(cw), _ptr(cb),
                                        buf.data_ptr(), nbytes, PRECISIONS[precision], _stream_handle(device)))
        self._buf[key] = (fp, buf)
        self.plans.clear()                      # plans bake the prepared buffers' addresses
        return buf, idim, odim


def proj_forward(head: PreparedHead, proj: torch.nn.Linear, x: torch.Tensor, precision: str) -> torch.Tensor:
    """y = x W^T + b on the prepared weights (rows = all leading dims)."""
    require_cuda(x, "proj_encoder input")
    x = x.detach().contiguous()
    buf, idim, odim = head.prepare(proj, None, x.device, precision)
    rows = x.numel() // idim
    y = torch.empty(*x.shape[:-1], head.cfg.d_model, dtype=torch.float32, device=x.device)
    ws = head.workspaces.get("proj", rows * idim * 4 + 256, x.device, _stream_handle(x.device))
    with torch.cuda.device(x.device):
        check(lib.avsr_proj_encoder(C.byref(head.cfg), buf.data_ptr(), x.data_ptr(), rows, idim, odim, y.data_ptr(),
                                    ws.data_ptr(), ws.numel(), PRECISIONS[precision], _stream_handle(x.device)))
    return y


def ctc_log_probs(head: PreparedHead, ctc_lo: torch.nn.Linear, hs: torch.Tensor, precision: str, want_logp: bool = True,
                  want_argmax: bool = False):
    """log_softmax(ctc_lo(hs)) (…, odim) and / or the greedy ids (…) on the prepared, padded weights."""
    require_cuda(hs, "CTC input")
    hs = hs.detach().contiguous()
    buf, idim, odim = head.prepare(None, ctc_lo, hs.device, precision)
    rows = hs.numel() // head.cfg.d_model
    logp = torch.empty(*hs.shape[:-1], odim, dtype=torch.float32, device=hs.device) if want_logp else None
    best = torch.empty(hs.shape[:-1], dtype=torch.int32, device=hs.device) if want_argmax else None
    nbytes = int(lib.avsr_ctc_workspace_bytes(C.byref(head.cfg), rows, odim))
    ws = head.workspaces.get("ctc", nbytes, hs.device, _stream_handle(hs.device))
    with torch.cuda.device(hs.device):
        check(lib.avsr_ctc_logprobs(C.byref(head.cfg), buf.data_ptr(), hs.data_ptr(), rows, idim, odim, _ptr(logp),
                                    _ptr(best), ws.data_ptr(), ws.numel(), PRECISIONS[precision], _stream_handle(hs.device)))
    return logp, (None if best is None else best.long())


def features_to_log_probs(proj: torch.nn.Linear, encoder, ctc, feats: torch.Tensor, masks: Optional[torch.Tensor] = None,
                          want_features: bool = True, want_argmax: bool = False, precision: Optional[str] = None):
    """Front-end features (B, T, idim) -> (encoder features (B, T, d) | None, CTC log-probs (B, T, odim), ids | None).

    ``proj`` is E2E.proj_encoder, ``encoder`` the drop-in ConformerEncoder, ``ctc`` E2E.ctc (anything with a ``ctc_lo``
    Linear): the reference's inference path e2e_asr_conformer.py:70-71 + ctc.py:77-84 in ONE library call --
    proj_encoder writes sqrt(d)-scaled rows straight into the residual stream, after_norm emits ctc_lo's operand, the
    ctc_lo GEMM leaves log-sum-exp partials for a single finishing pass.  A (B, T) shape that keeps coming back is replayed
    from a CUDA graph (``encoder.use_graph`` / ``graph_after``): then the returned tensors belong to the plan and are
    overwritten by the next call with that shape -- clone them to keep them."""
    from .espnet_dropin.attention import mask_to_lengths
    if encoder.training:
        raise NotImplementedError("features_to_log_probs: inference only (call .eval())")
    require_cuda(feats, "features")
    if feats.dim() != 3 or feats.size(2) != proj.in_features:
        raise ValueError(f"features must be (B, T, {proj.in_features}), got {tuple(feats.shape)}")
    precision = precision or encoder.precision or default_precision()
    B, T, _ = feats.shape
    dev = feats.device
    feats = feats.detach().contiguous()
    torch.empty(len(encoder.encoders)).uniform_()          # the CPU uniforms MultiSequential draws per call (repeat.py:23)
    lengths = None if masks is None else mask_to_lengths(masks, B, T, check=getattr(encoder, "check_mask", False))
    prepared = encoder._prepared(dev, precision)
    head = getattr(encoder, "_fused_head", None)
    if head is None:
        head = encoder._fused_head = PreparedHead(*encoder._cfg)
    hbuf, idim, odim = head.prepare(proj, ctc.ctc_lo, dev, precision)
    st = _stream_handle(dev)
    if B and T and encoder.use_graph and not getattr(encoder, "check_saturation", False):
        # CUDA-graph replay under the encoder's shape policy and threshold.  The plan owns its output tensors: the ones
        # returned here are overwritten by the next call with this shape.
        def build():
            nbytes = int(lib.avsr_head_plan_workspace_bytes(C.byref(head.cfg), B, T, idim, odim))
            ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
            eo = torch.empty(B, T, head.cfg.d_model, dtype=torch.float32, device=dev) if want_features else None
            lp = torch.empty(B, T, odim, dtype=torch.float32, device=dev)
            am = torch.empty(B, T, dtype=torch.int32, device=dev) if want_argmax else None
            plan = C.c_void_p()
            capture(dev, lambda cs: check(lib.avsr_head_plan_create(
                C.byref(head.cfg), prepared.data_ptr(), hbuf.data_ptr(), B, T, idim, odim, _ptr(eo), lp.data_ptr(),
                _ptr(am), ws.data_ptr(), nbytes, PRECISIONS[precision], cs, C.byref(plan))))
            return plan, ws, eo, lp, am
        head.plans.graph_after = encoder._engine.graph_after
        rec = head.plans.get((dev.index or 0, B, T, idim, odim, PRECISIONS[precision], prepared.data_ptr(),
                              hbuf.data_ptr(), st, want_features, want_argmax), build)
        if rec is not None:
            plan, _ws, eo, lp, am = rec
            with torch.cuda.device(dev):
                check(lib.avsr_head_plan_forward(plan, feats.data_ptr(), _ptr(lengths), st))
            return eo, lp, (None if am is None else am.long())
    enc_out = torch.empty(B, T, head.cfg.d_model, dtype=torch.float32, device=dev) if want_features else None
    logp = torch.empty(B, T, odim, dtype=torch.float32, device=dev)
    best = torch.empty(B, T, dtype=torch.int32, device=dev) if want_argmax else None
    if B and T:
        nbytes = int(lib.avsr_head_workspace_bytes(C.byref(head.cfg), B, T, idim, odim))
        ws = head.workspaces.get("fused", nbytes, dev, st)
        with torch.cuda.device(dev):
            check(lib.avsr_features_to_logprobs(C.byref(head.cfg), prepared.data_ptr(), hbuf.data_ptr(), feats.data_ptr(),
                                                _ptr(lengths), B, T, idim, odim, _ptr(enc_out), logp.data_ptr(),
                                                _ptr(best), ws.data_ptr(), ws.numel(), PRECISIONS[precision], st))
    return enc_out, logp, (None if best is None else best.long())
