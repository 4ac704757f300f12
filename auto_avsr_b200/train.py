"""Training slice of the encoder path (SURVEY.md 8f #2, first slice): ``torch.autograd.Function``s whose forward AND
backward run in libavsr_b200 -- LayerNorm, Linear (+ReLU) with dgrad / wgrad as the same tcgen05 GEMMs on transposed
operands, GLU, and the depthwise-conv + BatchNorm(batch statistics) + SiLU block.  Gradients land on the original
``nn.Parameter``s (autograd accumulates what ``backward`` returns), so DDP hooks, ``clip_grad_norm_`` and AdamW
(lightning.py:49, train.py:37-41) see them unchanged.  torch supplies device memory, the autograd tape, dropout masks
and the residual adds; no module falls back to PyTorch arithmetic for its own forward or backward.

The rel-pos attention core has a (correctness-first, fp32 CUDA-core) backward too, so a whole ``EncoderLayer`` /
``ConformerEncoder`` runs ``train()``: the reference's layer schedule with its dropouts (conformer_encoder.py:96-170).
SyncBatchNorm (train.py:31) is honoured: the per-channel sums are all-reduced between the library's passes.
Not built: dropout on attention probabilities (the reference trains with 0.0).

Backward GEMMs run with TF32 operands (fp32 range: gradients do not fit fp16's) unless ``precision="fp32"``."""
from __future__ import annotations

import ctypes as C
from typing import Optional

import torch

from . import ops
from ._cabi import check, lib
from ._cache import WorkspacePool
from .engine import _ptr, _stream_handle, require_cuda

_pool = WorkspacePool()


def _c(t: torch.Tensor) -> torch.Tensor:
    return t.detach().contiguous()


def bwd_precision(precision: str) -> str:
    return "fp32" if precision == "fp32" else "tf32"


# ------------------------------------------------------------------------------------------------ raw ops
def layernorm_bwd(x, gamma, dy):
    x, gamma, dy = _c(x), _c(gamma), _c(dy)
    d = x.size(-1)
    rows = x.numel() // d
    dx, dg, db = torch.empty_like(x), torch.empty_like(gamma), torch.empty_like(gamma)
    ws = _pool.get("train", int(lib.avsr_train_workspace_bytes(rows, d, 1)), x.device, _stream_handle(x.device))
    with torch.cuda.device(x.device):
        check(lib.avsr_layernorm_bwd(x.data_ptr(), gamma.data_ptr(), dy.data_ptr(), dx.data_ptr(), dg.data_ptr(), db.data_ptr(),
                                     rows, d, ws.data_ptr(), ws.numel(), _stream_handle(x.device)))
    return dx, dg, db


def colsum(y):
    y = _c(y)
    cols = y.size(-1)
    rows = y.numel() // cols
    out = torch.empty(cols, dtype=torch.float32, device=y.device)
    ws = _pool.get("train", 148 * cols * 4 + 1024, y.device, _stream_handle(y.device))
    with torch.cuda.device(y.device):
        check(lib.avsr_colsum(y.data_ptr(), out.data_ptr(), rows, cols, ws.data_ptr(), ws.numel(), _stream_handle(y.device)))
    return out


def transpose_padded(x2d, pad_to: int = 32):
    """(rows, cols) fp32 -> (cols, rows_padded) with zero padding of the new inner dim to a multiple of ``pad_to`` (the
    tensor-core GEMMs take K in 128-byte blocks)."""
    x2d = _c(x2d)
    rows, cols = x2d.shape
    ld = (rows + pad_to - 1) // pad_to * pad_to
    out = torch.zeros(cols, ld, dtype=torch.float32, device=x2d.device) if ld != rows else \
        torch.empty(cols, ld, dtype=torch.float32, device=x2d.device)
    with torch.cuda.device(x2d.device):
        check(lib.avsr_transpose(x2d.data_ptr(), out.data_ptr(), rows, cols, ld, _stream_handle(x2d.device)))
    return out


def relu_bwd(y, dy):
    y, dy = _c(y), _c(dy)
    dx = torch.empty_like(dy)
    with torch.cuda.device(y.device):
        check(lib.avsr_relu_bwd(y.data_ptr(), dy.data_ptr(), dx.data_ptr(), y.numel(), _stream_handle(y.device)))
    return dx


# ------------------------------------------------------------------------------------------------ autograd functions
class LayerNormFn(torch.autograd.Function):
    """LayerNorm(d, eps 1e-12) (layer_norm.py:21)."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        require_cuda(x, "LayerNorm input")
        ctx.save_for_backward(x, weight)
        return ops.layernorm(x, weight, bias)

    @staticmethod
    def backward(ctx, dy):
        x, weight = ctx.saved_tensors
        dx, dg, db = layernorm_bwd(x, weight, dy)
        return dx, dg, db


class LinearFn(torch.autograd.Function):
    """y = act(x W^T + b), act = identity | ReLU (positionwise_feed_forward.py:28-30, the pointwise convs of
    conformer_encoder.py:31,35).  Backward: dX = dY W and dW = dY^T X through the same GEMM entry on transposed operands,
    db = column sums of dY."""

    @staticmethod
    def forward(ctx, x, weight, bias, relu: bool, precision: str):
        require_cuda(x, "Linear input")
        w2 = weight.reshape(weight.size(0), -1)          # Conv1d(k=1) weights carry a trailing 1
        y = ops.linear(x, w2, bias, relu=relu, precision=precision)
        ctx.relu, ctx.precision, ctx.wshape = relu, precision, weight.shape
        ctx.save_for_backward(x, w2, y if relu else None)
        ctx.has_bias = bias is not None
        return y

    @staticmethod
    def backward(ctx, dy):
        x, w2, y = ctx.saved_tensors
        prec = bwd_precision(ctx.precision)
        dy = _c(dy)
        if ctx.relu:
            dy = relu_bwd(y, dy)
        n, k = w2.shape
        dy2, x2 = dy.reshape(-1, n), _c(x).reshape(-1, k)
        dx = dw = db = None
        if ctx.needs_input_grad[0]:
            wt = transpose_padded(w2, 32)                               # (k, n_padded): dX = dY W = dY (W^T)^T
            dyp = dy2
            if wt.size(1) != n:                                         # pad dY's columns like W^T's (zeros contribute 0)
                dyp = torch.zeros(dy2.size(0), wt.size(1), dtype=torch.float32, device=dy.device)
                dyp[:, :n] = dy2
            dx = ops.linear(dyp, wt, None, precision=prec).reshape(x.shape)
        if ctx.needs_input_grad[1]:
            dyt, xt = transpose_padded(dy2, 32), transpose_padded(x2, 32)   # (n, rows_p), (k, rows_p)
            dw = ops.linear(dyt, xt, None, precision=prec).reshape(ctx.wshape)
        if ctx.has_bias and ctx.needs_input_grad[2]:
            db = colsum(dy2)
        return dx, dw, db, None, None


class GluFn(torch.autograd.Function):
    """F.glu(x, dim=-1) on (…, 2C) (conformer_encoder.py:32 in channel-last layout)."""

    @staticmethod
    def forward(ctx, x):
        require_cuda(x, "GLU input")
        x = _c(x)
        Cc = x.size(-1) // 2
        rows = x.numel() // (2 * Cc)
        y = torch.empty(*x.shape[:-1], Cc, dtype=torch.float32, device=x.device)
        with torch.cuda.device(x.device):
            check(lib.avsr_glu_fwd(x.data_ptr(), y.data_ptr(), rows, Cc, _stream_handle(x.device)))
        ctx.save_for_backward(x)
        return y

    @staticmethod
    def backward(ctx, dy):
        (x,) = ctx.saved_tensors
        dy = _c(dy)
        Cc = x.size(-1) // 2
        rows = x.numel() // (2 * Cc)
        dx = torch.empty_like(x)
        with torch.cuda.device(x.device):
            check(lib.avsr_glu_bwd(x.data_ptr(), dy.data_ptr(), dx.data_ptr(), rows, Cc, _stream_handle(x.device)))
        return dx


def _chan_sums(v, dy=None, mean=None, invstd=None, gamma=None, beta=None):
    """(2, C): [sum v, sum v^2] over all rows, or (dy given) the BatchNorm+SiLU backward sums [sum ds, sum ds * x_hat]."""
    Cc = v.size(-1)
    rows = v.numel() // Cc
    out = torch.empty(2, Cc, dtype=torch.float32, device=v.device)
    ws = _pool.get("train", 148 * 2 * Cc * 4 + 1024, v.device, _stream_handle(v.device))
    with torch.cuda.device(v.device):
        check(lib.avsr_chan_sums(v.data_ptr(), _ptr(dy), _ptr(mean), _ptr(invstd), _ptr(gamma), _ptr(beta), out.data_ptr(),
                                 rows, Cc, ws.data_ptr(), ws.numel(), _stream_handle(v.device)))
    return out


def _dwconv_raw(x, w, b, flip: bool):
    B, T, Cc = x.shape
    K = w.size(-1)
    y = torch.empty_like(x)
    ws = _pool.get("train", (K + 2) * Cc * 4 + 1024, x.device, _stream_handle(x.device))
    with torch.cuda.device(x.device):
        check(lib.avsr_dwconv_raw(x.data_ptr(), w.data_ptr(), _ptr(b), y.data_ptr(), B, T, Cc, K, int(flip), ws.data_ptr(),
                                  ws.numel(), _stream_handle(x.device)))
    return y


class DwConvBnSiluFn(torch.autograd.Function):
    """depthwise Conv1d + BatchNorm1d / SyncBatchNorm (training: batch statistics over all B*T frames -- of ALL ranks of
    ``group`` when given --, running stats updated in place) + SiLU on (B, T, C) (conformer_encoder.py:33-34).

    The heavy passes (conv, per-channel sums, normalise + SiLU, their backward, tap gradients) run in libavsr_b200; the
    C-length statistics vectors are finalised here between them, which is where SyncBatchNorm's all-reduce goes
    (one packed [sum, sum^2, count] message forward, [sum ds, sum ds*x_hat] backward: torch/_functions.py:49-159)."""

    @staticmethod
    def forward(ctx, x, w, b, bn_w, bn_b, running_mean, running_var, momentum: float, eps: float, group):
        require_cuda(x, "conv module input")
        x, w, b, bn_w, bn_b = _c(x), _c(w), _c(b), _c(bn_w), _c(bn_b)
        B, T, Cc = x.shape
        conv = _dwconv_raw(x, w, b, False)
        sums = _chan_sums(conv)
        n = float(B * T)
        if group is not None:
            packed = torch.cat([sums.reshape(-1), torch.full((1,), n, dtype=torch.float32, device=x.device)])
            torch.distributed.all_reduce(packed, group=group)
            sums, n = packed[:-1].reshape(2, Cc), float(packed[-1].item())      # global row count (one host sync)
        sums64 = sums.double()
        mean = sums64[0] / n
        var = (sums64[1] / n - mean * mean).clamp_min_(0.0)
        invstd = torch.rsqrt(var + eps)
        if running_mean is not None:
            with torch.no_grad():
                unbiased = var * (n / max(n - 1.0, 1.0))
                running_mean.mul_(1.0 - momentum).add_(mean.to(running_mean.dtype), alpha=momentum)
                running_var.mul_(1.0 - momentum).add_(unbiased.to(running_var.dtype), alpha=momentum)
        mean, invstd = mean.float().contiguous(), invstd.float().contiguous()
        y = torch.empty_like(x)
        with torch.cuda.device(x.device):
            check(lib.avsr_bn_silu_fwd(conv.data_ptr(), mean.data_ptr(), invstd.data_ptr(), bn_w.data_ptr(), bn_b.data_ptr(),
                                       y.data_ptr(), B * T, Cc, _stream_handle(x.device)))
        ctx.save_for_backward(x, w, conv, mean, invstd, bn_w, bn_b)
        ctx.group, ctx.inv_count = group, 1.0 / n
        ctx.mark_non_differentiable(*[t for t in (running_mean, running_var) if t is not None])
        return y

    @staticmethod
    def backward(ctx, dy):
        x, w, conv, mean, invstd, bn_w, bn_b = ctx.saved_tensors
        dy = _c(dy)
        B, T, Cc = x.shape
        K = w.size(-1)
        local = _chan_sums(conv, dy, mean, invstd, bn_w, bn_b)            # [sum ds, sum ds * x_hat] of THIS rank
        dbt, dg = local[0].clone(), local[1].clone()                       # d beta, d gamma: local sums (DDP averages them)
        glob = local
        if ctx.group is not None:
            glob = local.clone()
            torch.distributed.all_reduce(glob, group=ctx.group)
        dconv = torch.empty_like(x)
        with torch.cuda.device(x.device):
            check(lib.avsr_bn_silu_bwd_dx(conv.data_ptr(), dy.data_ptr(), mean.data_ptr(), invstd.data_ptr(), bn_w.data_ptr(),
                                          bn_b.data_ptr(), glob[0].contiguous().data_ptr(), glob[1].contiguous().data_ptr(),
                                          float(ctx.inv_count), dconv.data_ptr(), B * T, Cc, _stream_handle(x.device)))
        dx = _dwconv_raw(dconv, w, None, True)                             # correlation with the flipped taps
        dw, db = torch.empty_like(w), torch.empty(Cc, device=x.device)
        ws = _pool.get("train", int(lib.avsr_train_workspace_bytes(B * T, Cc, K)), x.device, _stream_handle(x.device))
        with torch.cuda.device(x.device):
            check(lib.avsr_dwconv_wgrad(x.data_ptr(), dconv.data_ptr(), dw.data_ptr(), db.data_ptr(), B, T, Cc, K, ws.data_ptr(),
                                        ws.numel(), _stream_handle(x.device)))
        return dx, dw, db, dg, dbt, None, None, None, None, None


class AttentionCoreFn(torch.autograd.Function):
    """ctx = softmax(((q+u) k^T + rel_shift((q+v) p^T)) / 8, key mask) v  (attention.py:174-189 + :59-82) on projected
    q, k, v (B,T,H*64), p (2T-1,H*64).  Forward = the fused attention kernel of the module's precision; backward =
    avsr_relpos_attention_bwd (fp32, scores recomputed)."""

    @staticmethod
    def forward(ctx_, q, k, v, p, u, vb, lengths, n_heads: int, precision: str):
        require_cuda(q, "attention input")
        out = ops.relpos_attention(q, k, v, p, u, vb, lengths, n_heads, precision=precision)
        ctx_.save_for_backward(q, k, v, p, u, vb, out, lengths if lengths is not None else torch.empty(0, device=q.device))
        ctx_.n_heads, ctx_.masked = n_heads, lengths is not None
        return out

    @staticmethod
    def backward(ctx_, dctx):
        q, k, v, p, u, vb, out, lengths = ctx_.saved_tensors
        q, k, v, p, u, vb, out, dctx = (_c(t) for t in (q, k, v, p, u, vb, out, dctx))
        B, T, D = q.shape
        H = ctx_.n_heads
        dq_k, dq_p, dk, dv = (torch.empty_like(q) for _ in range(4))
        dp = torch.empty_like(p)
        ln = lengths.to(torch.int32).contiguous() if ctx_.masked else None
        ws = _pool.get("train", int(lib.avsr_relpos_attention_bwd_workspace_bytes(B, T, H)), q.device, _stream_handle(q.device))
        with torch.cuda.device(q.device):
            check(lib.avsr_relpos_attention_bwd(q.data_ptr(), k.data_ptr(), v.data_ptr(), p.data_ptr(), u.data_ptr(),
                                                vb.data_ptr(), _ptr(ln), out.data_ptr(), dctx.data_ptr(), dq_k.data_ptr(),
                                                dq_p.data_ptr(), dk.data_ptr(), dv.data_ptr(), dp.data_ptr(), B, T, H,
                                                ws.data_ptr(), ws.numel(), _stream_handle(q.device)))
        du = colsum(dq_k.reshape(-1, D)).reshape(u.shape)        # d pos_bias_u = sum over (b, t) of the k part of dq
        dvb = colsum(dq_p.reshape(-1, D)).reshape(vb.shape)
        return dq_k + dq_p, dk, dv, dp, du, dvb, None, None, None


# ------------------------------------------------------------------------------------------------ module forwards (train)
def feed_forward_train(m, x, precision: str):
    """PositionwiseFeedForward.forward in train mode: w_2(dropout(relu(w_1 x)))."""
    h = LinearFn.apply(x, m.w_1.weight, m.w_1.bias, True, precision)
    h = m.dropout(h)
    return LinearFn.apply(h, m.w_2.weight, m.w_2.bias, False, precision)


def conv_module_train(m, x, precision: str):
    """ConvolutionModule.forward in train mode on (B, T, C): pointwise_cov1 -> GLU -> depthwise + BatchNorm(batch stats)
    + SiLU -> pointwise_cov2.  ``m.norm`` stays a real BatchNorm1d: its running statistics and num_batches_tracked are
    updated like torch's (momentum None = cumulative average is not supported here)."""
    bn = m.norm
    group = None
    if isinstance(bn, torch.nn.SyncBatchNorm):        # what Lightning's sync_batchnorm=True (train.py:31) turns `norm` into
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            group = bn.process_group if bn.process_group is not None else dist.group.WORLD
            if dist.get_world_size(group) == 1:
                group = None
    elif type(bn) is not torch.nn.BatchNorm1d:
        raise NotImplementedError(f"conv_module.norm is {type(bn).__name__}: BatchNorm1d / SyncBatchNorm only")
    if bn.momentum is None:
        raise NotImplementedError("BatchNorm1d(momentum=None) (cumulative moving average) is not supported")
    h = LinearFn.apply(x, m.pointwise_cov1.weight, m.pointwise_cov1.bias, False, precision)
    g = GluFn.apply(h)
    track = bn.track_running_stats and bn.running_mean is not None
    y = DwConvBnSiluFn.apply(g, m.depthwise_conv.weight, m.depthwise_conv.bias, bn.weight, bn.bias,
                             bn.running_mean if track else None, bn.running_var if track else None, bn.momentum, bn.eps, group)
    if track and bn.num_batches_tracked is not None:
        bn.num_batches_tracked.add_(1)
    return LinearFn.apply(y, m.pointwise_cov2.weight, m.pointwise_cov2.bias, False, precision)


def attention_train(m, x, pos_emb, mask, precision: str):
    """RelPositionMultiHeadedAttention.forward (self-attention) in train mode -> (B, T, d)."""
    from .espnet_dropin.attention import mask_to_lengths
    if m.dropout.p > 0:
        raise NotImplementedError("dropout on the attention probabilities (attention_dropout_rate > 0) is not implemented "
                                  "in the fused kernel; auto_avsr trains with 0.0 (e2e_asr_conformer.py:33-39)")
    B, T, D = x.shape
    q = LinearFn.apply(x, m.linear_q.weight, m.linear_q.bias, False, precision)
    k = LinearFn.apply(x, m.linear_k.weight, m.linear_k.bias, False, precision)
    v = LinearFn.apply(x, m.linear_v.weight, m.linear_v.bias, False, precision)
    p = LinearFn.apply(pos_emb.reshape(2 * T - 1, D), m.linear_pos.weight, None, False, precision)
    lengths = None if mask is None else mask_to_lengths(mask, B, T)
    ctx = AttentionCoreFn.apply(q, k, v, p, m.pos_bias_u, m.pos_bias_v, lengths, m.h, precision)
    return LinearFn.apply(ctx, m.linear_out.weight, m.linear_out.bias, False, precision)
