"""Drop-in for ``espnet.nets.pytorch_backend.encoder.conformer_encoder`` of mpc001/auto_avsr.

Same class names, constructor signatures, sub-module / parameter names and state-dict keys as the
reference (espnet/nets/pytorch_backend/encoder/conformer_encoder.py:19,38,186), so ``E2E``
(e2e_asr_conformer.py:33-39), ``lightning.py`` and the released checkpoints keep working unchanged;
only ``forward`` differs: on a CUDA tensor it runs the hand-written sm_100a kernels of libavsr_b200.so.

Scope: inference forward (``eval()``: one fused C-ABI call, outputs carry no autograd graph) plus the FIRST SLICE of
training (SURVEY.md section 8f item 2): ``LayerNorm``, ``PositionwiseFeedForward`` and ``ConvolutionModule`` run forward
AND backward in libavsr_b200 (auto_avsr_b200/train.py: batch-statistics BatchNorm incl. running-stat update, dgrad /
wgrad as tensor-core GEMMs, gradients on the original Parameters).  The rel-pos attention backward is not built yet, so
``RelPositionMultiHeadedAttention`` / ``EncoderLayer`` / ``ConformerEncoder`` still raise ``NotImplementedError`` in
``train()`` instead of silently falling back to PyTorch.  CPU tensors raise too: there is no CPU path in this package.
"""
from __future__ import annotations

import copy
import logging
import os
from typing import Optional

import torch

from .. import ops
from ..engine import EncoderEngine, default_precision
from .attention import RelPositionMultiHeadedAttention, mask_to_lengths
from .embedding import RelPositionalEncoding
from .layer_norm import LayerNorm
from .positionwise_feed_forward import PositionwiseFeedForward
from .repeat import repeat


def _inference_only(module: torch.nn.Module, what: str) -> None:
    if module.training:
        raise NotImplementedError(
            f"{what}: the B200 path implements the inference forward only (call .eval()); training "
            "forward/backward is the next scope row (SURVEY.md 8f #2) and is not silently routed to PyTorch")


class ConvolutionModule(torch.nn.Module):
    """pointwise(C->2C) -> GLU -> depthwise(k) -> BatchNorm1d -> SiLU -> pointwise(C->C)
    (reference conformer_encoder.py:19-35; note its spelling ``pointwise_cov1/2``)."""

    def __init__(self, channels, kernel_size, bias=True):
        super().__init__()
        assert (kernel_size - 1) % 2 == 0
        self.pointwise_cov1 = torch.nn.Conv1d(channels, 2 * channels, 1, bias=bias)
        self.depthwise_conv = torch.nn.Conv1d(channels, channels, kernel_size, padding=(kernel_size - 1) // 2,
                                              groups=channels, bias=bias)
        self.norm = torch.nn.BatchNorm1d(channels)        # stays a real BatchNorm1d (SyncBN conversion, checkpoints)
        self.pointwise_cov2 = torch.nn.Conv1d(channels, channels, 1, bias=bias)
        self.activation = torch.nn.SiLU(inplace=True)
        self.precision: Optional[str] = None

    def forward(self, x, residual: Optional[torch.Tensor] = None):
        """x (B, T, C) -> (B, T, C); ``residual`` (extension) is added in the last GEMM's epilogue."""
        prec = self.precision or default_precision()
        if self.training:
            # training slice (SURVEY.md 8f #2): batch-statistics BatchNorm, forward and backward in libavsr_b200
            # (eval mode = the inference kernels below; their outputs carry no autograd graph)
            if not x.is_cuda:
                raise RuntimeError("ConvolutionModule: CPU tensor; auto_avsr_b200 has no CPU fallback")
            from ..train import conv_module_train
            y = conv_module_train(self, x, prec)
            return y if residual is None else residual + y
        C = self.pointwise_cov2.weight.size(0)
        g = ops.pointwise_glu(x, self.pointwise_cov1.weight, self.pointwise_cov1.bias, prec)
        h = ops.dwconv_bn_silu(g, self.depthwise_conv.weight, self.depthwise_conv.bias, self.norm.weight,
                               self.norm.bias, self.norm.running_mean, self.norm.running_var)
        return ops.linear(h, self.pointwise_cov2.weight.view(C, C), self.pointwise_cov2.bias, residual=residual,
                          precision=prec)


class EncoderLayer(torch.nn.Module):
    """macaron-FFN -> rel-pos MHA -> conv module -> FFN -> LayerNorm (reference conformer_encoder.py:38-170).

    Only the configuration the reference instantiates is implemented on the device
    (normalize_before=True, concat_after=False, macaron_style=True, conv module present, cache=None)."""

    def __init__(self, size, self_attn, feed_forward, conv_module, dropout_rate, normalize_before=True,
                 concat_after=False, macaron_style=False):
        super().__init__()
        self.self_attn = self_attn
        self.feed_forward = feed_forward
        self.ff_scale = 1.0
        self.conv_module = conv_module
        self.macaron_style = macaron_style
        self.norm_ff = LayerNorm(size)
        self.norm_mha = LayerNorm(size)
        if self.macaron_style:
            self.feed_forward_macaron = copy.deepcopy(feed_forward)
            self.ff_scale = 0.5
            self.norm_ff_macaron = LayerNorm(size)
        if self.conv_module is not None:
            self.norm_conv = LayerNorm(size)
            self.norm_final = LayerNorm(size)
        self.dropout = torch.nn.Dropout(dropout_rate)
        self.size = size
        self.normalize_before = normalize_before
        self.concat_after = concat_after
        if self.concat_after:
            self.concat_linear = torch.nn.Linear(size + size, size)

    def forward(self, x_input, mask, cache=None):
        if cache is not None or self.concat_after or not self.normalize_before:
            raise NotImplementedError("EncoderLayer: only normalize_before=True, concat_after=False, cache=None "
                                      "(the configuration auto_avsr instantiates) runs on the B200 path")
        if isinstance(x_input, tuple):
            x, pos_emb = x_input[0], x_input[1]
        else:
            raise NotImplementedError("EncoderLayer: the B200 path needs the (x, pos_emb) rel-pos input")
        if self.training:
            # the reference's schedule with its dropouts (conformer_encoder.py:110-162); every sub-module runs forward and
            # backward in libavsr_b200, torch adds the residuals and draws the dropout masks
            if self.macaron_style:
                x = x + self.ff_scale * self.dropout(self.feed_forward_macaron(self.norm_ff_macaron(x)))
            x = x + self.dropout(self.self_attn(self.norm_mha(x), None, None, pos_emb, mask))
            if self.conv_module is not None:
                x = x + self.dropout(self.conv_module(self.norm_conv(x)))
            x = x + self.ff_scale * self.dropout(self.feed_forward(self.norm_ff(x)))
            if self.conv_module is not None:
                x = self.norm_final(x)
            return (x, pos_emb), mask
        if self.macaron_style:
            x = self.feed_forward_macaron(self.norm_ff_macaron(x), residual=x, scale=self.ff_scale)
        x = self.self_attn(self.norm_mha(x), None, None, pos_emb, mask, residual=x)
        if self.conv_module is not None:
            x = self.conv_module(self.norm_conv(x), residual=x)
        x = self.feed_forward(self.norm_ff(x), residual=x, scale=self.ff_scale)
        if self.conv_module is not None:
            x = self.norm_final(x)
        return (x, pos_emb), mask


def _rename_state_dict(old_prefix, new_prefix, state_dict):
    old_keys = [k for k in state_dict if k.startswith(old_prefix)]
    if old_keys:
        logging.warning(f"Rename: {old_prefix} -> {new_prefix}")
    for k in old_keys:
        state_dict[k.replace(old_prefix, new_prefix)] = state_dict.pop(k)


def _pre_hook(state_dict, prefix, local_metadata, strict, missing_keys, unexpected_keys, error_msgs):
    # checkpoint compatibility, reference conformer_encoder.py:173-183
    _rename_state_dict(prefix + "input_layer.", prefix + "embed.", state_dict)
    _rename_state_dict(prefix + "norm.", prefix + "after_norm.", state_dict)


class ConformerEncoder(torch.nn.Module):
    """12-layer rel-pos Conformer encoder (reference conformer_encoder.py:186-282).

    ``forward(xs (B,T,d) f32, masks (B,1,T) bool | None) -> (xs (B,T,d), masks)``: one call into the C ABI
    (``avsr_plan_forward``: CUDA-graph replay of the whole 12-layer schedule).  Extra attributes:
    ``precision`` ("f16" default | "tf32" | "fp32" CUDA-core reference path), ``use_graph`` / ``graph_after`` (a
    shape runs on direct launches until seen ``graph_after`` times, then from its CUDA graph), ``assume_frozen`` (skip
    the per-call parameter-version check), ``check_saturation`` (diagnostic forward that raises ``SaturationError``
    when an fp16 operand hit +-65504; env AVSR_B200_CHECK_SAT=1), ``check_mask`` (verify that ``masks`` is a prefix
    mask; env AVSR_B200_CHECK_MASK=1), ``refresh_weights()``.
    """

    def __init__(self, attention_dim=768, attention_heads=12, linear_units=3072, num_blocks=12, dropout_rate=0.1,
                 positional_dropout_rate=0.1, attention_dropout_rate=0.0, normalize_before=True, concat_after=False,
                 macaron_style=True, use_cnn_module=True, zero_triu=False, cnn_module_kernel=31, padding_idx=-1,
                 relu_type="swish", layer_drop_rate=0.0):
        super().__init__()
        self._register_load_state_dict_pre_hook(_pre_hook)
        self.embed = torch.nn.Sequential(RelPositionalEncoding(attention_dim, positional_dropout_rate))
        self.normalize_before = normalize_before
        # relu_type is accepted and ignored exactly like the reference (its FFN is ReLU, SURVEY.md D5)
        self.encoders = repeat(
            num_blocks,
            lambda lnum: EncoderLayer(
                attention_dim,
                RelPositionMultiHeadedAttention(attention_heads, attention_dim, attention_dropout_rate, zero_triu),
                PositionwiseFeedForward(attention_dim, linear_units, dropout_rate),
                ConvolutionModule(attention_dim, cnn_module_kernel) if use_cnn_module else None,
                dropout_rate, normalize_before, concat_after, macaron_style),
            layer_drop_rate=0.0)
        if self.normalize_before:
            self.after_norm = LayerNorm(attention_dim)

        self._device_path_ok = (normalize_before and not concat_after and macaron_style and use_cnn_module
                                and not zero_triu and attention_dim == attention_heads * 64)
        self._cfg = (attention_dim, attention_heads, linear_units, num_blocks, cnn_module_kernel)
        self.precision: Optional[str] = None
        self.use_graph = True
        self.graph_after: Optional[int] = None      # None: EncoderEngine.GRAPH_AFTER (3); 1: capture at first sight
        self.assume_frozen = False
        self.check_saturation = os.environ.get("AVSR_B200_CHECK_SAT", "0") == "1"
        self.check_mask = os.environ.get("AVSR_B200_CHECK_MASK", "0") == "1"
        self._engine: Optional[EncoderEngine] = None
        self._tracked = None
        self._fingerprint = None

    # ---- weight tracking -------------------------------------------------------------------------
    def _apply(self, fn, *args, **kwargs):
        out = super()._apply(fn, *args, **kwargs)
        self.refresh_weights()
        return out

    def refresh_weights(self) -> None:
        """Call after editing parameters in a way that bypasses tensor version counters."""
        self._tracked = None
        self._fingerprint = None
        if getattr(self, "_engine", None) is not None:
            self._invalidate()

    def _invalidate(self) -> None:
        """Forget the prepared weights and every plan that bakes their address: the engine's and the fused head's."""
        self._engine.invalidate()
        head = getattr(self, "_fused_head", None)
        if head is not None:
            head.plans.clear()

    def _weights_fingerprint(self):
        if self._tracked is None:
            self._tracked = [t for t in self.state_dict(keep_vars=True).values() if t.is_floating_point()]
        ts = self._tracked
        return (sum(t._version for t in ts), ts[0].data_ptr(), ts[-1].data_ptr(), str(ts[0].device))

    def _prepared(self, device, precision):
        if self._engine is None:
            self._engine = EncoderEngine(*self._cfg)
        if self.graph_after is not None:
            self._engine.graph_after = int(self.graph_after)
        if not (self.assume_frozen and self._fingerprint is not None):
            fp = self._weights_fingerprint()
            if fp != self._fingerprint:
                self._invalidate()
                self._fingerprint = fp
        return self._engine.prepare(lambda: self.state_dict(keep_vars=True), device, precision)

    # ---- forward ---------------------------------------------------------------------------------
    def forward(self, xs, masks, taps: Optional[torch.Tensor] = None):
        if not self._device_path_ok:
            raise NotImplementedError("ConformerEncoder: only the auto_avsr configuration (normalize_before, macaron, "
                                      "cnn module, d_k = 64, zero_triu=False) runs on the B200 path")
        if not xs.is_cuda:
            raise RuntimeError("ConformerEncoder.forward: input is on the CPU; auto_avsr_b200 has no CPU fallback -- "
                               "move the encoder and its input to a CUDA (B200) device")
        precision = self.precision or default_precision()
        if self.training:
            # training (SURVEY.md 8f #2): module by module under autograd, every module's forward AND backward in
            # libavsr_b200 (auto_avsr_b200/train.py); MultiSequential draws the reference's CPU uniforms itself
            for m in self.modules():
                if hasattr(m, "precision") and m is not self and m.precision is None:
                    m.precision = precision
            xs, masks_ = self.embed(xs), masks
            xs, masks_ = self.encoders(xs, masks_)
            if isinstance(xs, tuple):
                xs = xs[0]
            if self.normalize_before:
                xs = self.after_norm(xs)
            return xs, masks
        torch.empty(len(self.encoders)).uniform_()     # the reference draws these CPU uniforms every call (repeat.py:23)
        lengths = None if masks is None else mask_to_lengths(masks, xs.size(0), xs.size(1), check=self.check_mask)
        prepared = self._prepared(xs.device, precision)
        out = self._engine.forward(prepared, xs.detach().float(), lengths, precision, use_graph=self.use_graph,
                                   taps=taps, check_saturation=self.check_saturation)
        return out, masks
