"""The head math the reference writes inline at the end of every model ``forward``
(model/final.py:41-44 and its seven copies; model/model.py:50-53 for the un-normalised form).

* :func:`cosine_logits`   - K0 + K1 (+ K1b in backward), drop-in for
      ``v = F.normalize(v, dim=1); t = F.normalize(t, dim=2); einsum('bchw,bkc->bkhw', v, t)``
* :class:`SegHeadLoss`    - K0 -> K1 -> K2 -> (K1b) fused: logits, upsampled softmax-CE and all
      gradients with no [B,C,H,W] tensor and no autograd graph in between.
* :class:`UpsampledCrossEntropyLoss` - K2 for a configured criterion (engine.py:94 on final.py:44):
      ``nn.CrossEntropyLoss(weight, ignore_index, reduction, label_smoothing)`` of the bilinearly upsampled score map.
"""
from __future__ import annotations

from typing import Optional, Tuple

import torch
from torch import Tensor, nn

from . import ops
from .model.loss import _UpsampleCE, _upsample_ce_loss


def _hw_shape(P: int, hw_shape) -> Tuple[int, int]:
    if hw_shape is not None:
        return int(hw_shape[0]), int(hw_shape[1])
    h = int(round(P ** 0.5))
    if h * h != P:
        raise ValueError(f"cannot infer a square grid from {P} patches; pass hw_shape=(h, w)")
    return h, h


class _CosineLogits(torch.autograd.Function):

    @staticmethod
    def forward(ctx, v: Tensor, t: Tensor, normalize: bool, logit_scale: float, hw_shape):
        t32 = t.float()
        t_hat, inv_t = ops.proto_normalize(t32, normalize)
        C = t.shape[-2]
        logits, v_hat, inv_v = ops.cosine_logits_fwd(v, t_hat, C, hw_shape, normalize, logit_scale)
        ctx.save_for_backward(logits, v_hat, inv_v, t_hat, inv_t)
        ctx.meta = (C, normalize, logit_scale, v.dtype, t.dtype, t.dim())
        return logits

    @staticmethod
    def backward(ctx, grad_logits: Tensor):
        logits, v_hat, inv_v, t_hat, inv_t = ctx.saved_tensors
        C, normalize, logit_scale, v_dtype, t_dtype, t_dim = ctx.meta
        g = ops.grad_to_bf16(grad_logits.float().contiguous())
        gv_dtype = torch.bfloat16 if v_dtype == torch.bfloat16 else torch.float32
        grad_v, grad_t = ops.cosine_logits_bwd(g, logits, v_hat, inv_v, t_hat, inv_t, C, normalize, logit_scale,
                                               grad_v_dtype=gv_dtype)
        if t_dim == 2:
            grad_t = grad_t[0]
        return grad_v.to(v_dtype), grad_t.to(t_dtype), None, None, None


def cosine_logits(v: Tensor, t: Tensor, *, normalize: bool = True, logit_scale: float = 1.0,
                  hw_shape: Optional[Tuple[int, int]] = None) -> Tensor:
    """v [B,P,D] (fp32/bf16), t [K,D] or [B,K,D] -> score map [B,K,h,w] fp32.

    normalize=True reproduces final.py:41-43; normalize=False model.py:50,53.  The reference has
    no temperature (only commented out, model.py:70,92): ``logit_scale=1.0`` is its behaviour.
    Operands are rounded to bf16 for the tensor cores; accumulation is fp32.
    """
    h, w = _hw_shape(v.shape[1], hw_shape)
    return _CosineLogits.apply(v, t, bool(normalize), float(logit_scale), (h, w))


class _UpsampleTokens(torch.autograd.Function):

    @staticmethod
    def forward(ctx, x: Tensor, hw_shape, out_dtype):
        ctx.meta = (hw_shape, x.dtype)
        return ops.bicubic4_tokens_fwd(x, hw_shape, out_dtype)

    @staticmethod
    def backward(ctx, gy: Tensor):
        hw_shape, xdt = ctx.meta
        gx = ops.bicubic4_tokens_bwd(gy, hw_shape, torch.bfloat16 if xdt == torch.bfloat16 else torch.float32)
        return gx.to(xdt), None, None


def upsample_tokens_bicubic4(x: Tensor, hw_shape: Optional[Tuple[int, int]] = None, out_dtype=torch.bfloat16) -> Tensor:
    """model.py:42-44 in one kernel: ``x [B, h*w, C]`` (the decoder's tokens) -> ``[B, 16*h*w, C]``, the bicubic x4 upsampled
    feature map still token-major - i.e. already the operand of ``TextToPatch.visual`` (bf16 by default: the tensor-core
    projection rounds its operands to bf16 anyway; pass ``torch.float32`` for the reference's dtype).  Differentiable."""
    h, w = _hw_shape(x.shape[1], hw_shape)
    return _UpsampleTokens.apply(x, (h, w), out_dtype)


class _SegHeadLoss(torch.autograd.Function):

    @staticmethod
    def forward(ctx, v, t, labels, ignore_index, normalize, logit_scale, hw_shape, reduction, weight=None,
                label_smoothing=0.0):
        t_hat, inv_t = ops.proto_normalize(t.float(), normalize)
        C = t.shape[-2]
        logits, v_hat, inv_v = ops.cosine_logits_fwd(v, t_hat, C, hw_shape, normalize, logit_scale)
        need_grad = ctx.needs_input_grad[0] or ctx.needs_input_grad[1]
        n_valid = ops.count_valid(labels, C, ignore_index)
        loss, _, gbf = _upsample_ce_loss(logits, labels, ignore_index, reduction, weight, label_smoothing,
                                        want_grad=need_grad, want_bf16=need_grad, n_valid=n_valid)
        if need_grad:
            ctx.save_for_backward(gbf, logits, v_hat, inv_v, t_hat, inv_t)
        ctx.meta = (C, normalize, logit_scale, v.dtype, t.dtype, t.dim())
        ctx.mark_non_differentiable(logits, n_valid)
        return loss.reshape(()), logits, n_valid

    @staticmethod
    def backward(ctx, grad_loss, _gl, _gn):
        gbf, logits, v_hat, inv_v, t_hat, inv_t = ctx.saved_tensors
        C, normalize, logit_scale, v_dtype, t_dtype, t_dim = ctx.meta
        gs = grad_loss.detach().float().reshape(1).contiguous()      # upstream scalar, stays on device
        gv_dtype = torch.bfloat16 if v_dtype == torch.bfloat16 else torch.float32
        grad_v, grad_t = ops.cosine_logits_bwd(gbf, logits, v_hat, inv_v, t_hat, inv_t, C, normalize, logit_scale,
                                               grad_scale=gs, grad_v_dtype=gv_dtype)
        if t_dim == 2:
            grad_t = grad_t[0]
        return grad_v.to(v_dtype), grad_t.to(t_dtype), None, None, None, None, None, None, None, None


def _check_ce_options(C: int, weight: Optional[Tensor], label_smoothing: float, reduction: str) -> None:
    """The argument errors nn.CrossEntropyLoss raises, before any device work."""
    if reduction not in ("mean", "sum"):
        raise NotImplementedError(
            "reduction='none' needs a backward that takes a per-pixel upstream gradient; the fused forward+backward "
            "kernels support reduction='mean' | 'sum'")
    if not 0.0 <= label_smoothing <= 1.0:
        raise RuntimeError(f"label_smoothing must be between 0.0 and 1.0. Got: {label_smoothing}")
    if weight is not None and (weight.dim() != 1 or weight.numel() != C):
        raise RuntimeError(f"weight tensor should be defined either for all {C} classes or no classes but got weight "
                           f"tensor of shape: {list(weight.shape)}")


class UpsampledCrossEntropyLoss(nn.CrossEntropyLoss):
    """``nn.CrossEntropyLoss(weight, ignore_index=..., reduction=..., label_smoothing=...)`` applied to
    ``F.interpolate(input, size=target.shape[-2:], mode="bilinear", align_corners=False)`` - the criterion of
    engine.py:94 on the score map of final.py:44 - without the upsampled [B,C,H,W] tensor: one fused K2 pass computes the
    loss and d loss / d input.

    forward(input [B,C,h,w] low-resolution scores (fp32 / bf16 / fp16), target [B,H,W] int64) -> scalar.  Any (H, W):
    power-of-two scales 4 / 8 / 16 take the fast kernels, the rest the generic one.  ``weight`` is a buffer (follows
    ``.to()`` and ``state_dict``); 'mean' divides by the summed weights of the counted pixels, like torch.  Labels outside
    [0, C) that are not ignore_index are skipped.  reduction='none' is not supported.  CUDA tensors only; no host
    synchronisation (CUDA-graph capturable)."""

    def __init__(self, weight: Optional[Tensor] = None, size_average=None, ignore_index: int = -100, reduce=None,
                 reduction: str = "mean", label_smoothing: float = 0.0) -> None:
        super().__init__(weight, size_average, ignore_index, reduce, reduction, label_smoothing)
        if self.reduction not in ("mean", "sum"):
            _check_ce_options(0, None, 0.0, self.reduction)

    def forward(self, input: Tensor, target: Tensor) -> Tensor:
        if input.dim() != 4 or target.dim() != 3 or target.shape[0] != input.shape[0]:
            raise ValueError(f"UpsampledCrossEntropyLoss: input must be [B,C,h,w] and target [B,H,W], got "
                             f"{tuple(input.shape)} / {tuple(target.shape)}")
        weight = self.weight
        _check_ce_options(input.shape[1], weight, float(self.label_smoothing), self.reduction)
        if target.device != input.device or (weight is not None and weight.device != input.device):
            raise RuntimeError("Expected all tensors to be on the same device, but found input on "
                               f"{input.device}, target on {target.device}"
                               + ("" if weight is None else f", weight on {weight.device}"))
        if weight is not None:
            weight = weight.detach().float().contiguous()
        return _UpsampleCE.apply(input, target, self.ignore_index, self.reduction, weight, float(self.label_smoothing))


class SegHeadLoss(nn.Module):
    """Fused head + criterion: ``criterion(F.interpolate(cosine_logits(v, t), 'bilinear', size=H), labels)``
    (final.py:41-44 + engine.py:94, or final.py:266-268 + loss.py:17-21 for the aux head).

    forward(v [B,P,D], t [K,D]|[B,K,D], labels [B,H,W] int64) -> (loss, low_logits [B,K,h,w], n_valid)

    ``weight`` (fp32 [K], a buffer) and ``label_smoothing`` are those of ``nn.CrossEntropyLoss`` (see
    :class:`UpsampledCrossEntropyLoss`); n_valid stays the number of counted pixels.
    """

    def __init__(self, ignore_index: int = -100, normalize: bool = True, logit_scale: float = 1.0,
                 reduction: str = "mean", weight: Optional[Tensor] = None, label_smoothing: float = 0.0) -> None:
        super().__init__()
        if reduction not in ("mean", "sum"):
            raise NotImplementedError("SegHeadLoss supports reduction='mean' | 'sum'")
        self.ignore_index = ignore_index
        self.normalize = normalize
        self.logit_scale = logit_scale
        self.reduction = reduction
        self.register_buffer("weight", weight)
        self.label_smoothing = label_smoothing

    def forward(self, v: Tensor, t: Tensor, labels: Tensor, hw_shape=None):
        h, w = _hw_shape(v.shape[1], hw_shape)
        weight = self.weight
        _check_ce_options(t.shape[-2], weight, float(self.label_smoothing), self.reduction)
        if weight is not None:
            weight = weight.detach().float().contiguous()
        return _SegHeadLoss.apply(v, t, labels, self.ignore_index, self.normalize, self.logit_scale, (h, w),
                                  self.reduction, weight, float(self.label_smoothing))
