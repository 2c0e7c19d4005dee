"""Mirror of the reference ``model/loss.py`` (same class names, ctor signatures, return values).

``AuxiliaryLoss`` (loss.py:12-21) runs on the fused K2 kernel: bilinear upsample to the label
size + softmax cross-entropy + their backward in one pass, with no upsampled tensor in memory.
It is also the drop-in for ``nn.CrossEntropyLoss`` applied to ``F.interpolate(score, 'bilinear')``
(final.py:44 + engine.py:94): feed it the low-resolution score map instead.
``ContrastiveLoss`` (loss.py:39-64) runs on the K4 kernels for CUDA inputs (class-axis CE per pixel + the row-axis
CE against the one-hot target, forward and backward); ``NPairLoss`` (loss.py:23-37) is kept as plain PyTorch.
"""
from typing import Callable, Optional, Union

import numpy as np
import torch
from torch import Tensor, nn

from .. import ops


def _upsample_ce_loss(low32, labels, ignore_index, reduction, weight, label_smoothing, want_grad, want_bf16=False,
                      n_valid=None):
    """K2 with the 'mean' denominator of nn.CrossEntropyLoss -> (loss fp32 [1], grad_low, grad_low_bf16), the gradients
    scaled by 1 / denominator: the number of counted pixels (n_valid, counted here unless given), or with a weight or a
    smoothing the summed class weights of the counted pixels (ops.ce_weight_sum).  All on the device."""
    mean = reduction == "mean"
    if weight is None and label_smoothing == 0:
        if n_valid is None:
            n_valid = ops.count_valid(labels, low32.shape[1], ignore_index)
        gscale = ops.mean_scale(n_valid) if mean else None
        loss_sum, grad, gbf = ops.upsample_ce(low32, labels, ignore_index, gscale, want_grad=want_grad,
                                              want_bf16=want_bf16)
        return (ops.finalize_loss(loss_sum, n_valid) if mean else loss_sum.float()), grad, gbf
    den = ops.ce_weight_sum(labels, low32.shape[1], ignore_index, weight) if mean else None
    # 1 / 0 = inf when nothing is counted: every gradient term of an uncounted pixel is a select, not a product
    gscale = torch.reciprocal(den).float() if mean else None
    loss_sum, grad, gbf = ops.upsample_ce(low32, labels, ignore_index, gscale, want_grad=want_grad, want_bf16=want_bf16,
                                          weight=weight, label_smoothing=label_smoothing)
    return (ops.weighted_mean_loss(loss_sum, den) if mean else loss_sum.float()), grad, gbf


class _UpsampleCE(torch.autograd.Function):

    @staticmethod
    def forward(ctx, low: Tensor, target: Tensor, ignore_index: int, reduction: str,
                weight: Optional[Tensor] = None, label_smoothing: float = 0.0):
        need_grad = ctx.needs_input_grad[0]
        loss, grad, _ = _upsample_ce_loss(low.float(), target, ignore_index, reduction, weight, label_smoothing,
                                         want_grad=need_grad)
        if need_grad:
            ctx.save_for_backward(grad)
        ctx.in_dtype = low.dtype
        return loss.reshape(())

    @staticmethod
    def backward(ctx, grad_out: Tensor):
        (grad,) = ctx.saved_tensors
        return (grad * grad_out).to(ctx.in_dtype), None, None, None, None, None


class AuxiliaryLoss(nn.CrossEntropyLoss):
    """loss.py:12-21.  forward(input [B,C,h,w], target [B,H,W] int64) -> scalar."""

    def __init__(self, weight: Optional[Tensor] = None, size_average=None, ignore_index: int = -100, reduce=None,
                 reduction: str = 'mean', label_smoothing: float = 0) -> None:
        super().__init__(weight, size_average, ignore_index, reduce, reduction, label_smoothing)
        if weight is not None or label_smoothing != 0 or self.reduction not in ("mean", "sum"):
            raise NotImplementedError(
                "the B200 AuxiliaryLoss kernel covers the reference's usage (no class weights, no label "
                "smoothing, reduction 'mean'|'sum'); there is deliberately no silent PyTorch fallback.  "
                "lc2is_b200.head.UpsampledCrossEntropyLoss takes class weights and label smoothing")

    def forward(self, input: Tensor, target: Tensor) -> Tensor:
        B, H, W = target.shape
        if W != H:
            # the reference passes size=H (an int): the output is H x H regardless of W (loss.py:19)
            raise ValueError("AuxiliaryLoss follows loss.py:19 (size=H): labels must be square")
        return _UpsampleCE.apply(input, target, self.ignore_index, self.reduction)


class NPairLoss(nn.Module):
    """loss.py:23-37 (PyTorch pass-through)."""

    def __init__(self, reduction: Union[Callable, None] = torch.mean) -> None:
        super().__init__()
        self.reduction = reduction

    def forward(self, x: Tensor, x_pos: Tensor, x_neg: Tensor):
        pos = torch.matmul(x, x_pos.transpose(0, 1))
        neg = torch.matmul(x, x_neg.transpose(0, 1)).sum(-1, keepdim=True)
        res = (pos / (pos + neg)).sum(-1)
        if self.reduction:
            res = self.reduction(res)
        return res


class _ContrastiveCE(torch.autograd.Function):
    """Both cross-entropies of loss.py:58-59 on the K4 kernels.  -> (total, loss_visual, loss_textual)."""

    @staticmethod
    def forward(ctx, outputs: Tensor, labels: Tensor, ignore_index: int):
        out32 = outputs.float().contiguous()
        B, hw, C = out32.shape
        w = labels.shape[2]
        sums, counts, col_lse, col_adj = ops.contrastive_fwd(out32, labels, ignore_index)
        n_counted, n_bad = counts.tolist()            # one sync, like F.one_hot's own range check (loss.py:54)
        if n_bad:
            raise RuntimeError("Class values must be smaller than num_classes.")
        n_text = float(B * w * C)
        loss_visual = (sums[0] / n_counted if n_counted else sums[0] * float("nan")).float()
        loss_textual = (sums[1] / n_text).float()
        ctx.save_for_backward(out32, labels, col_lse, col_adj)
        ctx.meta = (ignore_index, n_counted, n_text, outputs.dtype)
        return (loss_textual + loss_visual) / 2, loss_visual, loss_textual

    @staticmethod
    def backward(ctx, g_total: Tensor, g_visual: Tensor, g_textual: Tensor):
        out32, labels, col_lse, col_adj = ctx.saved_tensors
        ignore_index, n_counted, n_text, in_dtype = ctx.meta
        coef = torch.stack([(0.5 * g_total + g_visual) / max(n_counted, 1),
                            (0.5 * g_total + g_textual) / n_text]).float()
        grad = ops.contrastive_bwd(out32, labels, ignore_index, col_lse, col_adj, coef)
        return grad.to(in_dtype), None, None


class ContrastiveLoss(nn.Module):
    """loss.py:39-64, including the 151-way one-hot whose class axis torch takes to be the image-row axis
    (loss.py:51-60).  forward(outputs [B, h*w, 151], labels [B, h, w]) -> (total, loss_visual, loss_textual).

    Runs on the K4 kernels (CUDA tensors only - like AuxiliaryLoss there is deliberately no PyTorch / CPU fallback);
    covers the default criterion options (no class weights, no label smoothing, reduction 'mean')."""

    NUM_CLASSES = 151        # hard-coded in the reference (loss.py:54)

    def __init__(self, weight: Optional[Tensor] = None, size_average=None, ignore_index: int = -100, reduce=None,
                 reduction: str = 'mean', label_smoothing: float = 0) -> None:
        super().__init__()
        self.criterion = nn.CrossEntropyLoss(weight, size_average, ignore_index, reduce, reduction, label_smoothing)
        if weight is not None or label_smoothing != 0 or self.criterion.reduction != "mean":
            raise NotImplementedError(
                "the B200 ContrastiveLoss kernels cover no class weights, no label smoothing, reduction 'mean'; "
                "there is deliberately no silent PyTorch fallback")

    def forward(self, outputs: Tensor, labels: Tensor):
        if self.criterion.ignore_index >= 0:
            # what the reference's textual term raises (torch: probabilities target + non-negative ignore_index)
            raise RuntimeError("ignore_index is not supported for floating point target")
        side = int(np.sqrt(outputs.shape[1]).item())                      # loss.py:47
        if outputs.dim() != 3 or labels.dim() != 3 or side * side != outputs.shape[1]:
            raise ValueError("ContrastiveLoss: outputs must be [B, h*h, C] and labels [B, h, h]")
        if tuple(labels.shape) != (outputs.shape[0], side, side) or outputs.shape[2] != self.NUM_CLASSES:
            # the reference fails here too: the one-hot target [B,h,w,151] must have the shape of the [B,h,w,C] view
            raise ValueError(f"ContrastiveLoss: labels {tuple(labels.shape)} / outputs {tuple(outputs.shape)} do not "
                             f"give a [B,h,w,{self.NUM_CLASSES}] one-hot target of the outputs' shape (loss.py:51-58)")
        return _ContrastiveCE.apply(outputs, labels, self.criterion.ignore_index)
