"""Float64 reference of a configured criterion on the upsampled score map, for the weighted / label-smoothed K2 tests.
TEST INFRASTRUCTURE ONLY (nothing under lc2is_b200/ imports it)."""
from typing import Optional

import torch
import torch.nn.functional as F
from torch import Tensor


def upsample_ce_and_grad(low: Tensor, target: Tensor, ignore_index: int = -100, weight: Optional[Tensor] = None,
                         label_smoothing: float = 0.0, reduction: str = "mean"):
    """``F.cross_entropy(F.interpolate(low, size=target.shape[-2:], mode='bilinear'), target, weight, ignore_index,
    reduction, label_smoothing)`` (engine.py:94 on final.py:44) in float64, and d loss / d low via autograd.  torch's own
    ``F.cross_entropy`` is called (not restated): the 'mean' denominator of the smoothing term changed between torch
    releases.  Returns (loss, grad_low) as float64."""
    low = low.detach().double().clone().requires_grad_(True)
    up = F.interpolate(input=low, mode="bilinear", size=tuple(target.shape[-2:]), align_corners=False)
    w = None if weight is None else weight.detach().double()
    loss = F.cross_entropy(up, target, weight=w, ignore_index=ignore_index, reduction=reduction,
                           label_smoothing=label_smoothing)
    (g,) = torch.autograd.grad(loss, low)
    return loss.detach(), g
