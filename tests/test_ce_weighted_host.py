"""Host side of the weighted / label-smoothed upsample + cross-entropy (no GPU needed): the module's argument checks and
the float64 oracle against nn.CrossEntropyLoss(weight, ignore_index, label_smoothing) on F.interpolate."""
import pytest
import torch
import torch.nn.functional as F

from ce_weighted_reference import upsample_ce_and_grad
from lc2is_b200 import head


def test_module_rejects_unsupported_and_invalid_options():
    with pytest.raises(NotImplementedError):
        head.UpsampledCrossEntropyLoss(reduction="none")
    x = torch.zeros(1, 3, 2, 2)
    t = torch.zeros(1, 8, 8, dtype=torch.int64)
    for eps in (-0.1, 1.5):
        with pytest.raises(RuntimeError, match="label_smoothing"):
            head.UpsampledCrossEntropyLoss(label_smoothing=eps)(x, t)
    with pytest.raises(RuntimeError, match="weight tensor should be defined"):
        head.UpsampledCrossEntropyLoss(weight=torch.ones(4))(x, t)
    with pytest.raises(RuntimeError, match="weight tensor should be defined"):
        head.UpsampledCrossEntropyLoss(weight=torch.ones(3, 1))(x, t)
    with pytest.raises(ValueError):
        head.UpsampledCrossEntropyLoss()(x[0], t)
    with pytest.raises(RuntimeError, match="label_smoothing"):
        head.SegHeadLoss(label_smoothing=2.0)(torch.zeros(1, 4, 8), torch.zeros(3, 8), t)


def test_module_is_a_cross_entropy_loss():
    w = torch.rand(5)
    m = head.UpsampledCrossEntropyLoss(weight=w, ignore_index=3, reduction="sum", label_smoothing=0.2)
    assert isinstance(m, torch.nn.CrossEntropyLoss)
    assert torch.equal(m.state_dict()["weight"], w) and m.ignore_index == 3 and m.label_smoothing == 0.2
    assert "weight" not in head.SegHeadLoss().state_dict()
    assert torch.equal(head.SegHeadLoss(weight=w).state_dict()["weight"], w)


@pytest.mark.parametrize("reduction", ["mean", "sum"])
@pytest.mark.parametrize("eps", [0.0, 0.1])
@pytest.mark.parametrize("weighted", [False, True])
@pytest.mark.parametrize("size", [(16, 16), (12, 20)])
def test_oracle_matches_torch_criterion(size, weighted, eps, reduction):
    g = torch.Generator().manual_seed(7)
    B, C = 2, 6
    low = torch.randn(B, C, 4, 5, generator=g)
    target = torch.randint(0, C, (B, *size), generator=g)
    target[0, :2] = -100
    w = None
    if weighted:
        w = 0.2 + 2.8 * torch.rand(C, generator=g)
        w[1] = 0.0
    loss, grad = upsample_ce_and_grad(low, target, -100, w, eps, reduction)
    x = low.clone().requires_grad_(True)
    crit = torch.nn.CrossEntropyLoss(weight=w, ignore_index=-100, reduction=reduction, label_smoothing=eps)
    ref = crit(F.interpolate(x, size=size, mode="bilinear", align_corners=False), target)
    ref.backward()
    assert loss.dtype == torch.float64 and grad.shape == low.shape
    torch.testing.assert_close(loss.float(), ref.detach(), rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(grad.float(), x.grad, rtol=1e-4, atol=1e-6)
