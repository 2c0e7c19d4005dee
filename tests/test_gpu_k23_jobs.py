"""k23_rc_kernel (x16 fused K2+K3) with one 16 x 16 pixel group per warp job: the two half-warps sweep the two halves of
the (padded) class range and merge their partial sums and argmax candidates.  These cases aim at what that split can
get wrong: ties across the split, class counts whose padding differs, odd widths (no TMA staging), the exact slow path,
and the benchmark's own shapes.  Dyadic logits keep the upsampled values exact, so integer outputs compare bit for bit."""
import pytest
import torch
import torch.nn.functional as F

from oracle import head_oracle as O
from lc2is_b200 import ops, synthetic

pytestmark = pytest.mark.gpu
DEV = "cuda"
S = 16


def _per_image_ref(pred, lab, C):
    out = torch.zeros(pred.shape[0], 3, C, dtype=torch.int64, device=pred.device)
    for n in range(pred.shape[0]):
        cm = O.confusion_matrix(pred[n], lab[n], C)
        out[n, 0] = torch.diag(cm); out[n, 1] = cm.sum(1); out[n, 2] = cm.sum(0)
    return out


def _check(low, labels, ign, oracle=True):
    """Fused kernel against the split K2 (loss, gradient) and K3 (confusion matrix, per-image counts, predictions)
    kernels on the same packed labels, and against the float64 oracle on the device.  Returns the predictions."""
    N, C, h, w = low.shape
    H, W = S * h, S * w
    dl, dlab = low.to(DEV), labels.to(DEV)
    loss_sum, n_valid, grad, packed = ops.upsample_ce_split(dl, dlab, ign)
    assert ops._lib.lib.lc2is_ce_argmax_fused_supported(C, h, w, H, W)
    ls = torch.zeros(1, dtype=torch.float64, device=DEV)
    g = torch.zeros_like(dl)
    nv = torch.zeros(1, dtype=torch.int64, device=DEV)
    cm, pi, pred = ops.ce_argmax_fused(dl, packed, (H, W), ls, g, per_image=True, want_pred=True, onehot=True, n_valid=nv)
    cm3, pi3, pred3 = ops.argmax_confmat_packed(dl, packed, (H, W), per_image=True, want_pred=True)
    assert torch.equal(pred, pred3)
    assert torch.equal(cm, cm3)
    assert torch.equal(pi, pi3)
    assert int(nv) == int(n_valid)
    assert abs(float(ls) - float(loss_sum)) <= 1e-6 * abs(float(loss_sum))
    assert float((g - grad).abs().max()) <= 1e-5 * float(grad.abs().max())
    if oracle:
        target = torch.where((dlab >= 0) & (dlab < C), dlab, torch.full_like(dlab, ign))
        x = dl.double().requires_grad_(True)
        up = F.interpolate(x, mode="bilinear", scale_factor=S)
        ref_loss = F.cross_entropy(up, target, ignore_index=ign, reduction="sum")
        (ref_grad,) = torch.autograd.grad(ref_loss, x)
        pred_ref = O.argmax_logits(up.detach())                 # exact values: the first class of a tie wins
        del up
        assert torch.equal(pred, pred_ref)
        assert torch.equal(cm, O.confusion_matrix(pred_ref, dlab, C))
        assert torch.equal(pi, _per_image_ref(pred_ref, dlab, C))
        assert abs(float(ls) - float(ref_loss.detach())) <= 2e-6 * abs(float(ref_loss))
        assert float((g.double() - ref_grad).abs().max()) <= 1e-5 * float(ref_grad.abs().max())
    return pred


def test_ties_across_the_half_warp_split_keep_the_first_class():
    """C = 150 pads to 152: the lower half-warp sweeps classes 0..75, the upper 76..151, each in 9 chunks of 8 classes and
    a last chunk of 4 (72..75 and 148..151)."""
    N, C, h, w = 4, 150, 4, 4
    low = synthetic.make_dyadic_logits(N, C, h, w)
    top = float(low.max()) + 1.0
    low[0, 10] = top; low[0, 100] = top                        # one class in each half, over the whole image
    low[1, 75] = top; low[1, 76] = top                         # the last class of the lower half, the first of the upper
    low[2, 85] = top; low[2, 149] = top; low[2, 5] = top       # two upper-half chunks and the lower half
    low[3, 74] = top; low[3, 148] = top                        # the two short last chunks
    labels = synthetic.make_labels(N, S * h, S * w, C, block=8, ignore_frac=0.1)
    pred = _check(low, labels, 0)
    assert bool((pred[0] == 10).all()) and bool((pred[1] == 75).all()) and bool((pred[2] == 5).all())
    assert bool((pred[3] == 74).all())


def test_upper_half_wins_when_strictly_larger():
    N, C, h, w = 1, 150, 3, 4
    low = synthetic.make_dyadic_logits(N, C, h, w)
    top = float(low.max()) + 1.0
    low[0, 10] = top; low[0, 100] = top + 0.25
    labels = synthetic.make_labels(N, S * h, S * w, C, block=8)
    pred = _check(low, labels, 0)
    assert bool((pred == 100).all())


@pytest.mark.parametrize("N,C,h,w", [(2, 16, 3, 5), (2, 75, 4, 7), (2, 150, 3, 9), (1, 151, 5, 4), (2, 200, 2, 3),
                                     (1, 3, 2, 3), (2, 150, 4, 8), (1, 24, 3, 4)])
def test_class_counts_and_odd_widths(N, C, h, w):
    """Paddings of 0 / 5 / 2 / 1 / 0 / 5 classes, half-warp class ranges with and without a short last chunk (8, 40, 76,
    76, 100, 4 classes); odd widths stage the cells without TMA."""
    low = synthetic.make_dyadic_logits(N, C, h, w)
    labels = synthetic.make_labels(N, S * h, S * w, C, block=8, ignore_frac=0.1)
    labels[0, :2] = C + 3
    _check(low, labels, 0)


@pytest.mark.parametrize("w", [4, 5])
def test_wide_range_groups_take_the_exact_path(w):
    """Groups whose taps span more than the fast path's range at C = 150, inside and on the top / left border."""
    N, C, h = 2, 150, 4
    low = synthetic.make_dyadic_logits(N, C, h, w)
    low[0, 37, 1, 2] = 60.0
    low[0, 3, 0, 0] = -50.0
    low[1, 120, h - 1, w - 1] = 45.0
    labels = synthetic.make_labels(N, S * h, S * w, C, block=8, ignore_frac=0.1)
    _check(low, labels, 0)


@pytest.mark.parametrize("B", [16, 8])
def test_benchmark_shapes(B):
    """The benchmarked geometry (32 x 32 -> 512 x 512, C = 150) at B = 16 and at the cfg4 batch of 8."""
    C, h = 150, 32
    low = synthetic.make_dyadic_logits(B, C, h, h)
    labels = synthetic.make_labels(B, S * h, S * h, C, ignore_frac=0.1)
    _check(low, labels, 0)
