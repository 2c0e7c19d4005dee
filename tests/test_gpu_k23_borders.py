"""k23_rc_kernel (x16 fused K2+K3): the border groups (top / bottom row and left / right column of groups) run as
one-dimensional jobs - their index-clamped taps make the upsampled logit constant along one axis, so the kernel evaluates
16 pixels per class instead of 256 and sums the U tile along the constant axis before the class phase.  These cases aim
at what that path can get wrong, against the split K2 / K3 kernels (which keep the 2-D border handling) and the float64
oracle: shapes where border groups dominate, first-class ties across the half-warp split inside edge and corner groups,
labels that leave the border band ignored, and slow (wide-range or non-finite) groups next to fast border groups."""
import pytest
import torch
import torch.nn.functional as F

from oracle import head_oracle as O
from lc2is_b200 import ops, synthetic
from test_gpu_k23_jobs import _check

pytestmark = pytest.mark.gpu
DEV = "cuda"
S = 16


@pytest.mark.parametrize("N,C,h,w", [(2, 150, 1, 1), (2, 150, 1, 4), (2, 150, 1, 5), (2, 150, 2, 1), (1, 150, 2, 2),
                                     (2, 40, 2, 8), (1, 151, 2, 7), (2, 24, 5, 2), (1, 3, 1, 2), (2, 200, 2, 4)])
def test_border_dominated_shapes(N, C, h, w):
    """h or w of 1 (every group is a border group; 1 x 1: four corners) and 2 (one row or column of interior groups),
    non-square, with and without TMA staging (w % 4)."""
    low = synthetic.make_dyadic_logits(N, C, h, w)
    labels = synthetic.make_labels(N, S * h, S * w, C, block=8, ignore_frac=0.1)
    labels[0, :3] = C + 3
    _check(low, labels, 0)


def test_ties_across_the_half_warp_split_in_edge_and_corner_groups():
    """C = 150: the lower half-warp sweeps classes 0..75, the upper 76..151.  Equal maxima are placed on the cells that
    border groups interpolate, so whole edge / corner regions are exact ties between the two halves."""
    N, C, h, w = 2, 150, 4, 4
    low = synthetic.make_dyadic_logits(N, C, h, w)
    top = float(low.max()) + 1.0
    low[0, 10, 0, 0] = top; low[0, 100, 0, 0] = top                          # top-left corner
    low[0, 75, 0, 1:3] = top; low[0, 76, 0, 1:3] = top                        # top edge group kx = 1
    low[0, 74, 1:3, w - 1] = top; low[0, 148, 1:3, w - 1] = top               # right edge group ky = 1
    low[1, 5, h - 1, w - 1] = top; low[1, 149, h - 1, w - 1] = top + 0.25     # bottom-right: upper half strictly larger
    low[1, 20, 1:3, 0] = top; low[1, 120, 1:3, 0] = top; low[1, 3, 1:3, 0] = top   # left edge: three-way tie
    labels = synthetic.make_labels(N, S * h, S * w, C, block=8, ignore_frac=0.1)
    pred = _check(low, labels, 0)
    assert bool((pred[0, :8, :8] == 10).all())
    assert bool((pred[0, :8, 24:40] == 75).all())
    assert bool((pred[0, 24:40, -8:] == 74).all())
    assert bool((pred[1, -8:, -8:] == 149).all())
    assert bool((pred[1, 24:40, :8] == 3).all())


def test_ignored_and_out_of_range_labels_in_the_border_band():
    """The outer 8-pixel band (the pixels of the border groups) carries only ignored / out-of-range labels in image 0
    (border jobs count nothing and send no gradient) and a mix in image 1."""
    N, C, h, w = 2, 150, 4, 6
    H, W = S * h, S * w
    low = synthetic.make_dyadic_logits(N, C, h, w)
    labels = synthetic.make_labels(N, H, W, C, block=8, ignore_frac=0.05)
    band = torch.ones(H, W, dtype=torch.bool)
    band[8:H - 8, 8:W - 8] = False
    labels[0][band] = 0
    labels[0, :8, :W // 2] = C + 7
    g = torch.Generator().manual_seed(5)
    mix = band & (torch.rand(H, W, generator=g) < 0.5)
    labels[1][mix] = torch.where(torch.rand(H, W, generator=g) < 0.5, 0, C + 2)[mix]
    _check(low, labels, 0)


@pytest.mark.parametrize("w", [4, 5])
def test_wide_range_border_and_interior_groups(w):
    """A wide tap range on a border cell (slow border groups next to fast interior and border groups) and inside the
    map (slow interior groups next to fast border groups)."""
    N, C, h = 2, 150, 5
    low = synthetic.make_dyadic_logits(N, C, h, w)
    low[0, 37, 0, 2] = 60.0                                   # top edge
    low[0, 3, h - 1, w - 1] = -50.0                           # bottom-right corner
    low[1, 120, 2, 2] = 45.0                                  # interior only
    labels = synthetic.make_labels(N, S * h, S * w, C, block=8, ignore_frac=0.1)
    _check(low, labels, 0)


def test_non_finite_border_and_interior_groups():
    """+inf / NaN taps poison exactly the pixels that interpolate them (class 0), whether the group is a border group
    or an interior group next to fast border groups; the NaN in row 1 / column 1 is the hidden second tap (weight 0) of
    the top / left border groups, which the staged cells do not contain."""
    N, C, h, w = 3, 40, 4, 4
    H, W = S * h, S * w
    low = synthetic.make_dyadic_logits(N, C, h, w)
    low[0, 7, 0, 2] = float("inf")                            # top edge
    low[0, 9, 3, 0] = float("nan")                            # bottom-left corner
    low[1, 11, 1, 2] = float("nan")                           # interior, hidden tap of the top edge group kx = 2 ...
    low[1, 4, 2, 1] = float("-inf")                           # interior, hidden tap of the left edge group ky = 1
    low[2, 30, 1, 0] = float("nan")                           # hidden tap of the top-left corner group
    low[2, 2, 0, 1] = float("nan")
    labels = synthetic.make_labels(N, H, W, C, block=8)
    up = F.interpolate(low, mode="bilinear", scale_factor=S)
    pred_ref = O.argmax_reference(up)
    _, _, _, packed = ops.upsample_ce_split(low.to(DEV), labels.to(DEV), 0, want_grad=False)
    ls = torch.zeros(1, dtype=torch.float64, device=DEV)
    cm, _, pred = ops.ce_argmax_fused(low.to(DEV), packed, (H, W), ls, None, want_pred=True)
    cm3, _, pred3 = ops.argmax_confmat_packed(low.to(DEV), packed, (H, W), want_pred=True)
    assert torch.equal(pred, pred3)
    assert torch.equal(pred.cpu(), pred_ref)
    assert torch.equal(cm.cpu(), O.confusion_matrix(pred_ref, labels, C))
    assert torch.equal(cm, cm3)
