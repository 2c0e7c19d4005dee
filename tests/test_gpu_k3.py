"""K3 parity (bit-exact integer work) through the C ABI, against the CPU oracle."""
import os

import pytest
import torch
import torch.nn.functional as F

from oracle import head_oracle as O
from lc2is_b200 import metrics, ops, synthetic, utils

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _per_image_ref(pred, lab, C):
    out = torch.zeros(pred.shape[0], 3, C, dtype=torch.int64)
    for n in range(pred.shape[0]):
        cm = O.confusion_matrix(pred[n], lab[n], C)
        out[n, 0] = torch.diag(cm); out[n, 1] = cm.sum(1); out[n, 2] = cm.sum(0)
    return out


@pytest.mark.parametrize("N,C,H,W,dtype", [
    (3, 151, 64, 64, torch.float32),
    (2, 150, 128, 96, torch.float32),
    (2, 151, 64, 64, torch.bfloat16),
    (1, 7, 33, 31, torch.float32),        # ragged: HW not a multiple of 4 -> scalar path
    (1, 7, 33, 31, torch.bfloat16),
    (2, 300, 32, 32, torch.float32),      # C*C too large for the shared histogram -> global atomics
    (1, 1, 16, 16, torch.float32),
])
def test_full_res_confmat_bit_exact(N, C, H, W, dtype):
    g = torch.Generator().manual_seed(5)
    logits = torch.randn(N, C, H, W, generator=g).to(dtype)
    labels = torch.randint(0, C, (N, H, W), generator=g)
    labels[0, :2] = C + 3                                    # out-of-range targets are skipped
    labels[0, 2, :4] = -1
    pred_ref = O.argmax_logits(logits.float())
    cm, pi, pred = ops.argmax_confmat(logits.to(DEV), labels.to(DEV), per_image=True, want_pred=True)
    assert torch.equal(pred.cpu(), pred_ref)
    assert torch.equal(cm.cpu(), O.confusion_matrix(pred_ref, labels, C))
    assert torch.equal(pi.cpu(), _per_image_ref(pred_ref, labels, C))


def test_ties_first_index_and_nan():
    C = 9
    x = torch.zeros(1, C, 8, 8)
    x[0, 4] = 1.0; x[0, 6] = 1.0                              # tie -> first index (4)
    x[0, :, 0, 0] = float("nan")                               # NaN row -> class 0 (argmax(softmax) of all-NaN)
    x[0, 2, 1, 1] = float("inf")                               # +inf -> softmax is NaN everywhere -> class 0
    x[0, :, 2, 2] = float("-inf")                              # all -inf -> NaN -> 0
    labels = torch.full((1, 8, 8), 4, dtype=torch.int64)
    _, _, pred = ops.argmax_confmat(x.to(DEV), labels.to(DEV), want_pred=True)
    assert torch.equal(pred.cpu(), O.argmax_reference(x))


def test_accumulates_and_empty_batch():
    C = 5
    g = torch.Generator().manual_seed(6)
    logits = torch.randn(2, C, 16, 16, generator=g)
    labels = torch.randint(0, C, (2, 16, 16), generator=g)
    cm, _, _ = ops.argmax_confmat(logits.to(DEV), labels.to(DEV))
    cm, _, _ = ops.argmax_confmat(logits.to(DEV), labels.to(DEV), confmat=cm)
    assert torch.equal(cm.cpu(), 2 * O.confusion_matrix(O.argmax_logits(logits), labels, C))
    cm0, _, _ = ops.argmax_confmat(torch.zeros(0, C, 4, 4, device=DEV), torch.zeros(0, 4, 4, dtype=torch.int64, device=DEV))
    assert int(cm0.sum()) == 0


@pytest.mark.parametrize("s,h", [(4, 16), (16, 4), (8, 8)])
def test_fused_bilinear_dyadic_bit_exact(s, h):
    """Exactness set: bilinear xs of k/256 logits is exact in fp32 in any order -> bit-exact argmax."""
    N, C = 2, 151
    low = synthetic.make_dyadic_logits(N, C, h, h)
    H = s * h
    labels = synthetic.make_labels(N, H, H, C, block=8)
    up = F.interpolate(low, mode="bilinear", scale_factor=s)
    pred_ref = O.argmax_reference(up)
    cm, pi, pred = ops.argmax_confmat(low.to(DEV), labels.to(DEV), per_image=True, want_pred=True,
                                      size=(H, H), mode="bilinear")
    assert torch.equal(pred.cpu(), pred_ref)
    assert torch.equal(cm.cpu(), O.confusion_matrix(pred_ref, labels, C))
    assert torch.equal(pi.cpu(), _per_image_ref(pred_ref, labels, C))


def _safe_mask(up, tol):
    top2 = up.topk(2, dim=1).values
    return (top2[:, 0] - top2[:, 1]) > tol


@pytest.mark.parametrize("mode,s,h,H", [("bicubic", 4, 16, 64), ("bilinear", 4, 16, 64), ("bicubic", 16, 4, 64),
                                         ("bicubic", None, 13, 37), ("bilinear", None, 13, 37),
                                         ("bicubic", None, 16, 32)])
def test_fused_resize_argmax_tie_safe(mode, s, h, H):
    """Random fp32 logits: the fused kernel may differ from ATen only in fp32 evaluation order, so the
    argmax must agree on every pixel whose top-2 gap exceeds 1e-4 (SURVEY 7, 'bit-exact argmax')."""
    N, C = 2, 23
    g = torch.Generator().manual_seed(8)
    low = torch.randn(N, C, h, h, generator=g)
    up = F.interpolate(low, mode=mode, size=(H, H))
    labels = torch.randint(0, C, (N, H, H), generator=g)
    pred_ref = O.argmax_reference(up)
    _, _, pred = ops.argmax_confmat(low.to(DEV), labels.to(DEV), want_pred=True, size=(H, H), mode=mode)
    safe = _safe_mask(up, 1e-4)
    assert safe.float().mean() > 0.99
    assert torch.equal(pred.cpu()[safe], pred_ref[safe])


def test_labels_nearest_upsampled_in_kernel():
    """metrics.py:90: labels at the low grid, nearest x4."""
    N, C, h = 2, 11, 8
    low = synthetic.make_dyadic_logits(N, C, h, h)
    lab = torch.randint(0, C, (N, h, h), generator=torch.Generator().manual_seed(2))
    up = F.interpolate(low, mode="bilinear", scale_factor=4)
    labu = F.interpolate(lab.view(-1, 1, h, h).float(), mode="nearest", scale_factor=4).squeeze(1).long()
    cm, _, _ = ops.argmax_confmat(low.to(DEV), lab.to(DEV), size=(4 * h, 4 * h), mode="bilinear")
    assert torch.equal(cm.cpu(), O.confusion_matrix(O.argmax_reference(up), labu, C))


def test_metrics_api_matches_oracle_and_golden(golden_dir):
    g = torch.load(os.path.join(golden_dir, "metrics_small.pt"))
    C = g["outputs"].shape[1]
    got = metrics.compute_mIOU(g["outputs"], g["labels"], n_cls=C, ignore_index=0)     # CPU tensors in
    assert abs(got["mIOU_label"] - g["miou_label"]) < 1e-6
    up = F.interpolate(g["outputs"], mode="bicubic", scale_factor=4)
    lab = g["labels"].repeat_interleave(4, 1).repeat_interleave(4, 2)
    assert abs(metrics.compute_mIOU_tensor(up, lab, C, 0) - g["miou_global"]) < 1e-6
    cm = metrics.confusion_matrix(up.to(DEV), lab.to(DEV))
    assert torch.equal(cm.cpu(), g["confmats"].sum(0))
    # ragged ground truth (compute_gt_mIOU / segmentation_metrics / generate_masks)
    sizes = torch.tensor([[20, 28], [31, 17], [24, 24]])
    gt = [torch.randint(0, C, (int(a), int(b)), generator=torch.Generator().manual_seed(i)) for i, (a, b) in enumerate(sizes)]
    ref = O.compute_gt_mIOU(g["outputs"], gt, sizes, n_cls=C, ignore_index=0)["mIOU_gt"]
    got = metrics.segmentation_metrics(g["outputs"], g["labels"], gt, sizes, n_clas=C, ignore_index=0)
    assert abs(got["mIOU_gt"] - ref) < 1e-6 and abs(got["mIOU_label"] - g["miou_label"]) < 1e-6
    masks = utils.generate_masks(g["outputs"], sizes)
    for m, r in zip(masks, O.generate_masks(g["outputs"], sizes)):
        assert m.dtype == torch.int64 and torch.equal(m.cpu(), r)


def test_full_size_property_checksum():
    """BASELINE size (512^2, C=150): row sums of the confusion matrix == label histogram, column sums ==
    prediction histogram, total == pixel count; fused-from-low == materialised on dyadic logits."""
    N, C, h, H = 4, 150, 128, 512
    low = synthetic.make_dyadic_logits(N, C, h, h).to(DEV)
    labels = synthetic.make_labels(N, H, H, C).to(DEV)
    cm_f, _, pred = ops.argmax_confmat(low, labels, want_pred=True, size=(H, H), mode="bilinear")
    up = F.interpolate(low, mode="bilinear", scale_factor=4)
    cm_m, _, pred_m = ops.argmax_confmat(up, labels, want_pred=True)
    assert torch.equal(cm_f, cm_m) and torch.equal(pred, pred_m)
    assert torch.equal(pred_m, up.argmax(1))
    assert int(cm_f.sum()) == N * H * H
    assert torch.equal(cm_f.sum(1), torch.bincount(labels.flatten(), minlength=C))
    assert torch.equal(cm_f.sum(0), torch.bincount(pred.flatten(), minlength=C))


@pytest.mark.parametrize("s,h,C,ign", [(16, 6, 151, 0), (8, 12, 150, 0), (16, 3, 19, 5), (16, 5, 847, 0)])
def test_strip_kernel_packed_labels_bit_exact(s, h, C, ign):
    """k3_strip_kernel through the packed labels of the CE label prepass (what HeadStep runs): the matrix keeps
    the ignore_index row (bit 15 of the packed label only switches the pixel off for the cross-entropy) and
    skips labels outside [0,C); dyadic logits -> bit-exact against the oracle."""
    N = 3
    low = synthetic.make_dyadic_logits(N, C, h, h)
    H = s * h
    labels = synthetic.make_labels(N, H, H, C, block=8, ignore_frac=0.1, ignore_index=ign)
    labels[0, :2] = C + 3
    labels[1, 5, :7] = -1
    up = F.interpolate(low, mode="bilinear", scale_factor=s)
    pred_ref = O.argmax_reference(up)
    _, _, _, packed = ops.upsample_ce_split(low.to(DEV), labels.to(DEV), ign, want_grad=False)
    cm, pi, pred = ops.argmax_confmat_packed(low.to(DEV), packed, (H, H), per_image=True, want_pred=True)
    assert torch.equal(pred.cpu(), pred_ref)
    assert torch.equal(cm.cpu(), O.confusion_matrix(pred_ref, labels, C))
    assert torch.equal(pi.cpu(), _per_image_ref(pred_ref, labels, C))
    # and the int64-label entry (same kernel) agrees
    cm2, _, pred2 = ops.argmax_confmat(low.to(DEV), labels.to(DEV), want_pred=True, size=(H, H), mode="bilinear")
    assert torch.equal(cm2, cm) and torch.equal(pred2, pred)


def test_strip_kernel_non_finite_taps_and_ties():
    """+inf / NaN taps poison exactly the pixels that interpolate them (class 0, like argmax(softmax)); equal
    logits resolve to the first class, also across the 8-class chunks of the two-phase argmax."""
    N, C, h, s = 1, 21, 4, 16
    H = s * h
    low = torch.zeros(N, C, h, h)
    low[0, 3] = 0.5; low[0, 12] = 0.5; low[0, 20] = 0.5        # ties across chunks 0, 1, 2 -> class 3
    low[0, 7, 1, 1] = float("inf")
    low[0, 9, 2, 3] = float("nan")
    labels = torch.randint(0, C, (N, H, H), generator=torch.Generator().manual_seed(3))
    up = F.interpolate(low, mode="bilinear", scale_factor=s)
    pred_ref = O.argmax_reference(up)
    cm, _, pred = ops.argmax_confmat(low.to(DEV), labels.to(DEV), want_pred=True, size=(H, H), mode="bilinear")
    assert torch.equal(pred.cpu(), pred_ref)
    assert torch.equal(cm.cpu(), O.confusion_matrix(pred_ref, labels, C))


@pytest.mark.parametrize("N,C,h,ign,frac", [(3, 151, 6, 0, 0.1), (2, 150, 32, 0, 0.1), (1, 19, 3, 5, 0.3), (5, 37, 5, 0, 0.0),
                                               (3, 151, 8, 0, 0.1), (1, 19, 4, 5, 0.3), (2, 40, 12, 0, 0.2), (1, 200, 4, 0, 0.1)])
def test_fused_ce_argmax_kernel_matches_separate_kernels_and_oracle(N, C, h, ign, frac):
    """k23_rc_kernel (x16): the fused K2+K3 kernel gives the loss / gradient of the split K2 path and
    the bit-exact confusion matrix / per-image counts / masks of K3 (dyadic logits)."""
    s = 16
    H = s * h
    low = synthetic.make_dyadic_logits(N, C, h, h)
    labels = synthetic.make_labels(N, H, H, C, block=8, ignore_frac=frac, ignore_index=ign)
    labels[0, :2] = C + 3
    dl, dlab = low.to(DEV), labels.to(DEV)
    loss_sum, n_valid, grad, packed = ops.upsample_ce_split(dl, dlab, ign)           # separate kernels
    assert ops._lib.lib.lc2is_ce_argmax_fused_supported(C, h, h, H, H)
    ls2 = torch.zeros(1, dtype=torch.float64, device=DEV)
    g2 = torch.zeros_like(dl)
    packed2, nv2 = ops.pack_labels(dlab, C, ign)                 # pack + count only; -onehot comes from the argmax warps
    assert torch.equal(packed2, packed) and int(nv2) == int(n_valid)
    nv3 = torch.zeros(1, dtype=torch.int64, device=DEV)
    cm, pi, pred = ops.ce_argmax_fused(dl, packed2, (H, H), ls2, g2, per_image=True, want_pred=True, onehot=True,
                                       n_valid=nv3)
    assert int(nv3) == int(n_valid)                              # the CE warps' own count (host-packed labels)
    assert abs(float(ls2) - float(loss_sum)) <= 1e-6 * abs(float(loss_sum))
    assert float((g2 - grad).abs().max()) <= 1e-5 * float(grad.abs().max())
    up = F.interpolate(low, mode="bilinear", scale_factor=s)
    pred_ref = O.argmax_reference(up)
    assert torch.equal(pred.cpu(), pred_ref)
    assert torch.equal(cm.cpu(), O.confusion_matrix(pred_ref, labels, C))
    assert torch.equal(pi.cpu(), _per_image_ref(pred_ref, labels, C))
    ref_loss, ref_grad, nv = O.auxiliary_loss_and_grad(low, torch.where((labels >= 0) & (labels < C), labels, torch.full_like(labels, ign)), ign)
    assert abs(float(ls2) / nv - float(ref_loss)) <= 2e-6 * abs(float(ref_loss))
    assert float((g2.cpu() / nv - ref_grad).abs().max()) <= 1e-5 * float(ref_grad.abs().max()) + 1e-9


def test_fused_kernel_non_finite_taps():
    N, C, h, s = 1, 21, 4, 16
    H = s * h
    low = torch.zeros(N, C, h, h)
    low[0, 3] = 0.5; low[0, 12] = 0.5; low[0, 20] = 0.5
    low[0, 7, 1, 1] = float("inf")
    low[0, 9, 2, 3] = float("nan")
    labels = torch.randint(0, C, (N, H, H), generator=torch.Generator().manual_seed(3))
    up = F.interpolate(low, mode="bilinear", scale_factor=s)
    pred_ref = O.argmax_reference(up)
    _, _, _, packed = ops.upsample_ce_split(low.to(DEV), labels.to(DEV), 0, want_grad=False)
    ls = torch.zeros(1, dtype=torch.float64, device=DEV)
    cm, _, pred = ops.ce_argmax_fused(low.to(DEV), packed, (H, H), ls, None, want_pred=True)
    assert torch.equal(pred.cpu(), pred_ref)
    assert torch.equal(cm.cpu(), O.confusion_matrix(pred_ref, labels, C))


# ---------------------------------------------------------------------------------------------------------------------
# The reference's rule on BASELINE-shaped data: metrics.py:92 takes argmax(Softmax2d(x)), the kernels argmax(x).  In
# fp32 the softmax can round a near-tie onto one value and then the FIRST of the merged classes wins, so the two differ
# on a handful of pixels (SURVEY 7: ~2e-6 of them on cosine logits).  These tests state the bound and what a differing
# pixel must look like: the kernel's class IS the argmax of the logits, the reference's class is an earlier class whose
# softmax value the fp32 softmax made equal (materialised input) / whose logit is within fp32 evaluation-order noise
# (fused resize, where ATen and the kernel round the interpolation differently).
def _cosine_low(B, h, C, seed=11):
    v = synthetic.make_patch_embeddings(B, h * h, 512, seed=seed)
    t = synthetic.make_prototypes(C, 512)
    return O.cosine_logits_bf16_operands(v, t, hw_shape=(h, h))


def _check_rule(pred, up, max_frac, gap_tol):
    """pred (kernel) vs argmax(softmax(up)) (reference): few differing pixels, each a near-tie."""
    pred_ref = O.argmax_reference(up)
    diff = (pred != pred_ref)
    n_diff = int(diff.sum())
    assert n_diff <= max_frac * pred.numel(), (n_diff, pred.numel())
    if n_diff:
        idx = diff.nonzero()
        x = up[idx[:, 0], :, idx[:, 1], idx[:, 2]]                                   # [n_diff, C]
        vk = x.gather(1, pred[diff].view(-1, 1)).squeeze(1)
        vr = x.gather(1, pred_ref[diff].view(-1, 1)).squeeze(1)
        top = x.max(1).values
        assert float((top - vk).abs().max()) <= gap_tol and float((top - vr).abs().max()) <= gap_tol
    return n_diff


def test_argmax_rule_vs_reference_softmax_materialised():
    """(i) materialised [2,150,512,512] bilinear-upsampled bf16-operand cosine logits: the kernel sees the SAME fp32
    tensor as the reference, so a differing pixel can only be a softmax-merged near-tie and the kernel's class is the
    exact argmax of the logits."""
    B, C, h, H = 2, 150, 32, 512
    up = F.interpolate(_cosine_low(B, h, C), mode="bilinear", scale_factor=H // h)
    labels = synthetic.make_labels(B, H, H, C)
    _, _, pred = ops.argmax_confmat(up.to(DEV), labels.to(DEV), want_pred=True)
    pred = pred.cpu()
    assert torch.equal(pred, O.argmax_logits(up))                                    # the kernel's own rule, bit-exact
    n = _check_rule(pred, up, 2e-5, 2.0 ** -22)
    ref = O.argmax_reference(up)
    d = pred != ref
    if n:                                                                            # the reference picked an EARLIER class
        assert bool((ref[d] < pred[d]).all())


@pytest.mark.parametrize("s,h", [(16, 32), (4, 128)])
def test_argmax_rule_vs_reference_softmax_fused_bilinear(s, h):
    """(ii) fused bilinear x16 / x4 from the low-resolution cosine logits against argmax(softmax(interpolate(x)))."""
    B, C = 2, 150
    H = s * h
    low = _cosine_low(B, h, C, seed=12)
    up = F.interpolate(low, mode="bilinear", scale_factor=s)
    labels = synthetic.make_labels(B, H, H, C)
    cm, _, pred = ops.argmax_confmat(low.to(DEV), labels.to(DEV), want_pred=True, size=(H, H), mode="bilinear")
    _check_rule(pred.cpu(), up, 2e-5, 1e-6)
    assert int(cm.sum()) == B * H * H
    if s == 16:                                                                      # the fused K2+K3 kernel's argmax
        packed, _ = ops.pack_labels(labels.to(DEV), C, 0)
        ls = torch.zeros(1, dtype=torch.float64, device=DEV)
        _, _, pred2 = ops.ce_argmax_fused(low.to(DEV), packed, (H, H), ls, None, want_pred=True)
        _check_rule(pred2.cpu(), up, 2e-5, 1e-6)


def test_argmax_rule_vs_reference_softmax_bicubic_compute_miou():
    """(iii) the compute_mIOU path at size: bicubic x4, C=151, 128^2 -> 512^2 (metrics.py:89-92)."""
    N, C, h, s = 2, 151, 128, 4
    H = s * h
    low = _cosine_low(N, h, C, seed=13)
    labels = synthetic.make_labels(N, h, h, C, block=4)                              # labels at 128^2, nearest x4 (metrics.py:90)
    up = F.interpolate(low, mode="bicubic", scale_factor=s)
    lab_up = F.interpolate(labels[:, None].float(), mode="nearest", scale_factor=s)[:, 0].long()
    _, _, pred = ops.argmax_confmat(low.to(DEV), lab_up.to(DEV), want_pred=True, size=(H, H), mode="bicubic")
    n = _check_rule(pred.cpu(), up, 2e-5, 1e-6)
    got = metrics.compute_mIOU(low, labels, C)["mIOU_label"]
    ref = O.compute_mIOU(low, labels, C)["mIOU_label"]
    assert abs(got - ref) <= 1e-5 + 4.0 * n / (H * H), (got, ref, n)                 # exact when no pixel differs


def test_bf16_dominant_class_does_not_overflow_the_16bit_counters():
    """One (target, prediction) pair takes every pixel and a CTA sees > 65535 of them between image boundaries: the
    shared-memory counters are 16 bit and must be flushed on PIXELS (a bf16 item is 2048 pixels, an fp32 one 1024)."""
    N, C, H = 1, 4, 4096                                                              # 16.7 M pixels in one image
    logits = torch.zeros(N, C, H, H, dtype=torch.bfloat16, device=DEV)
    logits[:, 2] = 1.0
    labels = torch.full((N, H, H), 1, dtype=torch.int64, device=DEV)
    cm, _, _ = ops.argmax_confmat(logits, labels)
    ref = torch.zeros(C, C, dtype=torch.int64)
    ref[1, 2] = N * H * H
    assert torch.equal(cm.cpu(), ref)


# ---- ragged batch in one launch (lc2is_argmax_confmat_ragged; metrics.py:61-79, utils.py:15-22) -----------------------
def _ragged_case(N, C, h, sizes, seed, nonfinite=False):
    g = torch.Generator().manual_seed(seed)
    low = torch.randn(N, C, h, h, generator=g)
    if nonfinite:
        low[0, 3, 2, 5] = float("inf")
        low[1, 0, h - 1, 0] = float("nan")
        low[1, 4, 0, h - 1] = float("-inf")
    gt = [torch.randint(0, C, (a, b), generator=g) for a, b in sizes]
    gt[0][0, :3] = C + 5                                     # targets outside [0, C) are skipped
    return low, gt


@pytest.mark.parametrize("mode", ["bicubic", "bilinear"])
@pytest.mark.parametrize("nonfinite", [False, True])
def test_ragged_kernel_equals_the_per_image_kernel(mode, nonfinite):
    """One launch over the descriptor table == one lc2is_argmax_confmat_lowres call per image (k3_low_gen_kernel, the
    per-pixel ATen-order chains), bit for bit: masks, per-image counts and the confusion matrix.  Sizes: enlarged >= 3x
    (5-wide window), 1.5x - 3x (6-wide window), shrunk / barely enlarged (exact per-pixel path), single pixels, sizes
    that are not multiples of the 4 x 4 blocks or the 64 x 32 tiles."""
    C, h = 23, 16
    sizes = [(64, 64), (71, 50), (37, 90), (24, 31), (17, 19), (16, 16), (9, 7), (1, 1), (130, 67), (48, 3)]
    N = len(sizes)
    low, gt = _ragged_case(N, C, h, sizes, 11, nonfinite)
    flat = torch.cat([t.reshape(-1) for t in gt])
    cm = torch.zeros(C, C, dtype=torch.int64, device=DEV)
    _, pi, pred, desc = ops.argmax_confmat_ragged(low.to(DEV), sizes, flat.to(DEV), mode=mode, confmat=cm, want_pred=True)
    cm_ref = torch.zeros(C, C, dtype=torch.int64, device=DEV)
    for i, (H, W) in enumerate(sizes):
        _, pi_i, pred_i = ops.argmax_confmat(low[i:i + 1].to(DEV), gt[i].view(1, H, W).to(DEV), confmat=cm_ref,
                                             per_image=True, want_pred=True, size=(H, W), mode=mode)
        o = int(desc[i, 0])
        assert torch.equal(pred[o:o + H * W].view(H, W), pred_i[0]), (i, H, W)
        assert torch.equal(pi[i], pi_i[0]), (i, H, W)
    assert torch.equal(cm, cm_ref)
    assert int(cm.sum()) == sum(a * b for a, b in sizes) - 3


def test_ragged_kernel_vs_oracle_tie_safe_and_miou():
    """Against the reference lines on CPU (oracle): masks agree wherever the top-2 gap exceeds the fp32 evaluation-order
    noise, and compute_gt_mIOU / generate_masks through the mirror give the oracle's numbers."""
    C, h = 151, 32
    sizes = [(128, 128), (171, 96), (100, 133), (97, 255)]
    low, gt = _ragged_case(len(sizes), C, h, sizes, 5)
    for t in gt:
        t.clamp_(max=C - 1)
    masks = utils.generate_masks(low, torch.tensor(sizes))
    for i, (H, W) in enumerate(sizes):
        up = F.interpolate(low[i:i + 1], mode="bicubic", size=(H, W))
        safe = _safe_mask(up, 1e-4)[0]
        assert safe.float().mean() > 0.99
        assert torch.equal(masks[i].cpu()[safe], O.argmax_reference(up)[0][safe])
    ref = O.compute_gt_mIOU(low, gt, sizes, n_cls=C, ignore_index=0)["mIOU_gt"]
    got = metrics.compute_gt_mIOU(low, gt, torch.tensor(sizes), n_cls=C, ignore_index=0)["mIOU_gt"]
    assert abs(got - ref) < 2e-4                              # a handful of near-tie pixels out of 80 k


def test_ragged_entry_rejects_bad_arguments():
    low = torch.zeros(1, 3, 4, 4, device=DEV)
    with pytest.raises(Exception):
        ops.argmax_confmat_ragged(low, [(8, 8), (4, 4)], None, want_pred=True)          # one size per image
    with pytest.raises(Exception):
        ops.argmax_confmat_ragged(low, [(8, 8)], torch.zeros(3, dtype=torch.int64, device=DEV))   # label count


@pytest.mark.parametrize("mode", ["bilinear", "bicubic"])
def test_x4_block_kernel_non_finite_taps(mode):
    """k3_low_fast_kernel (x4): +-inf / NaN taps poison exactly the pixels they poison in argmax(softmax(interpolate(x)))
    (class 0) - the bilinear kernel detects them inside its class loop and re-evaluates the warp exactly."""
    g = torch.Generator().manual_seed(14)
    N, C, h = 2, 13, 12
    low = torch.randn(N, C, h, h, generator=g)
    low[0, 3, 4, 5] = float("inf")
    low[0, 7, 9, 2] = float("-inf")
    low[1, 0, 6, 6] = float("nan")
    low[1, 12, 11, 11] = float("inf")                       # corner cell (clamped taps)
    labels = torch.randint(0, C, (N, 4 * h, 4 * h), generator=g)
    up = F.interpolate(low, mode=mode, scale_factor=4)
    ref = O.argmax_reference(up)
    cm, _, pred = ops.argmax_confmat(low.to(DEV), labels.to(DEV), want_pred=True, size=(4 * h, 4 * h), mode=mode)
    finite = torch.isfinite(up).all(1)
    safe = _safe_mask(torch.nan_to_num(up, nan=0.0, posinf=0.0, neginf=0.0), 1e-4) | ~finite
    assert torch.equal(pred.cpu()[safe], ref[safe])
    assert (~finite).sum() > 0 and int(cm.sum()) == labels.numel()
