"""K2 weighted form: class weights and label smoothing in the fused bilinear-upsample + softmax-CE kernels
(UpsampledCrossEntropyLoss, SegHeadLoss(weight=, label_smoothing=), lc2is_upsample_ce_fwd_bwd_ex) against torch's own
F.cross_entropy on the float64 upsampled map (tests/ce_weighted_reference.py), at the tolerances of test_gpu_k2.py:
loss rel 2e-6, gradient <= 1e-5 * max|grad| (1e-5 / 1e-4 where the exact per-pixel slow paths run)."""
import ctypes

import pytest
import torch
import torch.nn.functional as F

from ce_weighted_reference import upsample_ce_and_grad
from oracle import head_oracle as O
from lc2is_b200 import _lib, head, ops, synthetic
from lc2is_b200.model import AuxiliaryLoss

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _check(loss, grad, ref_loss, ref_grad, loss_rtol=2e-6, g_rtol=1e-5):
    ref_loss, ref_grad = float(ref_loss), ref_grad.float()
    if ref_loss != ref_loss:                    # torch's 0/0: every counted pixel has weight 0
        assert float(loss) != float(loss) and not bool(torch.isfinite(grad).all()), float(loss)
        return
    assert abs(float(loss) - ref_loss) <= loss_rtol * abs(ref_loss) + 1e-7, (float(loss), ref_loss)
    tol = g_rtol * float(ref_grad.abs().max()) + 1e-9
    err = float((grad.float().cpu() - ref_grad).abs().max())
    assert err <= tol, (err, tol)


def _weight(C, seed=5):
    g = torch.Generator().manual_seed(seed)
    w = 0.2 + 2.8 * torch.rand(C, generator=g)
    w[C // 3] = 0.0
    return w


def _run(low, labels, ign, weight, eps, reduction, g_out=0.4):
    crit = head.UpsampledCrossEntropyLoss(weight=weight, ignore_index=ign, reduction=reduction,
                                          label_smoothing=eps).to(DEV)
    x = low.to(DEV).requires_grad_(True)
    loss = crit(x, labels.to(DEV))
    (loss * g_out).backward()
    return loss, x.grad


# (B, C, h, w, H, W, ignore_frac): every path of the one-call K2
SHAPES = {
    "x4": (2, 151, 32, 32, 128, 128, 0.1),
    "x8": (1, 151, 16, 16, 128, 128, 0.0),
    "x16": (2, 150, 8, 8, 128, 128, 0.0),
    "x16_c847_gtaps": (1, 847, 4, 4, 64, 64, 0.0),
    "generic_c847": (1, 847, 8, 8, 32, 32, 0.0),
    "generic_noninteger": (2, 5, 12, 12, 40, 40, 0.3),
    "single_pixel": (1, 3, 1, 1, 4, 4, 0.0),          # one label (class 1): weighted, it has weight 0 - torch's NaN
    "single_pixel_x16": (1, 3, 1, 1, 16, 16, 0.0),    # mixed labels: every tap clamps
    "nonsquare_x16": (2, 37, 8, 12, 128, 192, 0.1),
}


@pytest.mark.parametrize("reduction", ["mean", "sum"])
@pytest.mark.parametrize("ign", [0, -100])
@pytest.mark.parametrize("eps", [0.0, 0.1])
@pytest.mark.parametrize("weighted", [False, True])
@pytest.mark.parametrize("shape", list(SHAPES))
def test_weighted_vs_oracle(shape, weighted, eps, ign, reduction):
    B, C, h, w, H, W, frac = SHAPES[shape]
    g = torch.Generator().manual_seed(61)
    low = torch.randn(B, C, h, w, generator=g) * 2.0
    labels = synthetic.make_labels(B, H, W, C, block=8, ignore_frac=frac, ignore_index=max(ign, 0))
    weight = _weight(C) if weighted else None
    ref_loss, ref_grad = upsample_ce_and_grad(low, labels, ign, weight, eps, reduction)
    loss, grad = _run(low, labels, ign, weight, eps, reduction)
    _check(loss, grad, ref_loss, 0.4 * ref_grad)


def _kernel_names(fn):
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return sorted(e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA
                  and "k2_" in e.name)


@pytest.mark.parametrize("shape", ["x4", "x8", "x16", "generic_noninteger"])
def test_ex_without_options_is_the_unweighted_call(shape):
    """weight=NULL, eps=0: _ex launches the unweighted kernels; loss_sum bit for bit, the gradient up to the order of
    its float atomics."""
    B, C, h, w, H, W, frac = SHAPES[shape]
    g = torch.Generator().manual_seed(62)
    low = (torch.randn(B, C, h, w, generator=g) * 2.0).to(DEV)
    labels = synthetic.make_labels(B, H, W, C, block=8, ignore_frac=frac).to(DEV)
    gs = torch.tensor([0.37], device=DEV)
    outs = {}

    def call(ex):
        ls = torch.zeros(1, dtype=torch.float64, device=DEV)
        grad = torch.empty_like(low)
        st = _lib.stream_ptr()
        if ex:
            rc = _lib.lib.lc2is_upsample_ce_fwd_bwd_ex(low.data_ptr(), labels.data_ptr(), B, C, h, w, H, W, 0, None,
                                                       ctypes.c_float(0.0), gs.data_ptr(), ls.data_ptr(),
                                                       grad.data_ptr(), None, st)
        else:
            rc = _lib.lib.lc2is_upsample_ce_fwd_bwd(low.data_ptr(), labels.data_ptr(), B, C, h, w, H, W, 0,
                                                    gs.data_ptr(), ls.data_ptr(), grad.data_ptr(), None, st)
        assert rc == 0, _lib.last_error()
        outs[ex] = (ls, grad)

    names = [_kernel_names(lambda: call(ex)) for ex in (False, True)]
    assert names[0] == names[1] and names[0], names
    assert torch.equal(outs[False][0], outs[True][0])
    d = float((outs[False][1] - outs[True][1]).abs().max())
    assert d <= 2 ** -21 * float(outs[False][1].abs().max()), d


def test_ex_rejects_bad_smoothing():
    low = torch.zeros(1, 3, 2, 2, device=DEV)
    labels = torch.zeros(1, 8, 8, dtype=torch.int64, device=DEV)
    ls = torch.zeros(1, dtype=torch.float64, device=DEV)
    for eps in (-0.1, 1.5, float("nan")):
        rc = _lib.lib.lc2is_upsample_ce_fwd_bwd_ex(low.data_ptr(), labels.data_ptr(), 1, 3, 2, 2, 8, 8, -100, None,
                                                   ctypes.c_float(eps), None, ls.data_ptr(), None, None,
                                                   _lib.stream_ptr())
        assert rc == -1 and "label_smoothing" in _lib.last_error()


@pytest.mark.parametrize("shape", ["x4", "x16", "generic_noninteger"])
def test_uniform_weights_give_the_unweighted_mean(shape):
    B, C, h, w, H, W, frac = SHAPES[shape]
    g = torch.Generator().manual_seed(63)
    low = torch.randn(B, C, h, w, generator=g) * 2.0
    labels = synthetic.make_labels(B, H, W, C, block=8, ignore_frac=frac).to(DEV)
    x0 = low.to(DEV).requires_grad_(True)
    ref = AuxiliaryLoss(ignore_index=0)(x0, labels) if H == W else None
    if ref is None:
        ref = head.UpsampledCrossEntropyLoss(ignore_index=0)(x0, labels)
    ref.backward()
    x1 = low.to(DEV).requires_grad_(True)
    loss = head.UpsampledCrossEntropyLoss(weight=torch.full((C,), 2.5), ignore_index=0).to(DEV)(x1, labels)
    loss.backward()
    _check(loss, x1.grad, ref.detach().cpu(), x0.grad.cpu())


@pytest.mark.parametrize("s", [4, 8, 16])
def test_wide_dynamic_range_exact_fallback_weighted(s):
    """The construction of test_gpu_k2.py::test_wide_dynamic_range_takes_exact_fallback with weights and smoothing."""
    g = torch.Generator().manual_seed(23)
    low = torch.randn(1, 6, 8, 8, generator=g)
    low[0, 0, ::2, ::2] += 300.0
    low[0, 3, 1::2, 1::2] -= 200.0
    labels = torch.randint(0, 6, (1, 8 * s, 8 * s), generator=g)
    w = _weight(6)
    ref_loss, ref_grad = upsample_ce_and_grad(low, labels, -100, w, 0.1, "mean")
    loss, grad = _run(low, labels, -100, w, 0.1, "mean", g_out=1.0)
    assert torch.isfinite(loss) and torch.isfinite(grad).all()
    _check(loss, grad, ref_loss, ref_grad, loss_rtol=1e-5, g_rtol=1e-4)


@pytest.mark.parametrize("s,h", [(16, 6), (8, 12)])
def test_strip_mixed_fast_and_slow_groups_and_ignored_quadrant_weighted(s, h):
    g = torch.Generator().manual_seed(31)
    B, C, H = 2, 37, s * h
    low = torch.randn(B, C, h, h, generator=g)
    low[0, 5, 2, 3] += 500.0
    labels = torch.randint(0, C, (B, H, H), generator=g)
    labels[1, : H // 2, : H // 2] = 0
    w = _weight(C)
    for red in ("mean", "sum"):
        ref_loss, ref_grad = upsample_ce_and_grad(low, labels, 0, w, 0.1, red)
        loss, grad = _run(low, labels, 0, w, 0.1, red, g_out=1.0)
        _check(loss, grad, ref_loss, ref_grad, loss_rtol=1e-5, g_rtol=1e-4)


@pytest.mark.parametrize("shape", ["x4", "x16", "generic_noninteger"])
def test_edge_cases(shape):
    B, C, h, w, H, W, _ = SHAPES[shape]
    g = torch.Generator().manual_seed(64)
    low = torch.randn(B, C, h, w, generator=g)
    wt = _weight(C)
    # everything ignored: NaN loss, zero gradient
    labels = torch.zeros(B, H, W, dtype=torch.int64)
    for weight in (None, wt):
        loss, grad = _run(low, labels, 0, weight, 0.1, "mean", g_out=1.0)
        assert torch.isnan(loss) and float(grad.abs().max()) == 0.0
    # every counted pixel has weight 0: NaN, as torch gives (0 / 0, also with smoothing)
    labels = torch.full((B, H, W), C // 3, dtype=torch.int64)
    for eps in (0.0, 0.1):
        loss, grad = _run(low, labels, -100, wt, eps, "mean", g_out=1.0)
        ref_loss, _ = upsample_ce_and_grad(low, labels, -100, wt, eps, "mean")
        assert torch.isnan(loss) and torch.isnan(ref_loss) and not bool(torch.isfinite(grad).all())
    # labels outside [0, C) that are not ignore_index: not counted, not in the weight sum
    labels = synthetic.make_labels(B, H, W, C, block=4)
    labels[0, 0, :3] = C + 5
    labels[-1, -1, -2:] = -7
    ref_labels = labels.clone()
    ref_labels[(labels < 0) | (labels >= C)] = -100
    den = ops.ce_weight_sum(labels.to(DEV), C, -100, wt.to(DEV))
    assert abs(float(den) - float(wt[ref_labels[ref_labels >= 0]].double().sum())) <= 1e-9 * float(den)
    assert float(ops.ce_weight_sum(labels.to(DEV), C, -100)) == float((ref_labels >= 0).sum())
    for red in ("mean", "sum"):
        ref_loss, ref_grad = upsample_ce_and_grad(low, ref_labels, -100, wt, 0.1, red)
        loss, grad = _run(low, labels, -100, wt, 0.1, red, g_out=1.0)
        _check(loss, grad, ref_loss, ref_grad)


def test_module_surface_on_device():
    C = 5
    crit = head.UpsampledCrossEntropyLoss(weight=torch.ones(C), label_smoothing=0.1)
    with pytest.raises(RuntimeError, match="same device"):
        crit(torch.zeros(1, C, 2, 2, device=DEV), torch.zeros(1, 8, 8, dtype=torch.int64, device=DEV))
    crit = crit.to(DEV)
    assert crit.weight.is_cuda and "weight" in crit.state_dict()
    x = torch.randn(1, C, 2, 2, device=DEV, dtype=torch.bfloat16, requires_grad=True)
    loss = crit(x, torch.randint(0, C, (1, 8, 8), device=DEV))
    loss.backward()
    assert loss.dtype == torch.float32 and x.grad.dtype == torch.bfloat16 and torch.isfinite(loss)


def test_seg_head_loss_with_weight_and_smoothing():
    B, h, H, C, D = 2, 8, 128, 151, 512
    v = synthetic.make_patch_embeddings(B, h * h, D, dtype=torch.float32)
    t = synthetic.make_prototypes(C, D)
    labels = synthetic.make_labels(B, H, H, C, block=8, ignore_frac=0.1)
    w = _weight(C)
    vd = v.to(DEV).requires_grad_(True)
    td = t.to(DEV).requires_grad_(True)
    crit = head.SegHeadLoss(ignore_index=0, weight=w, label_smoothing=0.1).to(DEV)
    loss, low, n_valid = crit(vd, td, labels.to(DEV))
    (0.4 * loss).backward()
    assert int(n_valid) == int((labels != 0).sum())
    # the same chain through the public pieces
    v2 = v.to(DEV).requires_grad_(True)
    t2 = t.to(DEV).requires_grad_(True)
    l2 = head.UpsampledCrossEntropyLoss(weight=w, ignore_index=0, label_smoothing=0.1).to(DEV)(
        head.cosine_logits(v2, t2), labels.to(DEV))
    (0.4 * l2).backward()
    assert abs(float(loss) - float(l2)) <= 2e-6 * abs(float(l2))
    for a, b in ((vd.grad, v2.grad), (td.grad, t2.grad)):
        assert float((a - b).abs().max()) <= 1e-2 * float(b.abs().max())
    # the oracle chain, at the tolerances of test_gpu_k1.py::test_fused_head_loss_matches_oracle
    vr = v.clone().requires_grad_(True)
    tr = t.clone().requires_grad_(True)
    up = F.interpolate(O.cosine_logits(vr, tr), size=(H, H), mode="bilinear")
    ref = F.cross_entropy(up, labels, weight=w, ignore_index=0, label_smoothing=0.1)
    gv, gt = torch.autograd.grad(0.4 * ref, (vr, tr))
    assert abs(float(loss) - float(ref)) <= 1e-4 * float(ref)
    ev = float((vd.grad.cpu() - gv).abs().max() / gv.abs().max())
    et = float((td.grad.cpu() - gt).abs().max() / gt.abs().max())
    assert ev < 3e-2 and et < 3e-2, (ev, et)


def test_cuda_graph_capture_replays_eager():
    B, C, h, H = 2, 150, 8, 128
    g = torch.Generator().manual_seed(65)
    low = (torch.randn(B, C, h, h, generator=g) * 2.0).to(DEV)
    labels = synthetic.make_labels(B, H, H, C, block=8, ignore_frac=0.1).to(DEV)
    crit = head.UpsampledCrossEntropyLoss(weight=_weight(C), ignore_index=0, label_smoothing=0.1).to(DEV)
    x = low.clone().requires_grad_(True)
    eager = crit(x, labels)
    eager.backward()
    eager_grad = x.grad.clone()

    xs = low.clone().requires_grad_(True)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):                      # warm-up on a side stream, as torch's graph docs ask
        for _ in range(2):
            xs.grad = None
            crit(xs, labels).backward()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    xs.grad = None
    with torch.cuda.graph(graph):
        out = crit(xs, labels)
        out.backward()
    graph.replay()
    torch.cuda.synchronize()
    assert abs(float(out) - float(eager)) <= 2e-6 * abs(float(eager))
    assert float((xs.grad - eager_grad).abs().max()) <= 1e-6 * float(eager_grad.abs().max())


@pytest.mark.parametrize("h", [32, 128])
def test_full_size_against_eager_torch(h):
    """B=16, C=150, 512^2: the batch runs; 2 images are compared with eager torch on the device."""
    B, C, H = 16, 150, 512
    g = torch.Generator().manual_seed(66)
    low = (torch.randn(B, C, h, h, generator=g) * 0.2).to(DEV)
    labels = synthetic.make_labels(B, H, H, C, ignore_frac=0.1).to(DEV)
    w = _weight(C).to(DEV)
    ls, grad, _ = ops.upsample_ce(low, labels, 0, None, weight=w, label_smoothing=0.1)
    assert torch.isfinite(ls).all() and torch.isfinite(grad).all()
    x = low[:2].clone().requires_grad_(True)
    ref = F.cross_entropy(F.interpolate(x, mode="bilinear", size=H), labels[:2], weight=w, ignore_index=0,
                          reduction="sum", label_smoothing=0.1)
    ref.backward()
    ls2, grad2, _ = ops.upsample_ce(low[:2], labels[:2], 0, None, weight=w, label_smoothing=0.1)
    assert abs(float(ls2) - float(ref)) <= 2e-6 * abs(float(ref))
    assert float((grad2 - x.grad).abs().max()) <= 1e-5 * float(x.grad.abs().max())
