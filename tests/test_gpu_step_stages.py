"""The whole-step cross-entropy stages (lc2is_step_ce_labels / lc2is_step_ce / lc2is_step_argmax) against the explicit
kernel chain of their route (include/lc2is_b200.h) on the same logits and labels:

  n_valid, packed labels, confmat   bit for bit
  loss_sum                          bit for bit (each warp adds one fp32 partial to the double sum: exact in double at
                                    these sizes, so the order of the atomics does not show)
  grad_low                          |got - ref| <= 2^-16 * (the cell's total bilinear tap weight, which bounds each of
                                    the softmax and -onehot sums of the cell): the kernels add the contributions of
                                    several warps to a cell with fp32 reductions, in whatever order the warps reach it,
                                    so two runs of the same kernel may differ in the last bits

plus the launches each stage makes (fused 1/1/0, split and one-call 1/1/1), which with the loss_sum bits pins the route.
"""
import pytest
import torch
import torch.nn.functional as F

from lc2is_b200 import _lib, synthetic
from lc2is_b200._lib import BILINEAR, check, lib, ptr

gpu = pytest.mark.gpu
DEV = "cuda"
IGN = 0

# name: (B, C, h, w, H, W, route, launches of the labels / CE / argmax stage)
CASES = {
    "fused x16": (2, 150, 8, 8, 128, 128, "fused", (1, 1, 0)),
    "split x8": (2, 151, 16, 16, 128, 128, "split", (1, 1, 1)),
    "one-call x4": (2, 150, 32, 32, 128, 128, "one-call", (1, 1, 1)),
    "one-call generic": (2, 150, 12, 12, 40, 40, "one-call", (1, 1, 1)),
}


def _bits(x: torch.Tensor) -> torch.Tensor:
    return x.view({2: torch.int16, 4: torch.int32, 8: torch.int64}[x.element_size()])


def _route(C, h, w, H, W):
    if not lib.lc2is_ce_split_supported(h, w, H, W):
        return "one-call"
    return "fused" if lib.lc2is_ce_argmax_fused_supported(C, h, w, H, W) else "split"


def _buffers(B, C, h, w, H, W, route):
    z = lambda *s, dt: torch.zeros(*s, dtype=dt, device=DEV)
    return dict(packed=z(B, H, W, dt=torch.uint16) if route != "one-call" else None, n_valid=z(1, dt=torch.int64),
                loss_sum=z(1, dt=torch.float64), grad_low=z(B, C, h, w, dt=torch.float32), confmat=z(C, C, dt=torch.int64))


def _entries(o, logits, labels, B, C, h, w, H, W, st):
    """The three stage entries; -> the launches each one made."""
    counts = []
    for call in (
            lambda: lib.lc2is_step_ce_labels(ptr(labels), B, C, h, w, H, W, IGN, ptr(o["packed"]), ptr(o["n_valid"]),
                                             ptr(o["grad_low"]), st),
            lambda: lib.lc2is_step_ce(ptr(logits), ptr(labels), ptr(o["packed"]), B, C, h, w, H, W, IGN,
                                      ptr(o["loss_sum"]), ptr(o["grad_low"]), ptr(o["confmat"]), st),
            lambda: lib.lc2is_step_argmax(ptr(logits), ptr(labels), ptr(o["packed"]), B, C, h, w, H, W,
                                          ptr(o["confmat"]), st)):
        n0 = _lib.launch_count()
        check(call(), "stage entry")
        counts.append(_lib.launch_count() - n0)
    return tuple(counts)


def _chain(o, logits, labels, B, C, h, w, H, W, route, st):
    """The route's kernels called one by one, as the header's table lists them."""
    lg, lab, pk, glow = ptr(logits), ptr(labels), ptr(o["packed"]), ptr(o["grad_low"])
    if route == "fused":
        check(lib.lc2is_pack_labels(lab, B * H * W, C, IGN, pk, ptr(o["n_valid"]), st), "pack_labels")
        check(lib.lc2is_ce_argmax_fused_packed(lg, pk, B, C, h, w, H, W, ptr(o["loss_sum"]), glow, 1, None,
                                               ptr(o["confmat"]), None, None, st), "ce_argmax_fused_packed")
    elif route == "split":
        check(lib.lc2is_ce_labels_prepass(lab, B, C, h, w, H, W, IGN, pk, ptr(o["n_valid"]), glow, st), "prepass")
        check(lib.lc2is_upsample_ce_packed(lg, pk, B, C, h, w, H, W, ptr(o["loss_sum"]), glow, st), "upsample_ce_packed")
        check(lib.lc2is_argmax_confmat_lowres_packed(lg, B, C, h, w, H, W, pk, ptr(o["confmat"]), None, None, st),
              "argmax_confmat_lowres_packed")
    else:
        check(lib.lc2is_count_valid(lab, B * H * W, C, IGN, ptr(o["n_valid"]), st), "count_valid")
        check(lib.lc2is_upsample_ce_fwd_bwd(lg, lab, B, C, h, w, H, W, IGN, None, ptr(o["loss_sum"]), glow, None, st),
              "upsample_ce_fwd_bwd")
        check(lib.lc2is_argmax_confmat_lowres(lg, B, C, h, w, H, W, BILINEAR, lab, H, W, ptr(o["confmat"]), None, None,
                                              st), "argmax_confmat_lowres")


def _tap_weight(h, w, H, W):
    """[h, w]: each low-resolution cell's total bilinear tap weight over the H x W output pixels."""
    x = torch.zeros(1, 1, h, w, dtype=torch.float64, device=DEV, requires_grad=True)
    F.interpolate(x, size=(H, W), mode="bilinear", align_corners=False).sum().backward()
    return x.grad[0, 0].float()


@gpu
@pytest.mark.parametrize("case", list(CASES))
def test_stages_match_the_kernel_chain(case):
    B, C, h, w, H, W, route, launches = CASES[case]
    assert _route(C, h, w, H, W) == route
    g = torch.Generator().manual_seed(7)
    logits = (3 * torch.randn(B, C, h, w, generator=g)).to(DEV)
    labels = synthetic.make_labels(B, H, W, C, block=8, ignore_frac=0.1, ignore_index=IGN)
    labels[0, 0, :4] = torch.tensor([C, 255, -1, 2 ** 40])           # never counted, never in the matrix
    labels = labels.to(DEV)
    st = torch.cuda.current_stream().cuda_stream
    got, ref = _buffers(B, C, h, w, H, W, route), _buffers(B, C, h, w, H, W, route)
    assert _entries(got, logits, labels, B, C, h, w, H, W, st) == launches
    _chain(ref, logits, labels, B, C, h, w, H, W, route, st)
    torch.cuda.synchronize()
    for k in ("n_valid", "packed", "loss_sum", "confmat"):
        if ref[k] is not None:
            assert torch.equal(_bits(got[k]), _bits(ref[k])), (case, k)
    assert int(ref["n_valid"]) > 0 and int(ref["confmat"].sum()) > 0
    d = (got["grad_low"] - ref["grad_low"]).abs()
    bound = 2.0 ** -16 * _tap_weight(h, w, H, W)
    assert bool((d <= bound).all()), (case, "grad_low", float((d / bound).max()))
    print(f"step-stages {case}: grad_low {int((_bits(got['grad_low']) != _bits(ref['grad_low'])).sum())} of "
          f"{ref['grad_low'].numel()} elements differ in their bits, max |d| / bound {float((d / bound).max()):.3g}")


@gpu
@pytest.mark.parametrize("case", ["fused x16", "split x8"])
def test_packed_labels_needed_on_split_geometries(case):
    B, C, h, w, H, W, _, _ = CASES[case]
    st = torch.cuda.current_stream().cuda_stream
    o = _buffers(B, C, h, w, H, W, "one-call")                       # (no packed buffer)
    logits = torch.zeros(B, C, h, w, device=DEV)
    labels = torch.zeros(B, H, W, dtype=torch.int64, device=DEV)
    n0 = _lib.launch_count()
    assert lib.lc2is_step_ce_labels(ptr(labels), B, C, h, w, H, W, IGN, None, ptr(o["n_valid"]), ptr(o["grad_low"]),
                                    st) == -1
    assert "d_labels_packed" in _lib.last_error()
    assert lib.lc2is_step_ce(ptr(logits), ptr(labels), None, B, C, h, w, H, W, IGN, ptr(o["loss_sum"]),
                             ptr(o["grad_low"]), ptr(o["confmat"]), st) == -1
    assert lib.lc2is_step_argmax(ptr(logits), ptr(labels), None, B, C, h, w, H, W, ptr(o["confmat"]), st) == -1
    assert _lib.launch_count() == n0


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-device error path")
def test_stage_entries_need_a_device():
    assert lib.lc2is_step_ce_labels(None, 1, 150, 8, 8, 128, 128, IGN, None, None, None, None) == -3
    assert "no CPU fallback" in _lib.last_error()
    assert lib.lc2is_step_ce(None, None, None, 1, 150, 8, 8, 128, 128, IGN, None, None, None, None) == -3
    assert lib.lc2is_step_argmax(None, None, None, 1, 150, 8, 8, 128, 128, None, None) == -3
