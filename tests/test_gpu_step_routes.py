"""Every route of the whole-step entries - HeadStep (lc2is_b200/step.py) and lc2is_head_step_host[_submit] (csrc/api.cu,
head_step_enqueue) - run once and checked on every output the step leaves behind, against references built from the
step's OWN intermediate buffers (the method of test_gpu_k1b_exact.py, applied to the whole step):

  n_valid    exactly #{labels in [0, C) other than ignore_index}; on the split routes the packed labels equal
             ops.pack_labels of the int64 map bit for bit (host step: 1- and 2-byte host labels and the raw int64 share)
  forward    t_hat / inv_t == ops.proto_normalize(t) bit for bit; inv_v within rtol 1e-5 of 1/||v|| (exactly 1 without
             normalize); v_hat == bf16_rn(fp32(v * inv_v)) bit for bit where the step forms it; logits within
             2e-6 * max(|ref|, scale) of the float64 product of the step's bf16 operands (test_gpu_k1.py's bound)
  loss_sum,  float64 autograd of F.cross_entropy(F.interpolate(logits, (H, W), bilinear), target, reduction="sum") on the
  grad_low   step's logits, one image at a time on the device, targets outside [0, C) mapped to ignore_index: loss rel
             2e-6 and |grad_low - ref| <= 1e-5 * max|ref| (test_gpu_k2.py's bounds, un-scaled); loss == fp32(loss_sum /
             n_valid) exactly and |gscale * n_valid - 1| <= 1e-6
  grad_v,    tests/k1b_reference.py on grad_low, the logits, the raw V (or v_hat), inv_v, t_hat, inv_t and gscale:
  grad_t     |got - ref| <= TAU * A per element (grad_t: _dt_tau's tau where the dT chain is deep), plus 2^-8 |ref| for
             the bf16 grad_v; grad_v starts as NaN (HeadStep) or as 0xFF bytes (the host step's workspace), so an
             element that no kernel writes fails
  confmat    row sums == the histogram of the labels in [0, C); |cm - cm64|_1 <= 2 * #{counted pixels whose float64
             top-2 gap is <= 1e-5 * max(1, max|up|)}, cm64 the float64 argmax of the upsampled own logits; and bit-identical
             to the public op that runs the same kernel on the step's logits (ops.argmax_confmat on the one-call routes,
             ops.argmax_confmat_packed on the split routes, ops.ce_argmax_fused at x16)

Each case asserts the route it means to test before it runs anything else: step.split / step.fused / fuse_norm, or for
the host step the library's own predicates (lc2is_ce_split_supported, lc2is_ce_argmax_fused_supported,
lc2is_host_label_bytes).  The host step keeps everything in its workspace; the tests read it through a mirror of
step_layout (api.cu).  A CPU test holds the mirror's total to lc2is_head_step_workspace, and on the GPU the mirror's v_in
region must hold the input V and its t_hat region ops.proto_normalize(t), bit for bit.

Measured on one B200 (1000 W power limit); share of each bound used, worst over the route's cases (grad_v, grad_t: worst
|got - ref| / A and bound use):
    route                         logits  loss    grad_low  grad_v               grad_t                 |cm - cm64|_1
    HeadStep fused x16 (G-A)      0.39    0.013   0.014     2.4e-3 (0.99)        3.9e-7 (0.026)         0 (109 near ties)
    HeadStep one-call x4 (G-B)    0.41    0.003   0.008     3.5e-3 (0.99)        2.3e-5 (0.40 of 3.8 TAU)  0 (17)
    HeadStep split x16 (cfg5)     0.39    0.023   0.010     2.2e-3 (0.99)        7.6e-7 (0.027)         0 (79)
    HeadStep split x8, staged /
      global taps / ignore -100   0.37    0.018   0.016     2.8e-3 (0.99)        2.2e-7 (0.015)         0
    HeadStep one-call generic     0.32    0.019   0.087     3.2e-3 (0.99)        2.5e-7 (0.016)         0
    HeadStep options (fp32 V,
      normalize=False, scale)     0.47    0.012   0.23      2.5e-3 (0.98)        3.1e-7 (0.020)         0
    HeadStep two calls, capture,
      backward=False, non-square  0.38    0.015   0.012     3.4e-3 (0.99)        2.2e-7 (0.014)         0
    host step, every route        0.36    0.016   0.016     3.5e-3 (0.99)        2.4e-7 (0.016)         0
    host step e2e (G-A, depth 2)  0.41    0.013   0.013     2.5e-3 (0.99)        4.9e-7 (0.032)         2 (104 near ties)
The bf16 grad_v's use is its own output rounding (test_gpu_k1b_exact.py); its fp32 error stays at the K1b tests' level.
The file runs in about 9 s.
"""
import math
from types import SimpleNamespace

import pytest
import torch
import torch.nn.functional as F

from k1b_reference import TAU, check_bound, k1b_reference
from lc2is_b200 import _lib, ops, synthetic
from lc2is_b200._lib import lib

gpu = pytest.mark.gpu
DEV = "cuda"
D = 512


def _f32(x: float) -> float:
    """The value the kernels see for a float argument (c_float)."""
    return float(torch.tensor(x, dtype=torch.float32))


def _bits(x: torch.Tensor) -> torch.Tensor:
    return x.view({2: torch.int16, 4: torch.int32, 8: torch.int64}[x.element_size()])


def _inputs(B, h, w, H, W, C, ign=0, v_dtype=torch.bfloat16, v_mult=1.0, seed=0):
    """Patch embeddings with a cosine of about 0.7 to one prototype per 2 x 2 block of patches (so that the argmax has
    real class boundaries) and row norms spread over 4x, the prototypes [C, D], and ADE-like labels with ignore_index on
    10 % of the pixels and four values that are not class ids.  CPU tensors."""
    g = torch.Generator().manual_seed(100 + seed)
    t = synthetic.make_prototypes(C, D, seed=synthetic.SEED + seed)
    cls = torch.randint(0, C, (B, (h + 1) // 2, (w + 1) // 2), generator=g)
    cls = cls.repeat_interleave(2, 1).repeat_interleave(2, 2)[:, :h, :w].reshape(B, h * w)
    v = torch.randn(B, h * w, D, generator=g) + t[cls]
    v = v * (0.5 + 1.5 * torch.rand(B, h * w, 1, generator=g)) * v_mult
    labels = synthetic.make_labels(B, H, W, C, seed=synthetic.SEED + seed, block=8, ignore_frac=0.1, ignore_index=ign)
    labels[0, 0, :4] = torch.tensor([C, 255, -1, 2 ** 40])          # never counted, never in the matrix (255 is a class
    return v.to(v_dtype), t, labels                                  # id for C > 255)


def _dt_tau(B, hw, C, D=D):
    """The grad_t bound's tau: TAU, or 2^-23 per fp32 addition of the deepest dT accumulation chain where that is more.
    K1b's dT GEMM sums the pixels split-K: each CTA accumulates its range of 64-pixel blocks (4 MMAs of K = 16 each) in
    one fp32 tensor-memory accumulator, and the slices meet in fp32 reductions (k1b_bwd.cu, the dT launch; the slice
    count follows from the SM count and the class / channel tiles).  TAU allows 128 roundings at the full abs-sum A,
    which holds while the partial sums random-walk (test_gpu_k1b_exact.py's random G).  K2's gradient is softmax -
    onehot: for every class but the label it is positive, so at G-B (B = 16, hw = 16384: 111 blocks, 444 MMAs a chain)
    the partial sums grow with the chain and their roundings add up, measured up to 2.3e-5 A = 1.5 TAU.  Each addition
    errs by at most one ulp of a partial sum <= A, so 2^-23 * (MMAs + slices) bounds it (3.8 TAU at G-B); a 64-pixel block
    dropped from that chain would still be about 4x over it."""
    Cp = _lib.class_pad(C)
    n0 = -(-Cp // 256)
    nb = -(-(-(-Cp // n0)) // 16) * 16
    items = -(-D // 128) * -(-Cp // nb)
    blocks = B * -(-hw // 64)
    ksplit = max(1, min(torch.cuda.get_device_properties(0).multi_processor_count // items, blocks))
    return max(TAU, 2.0 ** -23 * (4 * -(-blocks // ksplit) + ksplit))


# ---- the checks -------------------------------------------------------------------------------------------------------
def _check_step(o, case, cm_before=None):
    """Checks every output of one call (see the module docstring).  `o` holds the call's device buffers and settings;
    `cm_before` is the accumulated matrix before the call.  -> the measured bound uses, which it also prints."""
    B, C, h, w = o.logits.shape
    H, W, ign, hw = o.H, o.W, o.ign, h * w
    lab = o.labels
    inr = (lab >= 0) & (lab < C)
    # 1. the valid count and the packed labels
    assert o.n_valid == int((inr & (lab != ign)).sum()), (case, "n_valid", o.n_valid)
    if o.packed is not None:
        want, _ = ops.pack_labels(lab, C, ign)
        assert torch.equal(_bits(o.packed), _bits(want)), (case, "packed labels")
    # 2. the forward: operands and logits
    t_hat, inv_t = ops.proto_normalize(o.t, o.normalize)
    assert torch.equal(_bits(o.t_hat), _bits(t_hat)) and torch.equal(_bits(o.inv_t.reshape(1, C)), _bits(inv_t)), \
        (case, "t_hat / inv_t")
    vf = o.v.reshape(B * hw, D).float()
    if o.normalize:
        e = float((o.inv_v.double() * vf.double().norm(dim=1) - 1).abs().max())
        assert e <= 1e-5, (case, "inv_v", e)
    else:
        assert bool((o.inv_v == 1).all()), (case, "inv_v without normalize")
    if o.raw_v:
        assert torch.equal(_bits(o.V), _bits(o.v.reshape(B * hw, D))), (case, "raw V")
    else:
        assert torch.equal(_bits(o.V), _bits((vf * o.inv_v.unsqueeze(1)).to(torch.bfloat16))), (case, "v_hat")
    ref = o.scale * torch.einsum("bpd,cd->bcp", o.V.reshape(B, hw, D).double(), o.t_hat[0, :C].double())
    if o.raw_v:                                    # normalisation inside the GEMM: the fp32 row factor scales the accumulator
        ref = ref * o.inv_v.reshape(B, 1, hw).double()
    e_log = float((o.logits.reshape(B, C, hw).double() - ref).abs().max()) / (2e-6 * max(float(ref.abs().max()), o.scale))
    assert e_log <= 1, (case, "logits", e_log)
    del ref
    # 3. + 5. loss_sum and grad_low against float64 autograd, the matrix against the float64 argmax, one image at a time
    loss_ref, g_err, g_max, near = 0.0, 0.0, 0.0, 0
    cm64 = torch.zeros(C * C, dtype=torch.int64, device=lab.device)
    for b in range(B):
        x = o.logits[b:b + 1].double().requires_grad_(o.backward)
        up = F.interpolate(x, size=(H, W), mode="bilinear", align_corners=False)
        tgt = torch.where(inr[b:b + 1], lab[b:b + 1], torch.full_like(lab[b:b + 1], ign))
        loss = F.cross_entropy(up, tgt, ignore_index=ign, reduction="sum")
        with torch.no_grad():
            top = up[0].topk(2, dim=0).values
            m = inr[b]
            near += int(((top[0] - top[1]) <= 1e-5 * max(1.0, float(up.abs().max())))[m].sum())
            cm64 += torch.bincount(lab[b][m] * C + up[0].argmax(0)[m], minlength=C * C)
            del top
        if o.backward:
            loss.backward()
            d = (o.grad_low[b].double() - x.grad[0]).abs().nan_to_num(float("inf"))     # NaN: unwritten, fails
            g_err = max(g_err, float(d.max()))
            g_max = max(g_max, float(x.grad.abs().max()))
        loss_ref += float(loss)
        del x, up, loss
    e_loss = abs(o.loss_sum - loss_ref) / (2e-6 * abs(loss_ref))
    assert e_loss <= 1, (case, "loss_sum", o.loss_sum, loss_ref)
    assert o.loss == _f32(o.loss_sum / o.n_valid), (case, "loss", o.loss)
    assert abs(o.gscale * o.n_valid - 1) <= 1e-6, (case, "gscale", o.gscale)
    use = {"logits": e_log, "loss": e_loss}
    # 4. grad_v and grad_t against the K1b reference on the step's own operands
    if o.backward:
        use["grad_low"] = g_err / (1e-5 * g_max)
        assert use["grad_low"] <= 1, (case, "grad_low", g_err, g_max)
        ref = k1b_reference(o.grad_low, o.logits, o.V, o.inv_v, o.t_hat, o.inv_t, normalize=o.normalize, scale=o.scale,
                            g=o.gscale, raw_v=o.raw_v)
        use["grad_v"] = check_bound(f"{case} grad_v", o.grad_v, ref.grad_v, ref.grad_v_A, bf16_out=True)
        use["grad_t"] = check_bound(f"{case} grad_t", o.grad_t, ref.grad_t, ref.grad_t_A, tau=_dt_tau(B, hw, C))
        del ref
    # 5. the confusion matrix
    cm = o.confmat if cm_before is None else o.confmat - cm_before
    assert torch.equal(cm.sum(1), torch.bincount(lab[inr], minlength=C)), (case, "confmat row sums")
    diff = int((cm.flatten() - cm64).abs().sum())
    assert diff <= 2 * near, (case, "confmat vs float64 argmax", diff, near)
    if o.route == "one-call":
        same = ops.argmax_confmat(o.logits, lab, size=(H, W), mode="bilinear")[0]
    elif o.route == "split":
        same = ops.argmax_confmat_packed(o.logits, o.packed, (H, W))[0]
    else:
        same = ops.ce_argmax_fused(o.logits, o.packed, (H, W), torch.zeros(1, dtype=torch.float64, device=lab.device),
                                   torch.zeros_like(o.logits), onehot=True)[0]
    assert torch.equal(cm, same), (case, "confmat vs the public op", int((cm - same).abs().sum()))
    use["confmat"] = (diff, near)
    print(f"step-routes {case}: " + "  ".join(
        f"{k} {v[0]:.3g}/A (bound use {v[1]:.3g})" if k in ("grad_v", "grad_t") else
        f"{k} L1 {v[0]} (near ties {v[1]})" if k == "confmat" else f"{k} bound use {v:.3g}" for k, v in use.items()))
    return use


# ---- HeadStep ---------------------------------------------------------------------------------------------------------
def _head_out(step, v, t, labels):
    """The most recent call's buffers of a HeadStep."""
    blk = step._blk
    raw = step._fuse(v)
    return SimpleNamespace(
        v=v, t=t, labels=labels, H=step.H, W=step.W, ign=step.ignore_index, scale=_f32(step.logit_scale),
        normalize=step.normalize, raw_v=raw, backward=step.backward, V=v.reshape(-1, D) if raw else step.v_hat,
        logits=step.logits, inv_v=step.inv_v, t_hat=step.t_hat, inv_t=step.inv_t, grad_low=blk.grad_low,
        grad_v=step.grad_v, grad_t=blk.grad_t, n_valid=int(blk.n_valid), loss_sum=float(blk.loss_sum),
        loss=float(step.loss), gscale=float(blk.gscale), confmat=step.confmat,
        packed=step.labels_packed if step.split else None,
        route="fused" if step.fused else "split" if step.split else "one-call")


def _head_step(B, h, w, H, W, C, route, *, ign=0, scale=1.0, normalize=True, v_dtype=torch.bfloat16, backward=True):
    """A HeadStep that takes `route` = (split, fused, fuse_norm), asserted before anything runs; grad_v set to NaN."""
    from lc2is_b200.step import HeadStep
    step = HeadStep(B, h, w, H, W, C, D, ignore_index=ign, logit_scale=scale, normalize=normalize, backward=backward,
                    v_dtype=v_dtype)
    assert (step.split, step.fused, step.fuse_norm) == route, (step.split, step.fused, step.fuse_norm)
    step.grad_v.fill_(float("nan"))
    return step


def _dev(*xs):
    return tuple(x.to(DEV) for x in xs)


FUSED, SPLIT, ONE_CALL = (True, True, True), (True, False, True), (False, False, True)
# (B, h, w, H, W, C, route, options)
HEAD_CASES = {
    "G-A fused x16": (16, 32, 32, 512, 512, 150, FUSED, {}),
    "G-B one-call x4": (16, 128, 128, 512, 512, 150, ONE_CALL, {}),
    "cfg5 split x16 global taps": (8, 64, 64, 1024, 1024, 847, SPLIT, {}),
    "split x8 staged": (2, 16, 16, 128, 128, 151, SPLIT, {}),
    "split x8 global taps": (2, 16, 16, 128, 128, 240, SPLIT, {}),      # (C + 2) * 128 B > 28 KB: taps stay in global memory
    "one-call generic": (2, 12, 12, 40, 40, 150, ONE_CALL, {}),
    "fused non-square": (2, 8, 12, 128, 192, 150, FUSED, {}),
    "one-call x4 non-square": (2, 16, 24, 64, 96, 150, ONE_CALL, {}),
    "fp32 V": (2, 8, 8, 128, 128, 150, (True, True, False), dict(v_dtype=torch.float32)),
    "normalize=False": (2, 8, 8, 128, 128, 150, (True, True, False), dict(normalize=False, v_mult=0.01)),
    "logit_scale": (2, 8, 8, 128, 128, 150, FUSED, dict(scale=14.285714)),
    "ignore_index=-100": (2, 16, 16, 128, 128, 151, SPLIT, dict(ign=-100)),
}


@gpu
@pytest.mark.parametrize("case", list(HEAD_CASES))
def test_head_step_route(case):
    B, h, w, H, W, C, route, opt = HEAD_CASES[case]
    opt = dict(opt)
    v_mult = opt.pop("v_mult", 1.0)
    step = _head_step(B, h, w, H, W, C, route, **opt)
    v, t, labels = _dev(*_inputs(B, h, w, H, W, C, ign=step.ignore_index, v_dtype=step.v_dtype, v_mult=v_mult))
    step(v, t, labels)
    torch.cuda.synchronize()
    _check_step(_head_out(step, v, t, labels), case)


SMALL = {"fused": (2, 8, 8, 128, 128, 150, FUSED), "split": (2, 16, 16, 128, 128, 151, SPLIT),
         "one-call": (2, 32, 32, 128, 128, 150, ONE_CALL)}


@gpu
def test_head_step_two_calls_use_both_blocks():
    """Two calls on different inputs: the second call's results sit in the other accumulator block, each call meets the
    references of its own buffers, the first block is left as the first call wrote it, and the matrix is the sum."""
    B, h, w, H, W, C, route = SMALL["fused"]
    step = _head_step(B, h, w, H, W, C, route)
    v, t, labels = _dev(*_inputs(B, h, w, H, W, C, seed=0))
    step(v, t, labels)
    torch.cuda.synchronize()
    k1 = step._cur
    _check_step(_head_out(step, v, t, labels), "two calls, first")
    first = [x.clone() for x in (step._blocks[k1].acc32, step.confmat)]
    v2, t2, labels2 = _dev(*_inputs(B, h, w, H, W, C, seed=1))
    step.grad_v.fill_(float("nan"))
    step(v2, t2, labels2)
    torch.cuda.synchronize()
    assert step._cur == k1 ^ 1
    assert torch.equal(_bits(step._blocks[k1].acc32), _bits(first[0])), "the second call wrote into the first block"
    _check_step(_head_out(step, v2, t2, labels2), "two calls, second", cm_before=first[1])


@gpu
@pytest.mark.parametrize("route", list(SMALL))
def test_head_step_without_backward(route):
    """backward=False: the same n_valid and matrix as a training call, the loss to 1e-6, the loss checks, and gradient
    buffers left as they were (grad_v NaN, the zero-filled block's grad_low / grad_t zero)."""
    B, h, w, H, W, C, rt = SMALL[route]
    v, t, labels = _dev(*_inputs(B, h, w, H, W, C, seed=2))
    train = _head_step(B, h, w, H, W, C, rt)
    train(v, t, labels)
    ev = _head_step(B, h, w, H, W, C, rt, backward=False)
    ev(v, t, labels)
    torch.cuda.synchronize()
    o = _head_out(ev, v, t, labels)
    _check_step(o, f"backward=False {route}")
    assert int(ev.n_valid) == int(train.n_valid) and torch.equal(ev.confmat, train.confmat)
    assert abs(float(ev.loss) - float(train.loss)) <= 1e-6 * abs(float(train.loss))
    assert bool(ev.grad_v.isnan().all())
    assert not bool(ev.grad_low.any()) and not bool(ev.grad_t.any())


@gpu
@pytest.mark.parametrize("route", list(SMALL))
def test_head_step_capture_replay(route):
    """capture() replayed against an eager call on the same inputs: n_valid, the packed labels and the matrix's
    increment bit-identical; every output meets the references of the replay's own buffers."""
    B, h, w, H, W, C, rt = SMALL[route]
    v, t, labels = _dev(*_inputs(B, h, w, H, W, C, seed=3))
    step = _head_step(B, h, w, H, W, C, rt)
    step(v, t, labels)
    torch.cuda.synchronize()
    eager = _head_out(step, v, t, labels)
    n_eager, cm_eager = eager.n_valid, step.confmat.clone()
    packed_eager = None if eager.packed is None else eager.packed.clone()
    replays = [step.capture(v, t, labels) for _ in range(2)]          # one graph per accumulator block, as the bench
    for k, replay in enumerate(replays):
        step.grad_v.fill_(float("nan"))
        cm_before = step.confmat.clone()
        replay()
        torch.cuda.synchronize()
        o = _head_out(step, v, t, labels)
        assert o.n_valid == n_eager and torch.equal(step.confmat - cm_before, cm_eager)
        if packed_eager is not None:
            assert torch.equal(_bits(o.packed), _bits(packed_eager))
        _check_step(o, f"capture {route} replay {k}", cm_before=cm_before)


# ---- the host step ----------------------------------------------------------------------------------------------------
_REGIONS = ("v_in", "labels", "packed", "t_in", "t_hat", "inv_t", "v_hat", "inv_v", "logits", "grad_low", "grad_v",
            "grad_t", "bwd_ws", "confmat", "scalars")


def _ws_layout(B, hw, D, C, H, W):
    """Mirror of step_layout (csrc/api.cu): {region: byte offset} and the total; each region starts 256-byte aligned.
    scalars: [0] double loss_sum, [8] int64 n_valid, [16] float gscale, [20] float loss."""
    M, Cp = B * hw, _lib.class_pad(C)
    sizes = (M * D * 2, B * H * W * 8, B * H * W * 2, C * D * 4, Cp * D * 2, C * 4, M * D * 2, M * 4, M * C * 4, M * C * 4,
             M * D * 2, C * D * 4, int(lib.lc2is_cosine_logits_bwd_workspace(B, hw, D, 1, C)), C * C * 8, 256)
    off, o = {}, 0
    for name, n in zip(_REGIONS, sizes):
        off[name] = o
        o += -(-n // 256) * 256
    return off, o


@pytest.mark.parametrize("B,hw,Dm,C,H,W", [
    (16, 1024, 512, 150, 512, 512), (16, 16384, 512, 150, 512, 512), (8, 4096, 512, 847, 1024, 1024),
    (5, 64, 512, 150, 128, 128), (3, 256, 512, 300, 128, 128), (3, 96, 512, 150, 128, 192), (2, 144, 512, 19, 40, 40),
    (1, 8, 64, 3, 32, 32), (7, 200, 320, 41, 100, 75), (2, 64, 768, 1000, 512, 512)])
def test_host_workspace_mirror_matches_the_library(B, hw, Dm, C, H, W):
    """The tests' mirror of the host step's workspace layout has the library's size (no device needed)."""
    off, total = _ws_layout(B, hw, Dm, C, H, W)
    assert total == int(lib.lc2is_head_step_workspace(B, hw, Dm, C, H, W))
    assert all(o % 256 == 0 for o in off.values())


def _host_route(hs):
    B, h, w, Dm, C, H, W = hs.args
    split = bool(lib.lc2is_ce_split_supported(h, w, H, W))
    fused = split and bool(lib.lc2is_ce_argmax_fused_supported(C, h, w, H, W))
    return split, fused, hs.label_bytes if hs.host_pack else 8


def _region(ws, off, name, dtype, *shape):
    n = math.prod(shape) * torch.empty((), dtype=dtype).element_size()
    return ws[off[name]:off[name] + n].view(dtype).view(*shape)


def _host_out(hs, slot, v, t, labels):
    """The buffers a host step left in `slot`'s workspace (v, t, labels: the inputs, on the device)."""
    B, h, w, Dm, C, H, W = hs.args
    off, _ = _ws_layout(B, h * w, Dm, C, H, W)
    ws, M = slot.ws, B * h * w
    split, fused, _ = _host_route(hs)
    sc = ws[off["scalars"]:off["scalars"] + 24]
    r = lambda name, dtype, *shape: _region(ws, off, name, dtype, *shape)
    o = SimpleNamespace(
        v=v, t=t, labels=labels, H=H, W=W, ign=hs.ignore_index, scale=_f32(hs.logit_scale), normalize=True, raw_v=True,
        backward=hs.backward, V=r("v_in", torch.bfloat16, M, Dm), logits=r("logits", torch.float32, B, C, h, w),
        inv_v=r("inv_v", torch.float32, M), t_hat=r("t_hat", torch.bfloat16, 1, _lib.class_pad(C), Dm),
        inv_t=r("inv_t", torch.float32, 1, C), grad_low=r("grad_low", torch.float32, B, C, h, w),
        grad_v=r("grad_v", torch.bfloat16, B, h * w, Dm), grad_t=r("grad_t", torch.float32, 1, C, Dm),
        n_valid=int(sc[8:16].view(torch.int64)), loss_sum=float(sc[0:8].view(torch.float64)),
        gscale=float(sc[16:20].view(torch.float32)), loss=float(sc[20:24].view(torch.float32)),
        confmat=r("confmat", torch.int64, C, C), packed=r("packed", torch.uint16, B, H, W) if split else None,
        route="fused" if fused else "split" if split else "one-call")
    # the host copies of the results are the workspace's
    assert float(slot.out_loss) == o.loss and int(slot.out_n_valid) == o.n_valid
    assert torch.equal(slot.out_confmat, o.confmat.cpu())
    return o


def _host_step(B, h, w, H, W, C, route, **kw):
    """A HostStep that takes `route` = (split, fused, label bytes), asserted first; every workspace set to 0xFF."""
    from lc2is_b200.step import HostStep
    hs = HostStep(B, h, w, H, W, C, D, ignore_index=0, **kw)
    got = _host_route(hs)
    assert got == route or (route[2] is None and got[:2] == route[:2]), got
    for s in hs.slots:
        s.ws.fill_(0xFF)
    return hs


def _pinned(v, t, labels):
    return v.pin_memory(), t.pin_memory(), labels.pin_memory()


def _agrees_with_head_step(o, B, h, w, H, W, C, v, t, labels):
    """HeadStep on the same inputs: n_valid and the matrix exactly, the loss to 2e-6."""
    from lc2is_b200.step import HeadStep
    step = HeadStep(B, h, w, H, W, C, D, ignore_index=o.ign, logit_scale=o.scale)
    step(v, t, labels)
    torch.cuda.synchronize()
    assert int(step.n_valid) == o.n_valid and torch.equal(step.confmat, o.confmat)
    assert abs(float(step.loss) - o.loss) <= 2e-6 * abs(float(step.loss))


@gpu
@pytest.mark.parametrize("pipelined", [False, True])
@pytest.mark.parametrize("raw", [0, 2, 5])
def test_host_step_fused_chunks(raw, pipelined):
    """x16 with B = 5: 2 uneven chunks (3 + 2 images) with host-packed labels, 4 (2 + 2 + 1) when all five label maps
    cross as int64 (raw = 5), 1 without a copy stream; raw = 2 puts the raw share inside the last chunk."""
    B, h, w, H, W, C = 5, 8, 8, 128, 128, 150
    hs = _host_step(B, h, w, H, W, C, (True, True, 8 if raw == B else 1), pipelined=pipelined, raw_images=raw)
    v, t, labels = _inputs(B, h, w, H, W, C, seed=4)
    hs(*_pinned(v, t, labels))
    vd, td, ld = _dev(v, t, labels)
    o = _host_out(hs, hs.slots[0], vd, td, ld)
    _check_step(o, f"host fused x16 raw {raw} pipelined {int(pipelined)}")
    _agrees_with_head_step(o, B, h, w, H, W, C, vd, td, ld)


HOST_CASES = {
    "x8 one-byte labels": (3, 16, 16, 128, 128, 151, (True, False, 1), 1),
    "C=300 two-byte labels": (3, 8, 8, 128, 128, 300, (True, True, 2), 1),
    "one-call x4": (2, 32, 32, 128, 128, 150, (False, False, 8), None),
    "fused non-square": (3, 8, 12, 128, 192, 150, (True, True, 1), 1),
}


@gpu
@pytest.mark.parametrize("case", list(HOST_CASES))
def test_host_step_route(case):
    B, h, w, H, W, C, route, raw = HOST_CASES[case]
    hs = _host_step(B, h, w, H, W, C, route, raw_images=raw)
    v, t, labels = _inputs(B, h, w, H, W, C, seed=5)
    hs(*_pinned(v, t, labels))
    vd, td, ld = _dev(v, t, labels)
    o = _host_out(hs, hs.slots[0], vd, td, ld)
    _check_step(o, f"host {case}")
    _agrees_with_head_step(o, B, h, w, H, W, C, vd, td, ld)


@gpu
def test_host_step_without_backward():
    """backward=False: the training step's n_valid, matrix and loss (to 1e-6); no gradient region is written."""
    B, h, w, H, W, C = 3, 8, 8, 128, 128, 150
    v, t, labels = _inputs(B, h, w, H, W, C, seed=6)
    hs = _host_step(B, h, w, H, W, C, (True, True, 1), backward=False, raw_images=1)
    hs(*_pinned(v, t, labels))
    vd, td, ld = _dev(v, t, labels)
    o = _host_out(hs, hs.slots[0], vd, td, ld)
    _check_step(o, "host backward=False")
    for g in (o.grad_low, o.grad_v, o.grad_t):
        assert bool((g.view(torch.uint8) == 0xFF).all())
    _agrees_with_head_step(o, B, h, w, H, W, C, vd, td, ld)
    train = _host_step(B, h, w, H, W, C, (True, True, 1), raw_images=1)
    train(*_pinned(v, t, labels))
    assert int(train.out_n_valid) == o.n_valid and torch.equal(train.out_confmat, o.confmat.cpu())
    assert abs(float(train.out_loss) - o.loss) <= 1e-6 * abs(o.loss)


@gpu
@pytest.mark.parametrize("B,h,H,raw,label_bytes", [pytest.param(4, 8, 128, 1, 1, id="small"),
                                                   pytest.param(16, 32, 512, None, None, id="bench-e2e-G-A")])
def test_host_step_submit_wait(B, h, H, raw, label_bytes):
    """Two steps in flight (depth 2) on different inputs: each slot's workspace holds its own step.  The G-A case is the
    benchmark's e2e leg, with the label split it calibrates itself."""
    C = 150
    hs = _host_step(B, h, h, H, H, C, (True, True, label_bytes), depth=2, raw_images=raw)
    batches = [_inputs(B, h, h, H, H, C, seed=7 + k) for k in range(2)]
    pinned = [_pinned(*x) for x in batches]
    for x in pinned:
        hs.submit(*x)
    for k, s in enumerate(hs.slots):
        hs.wait()
        vd, td, ld = _dev(*batches[k])
        o = _host_out(hs, s, vd, td, ld)
        _check_step(o, f"host submit B{B} slot {k} (n_raw {hs.n_raw})")
        _agrees_with_head_step(o, B, h, h, H, H, C, vd, td, ld)
