"""K1b (lc2is_cosine_logits_bwd[_ex]: k1b_prep[_f32]_kernel, k1b_dv_kernel, k1b_dt_kernel, k1b_dt_finish_kernel) against the
float64 reference of tests/k1b_reference.py built from the kernel's OWN operands: the forward's logits, v_hat (or the raw
V and inv_v), t_hat, inv_t, and the gradient G as the kernels consume it (bf16_rn(G), or bf16_rn(fp32(G * inv_v)) under
LC2IS_BWD_RAW_V; the projections from the unrounded G).

Bound, per element: |got - ref| <= TAU * A, where A is the same expression with every factor replaced by its absolute
value (the abs-sum that bounds the error of the fp32 accumulations), plus 2^-8 |ref| for a bf16 grad_v (its own output
rounding).  The maxima are also taken per [128 rows x 64 channels] block, so a failure names the block (one skipped or
stale tile), and grad_v starts as NaN, so an unwritten element fails too.  TAU = 2^-16 is 2^7 x the fp32 unit round-off:
room for 128 roundings at the full abs-sum, where the deepest chain here - 110 64-pixel blocks x 4 MMAs of one dT split-K
slice at B = 16, hw = 16384, then the slice reductions - is a random walk far below that.  Against the fp32-oracle tests'
2e-2 * max|grad| it is more than 100x tighter: it sees one dropped 64-pixel block of a 16384-pixel sum, a stale row factor
on one tile, and the projections formed from the rounded G.  Worst |got - ref| / A measured on one B200 (1000 W power
limit), over every case of this file:
    fp32 outputs                                   grad_v 2.9e-7 (2^-21.7)   grad_t 1.1e-7 (2^-23.1)
        step call, fp32 grad_v (every shape)       grad_v 2.9e-7             grad_t 1.1e-7
        path cross, fp32 grad_v                    grad_v 1.7e-7             grad_t 9.1e-8
        LC2IS_BWD_REUSE_PREP two-call form         grad_v 1.8e-7             grad_t 3.0e-8
        head.cosine_logits, fp32 V                 grad_v 2.1e-7             grad_t 7.5e-8
        HeadStep at G-A                                                      grad_t 1.1e-7
    i.e. at most 1/50 of TAU; the file runs in about 10 s.  A bf16 grad_v uses up to 0.99 of its bound: that is its own
    rounding (at most 2^-8 |x|, reached just above a power of two), not kernel error - the fp32 error under it is the
    1/50 of TAU * A above, so the float atomics' order cannot move a case over the bound.
The forward outputs each case needs are checked too: logits against a float64 product of the kernel's own bf16 operands
at test_gpu_k1.py::test_logits' bound (2e-6 * max(|ref|, scale)), here also for per-image prompts and D in {64, 320, 768}.
"""
import itertools

import pytest
import torch

from k1b_reference import check_bound as _check, k1b_reference
from lc2is_b200 import _lib, head, ops
from lc2is_b200._lib import BF16, BWD_RAW_V, BWD_REUSE_PREP, F32, lib, ptr, stream_ptr

pytestmark = pytest.mark.gpu
DEV = "cuda"
ERR_ARG, ERR_SHAPE = -1, -2


def _f32(x: float) -> float:
    """The value the kernels see for a float argument (c_float)."""
    return float(torch.tensor(x, dtype=torch.float32))


def _inputs(B, hw, C, D, n_sets=1, v_dtype=torch.bfloat16, seed=0):
    """Patch embeddings with row norms spread over 4x and a large cosine to one prototype (so that r, the row factors
    and the logits differ from row to row and matter), prototypes [C, D] or [n_sets, C, D], and an fp32 gradient."""
    g = torch.Generator(device=DEV).manual_seed(1000 + seed)
    t = torch.randn(n_sets, C, D, generator=g, device=DEV) * 1.05
    cls = torch.randint(0, C, (B, hw), generator=g, device=DEV)
    sets = torch.arange(B, device=DEV).unsqueeze(1) if n_sets > 1 else 0
    v = torch.randn(B, hw, D, generator=g, device=DEV) + 2.0 * t[sets, cls]
    v = v * (0.5 + 1.5 * torch.rand(B, hw, 1, generator=g, device=DEV))
    G = torch.randn(B, C, hw, generator=g, device=DEV) * 1e-3
    return v.to(v_dtype), (t[0] if n_sets == 1 else t), G


def _forward(v, t, C, normalize, scale, raw_v):
    """K0 + K1 as the library runs them -> (logits, the backward's V operand, inv_v, t_hat, inv_t)."""
    B, hw, D = v.shape
    t_hat, inv_t = ops.proto_normalize(t, normalize)
    logits, v_hat, inv_v = ops.cosine_logits_fwd(v, t_hat, C, (1, hw), normalize, scale, fuse_norm=raw_v)
    return logits, (v.reshape(B * hw, D) if raw_v else v_hat), inv_v, t_hat, inv_t


def _check_forward(logits, V, inv_v, t_hat, C, scale, raw_v, dev):
    B, hw = logits.shape[0], logits[0, 0].numel()
    n_sets, _, D = t_hat.shape
    T = t_hat[:, :C].to(dev).double()
    ref = scale * torch.einsum("bpd,bcd->bcp", V.reshape(B, hw, D).to(dev).double(), T.expand(B, -1, -1) if n_sets == 1 else T)
    if raw_v:                                      # normalisation inside the GEMM: the fp32 row factor scales the accumulator
        ref = ref * inv_v.reshape(B, 1, hw).to(dev).double()
    err = float((logits.reshape(B, C, hw).to(dev).double() - ref).abs().max())
    assert err <= 2e-6 * max(float(ref.abs().max()), scale), ("logits", err)


def _bf16_grad(G, C):
    """The bf16 [B, C_pad, hw] operand form of an fp32 [B, C, hw] gradient, pad rows zero (built by torch)."""
    B, _, hw = G.shape
    out = torch.zeros(B, _lib.class_pad(C), hw, dtype=torch.bfloat16, device=G.device)
    out[:, :C] = G.to(torch.bfloat16)
    return out


def _bwd(G, logits, V, inv_v, t_hat, inv_t, C, *, normalize=True, scale=1.0, gscale=None, gv=None, gt=None, ws=None,
         flags=0, B=None, hw=None, D=None, n_sets=None, g_dtype=None):
    """One lc2is_cosine_logits_bwd_ex call; returns its code.  Shape arguments default to the tensors' own."""
    B = logits.shape[0] if B is None else B
    hw = logits[0, 0].numel() if hw is None else hw
    D = t_hat.shape[2] if D is None else D
    n_sets = t_hat.shape[0] if n_sets is None else n_sets
    if ws is None:
        n = int(lib.lc2is_cosine_logits_bwd_workspace(max(B, 1), hw, D, n_sets, C))
        ws = torch.empty(max(n, 256), dtype=torch.uint8, device=DEV)
    return lib.lc2is_cosine_logits_bwd_ex(ptr(G), ops._dt(G) if g_dtype is None else g_dtype, ptr(logits), ptr(V),
                                          ptr(inv_v), ptr(t_hat), ptr(inv_t), B, hw, D, n_sets, C, int(normalize),
                                          float(scale), ptr(gscale), ptr(gv), ops._dt(gv) if gv is not None else F32,
                                          ptr(gt), ptr(ws), stream_ptr(), flags)


def _report(case, gv, gt):
    print(f"k1b-exact {case}: grad_v |d|/A {gv[0]:.3g} (bound use {gv[1]:.3g})  "
          f"grad_t |d|/A {gt[0]:.3g} (bound use {gt[1]:.3g})")


def _run(B, hw, C, D, *, n_sets=1, g_dtype=torch.float32, normalize=True, raw_v=False, gv_dtype=torch.float32,
         scale=1.0, gscale=None, seed=0, case=""):
    """Forward + one backward call on the library, checked against the reference built from the call's operands."""
    scale = _f32(scale)
    v, t, G = _inputs(B, hw, C, D, n_sets, seed=seed)
    logits, V, inv_v, t_hat, inv_t = _forward(v, t, C, normalize, scale, raw_v)
    Gk = G if g_dtype == torch.float32 else _bf16_grad(G, C)
    gs = None if gscale is None else torch.tensor([gscale], dtype=torch.float32, device=DEV)
    gv = torch.full((B, hw, D), float("nan"), dtype=gv_dtype, device=DEV)
    gt = torch.zeros(n_sets, C, D, dtype=torch.float32, device=DEV)
    rc = _bwd(Gk, logits, V, inv_v, t_hat, inv_t, C, normalize=normalize, scale=scale, gscale=gs, gv=gv, gt=gt,
              flags=BWD_RAW_V if raw_v else 0)
    assert rc == 0, _lib.last_error()
    torch.cuda.synchronize()
    dev = DEV if B * hw >= 8192 else "cpu"
    _check_forward(logits, V, inv_v, t_hat, C, scale, raw_v, dev)
    mv = lambda x: None if x is None else x.to(dev)
    ref = k1b_reference(mv(Gk), mv(logits), mv(V), mv(inv_v), mv(t_hat), mv(inv_t), normalize=normalize, scale=scale,
                        g=1.0 if gs is None else float(gs), raw_v=raw_v)
    rv = _check(f"{case} grad_v", gv, ref.grad_v, ref.grad_v_A, bf16_out=gv_dtype == torch.bfloat16)
    rt = _check(f"{case} grad_t", gt, ref.grad_t, ref.grad_t_A)
    _report(case, rv, rt)


# (B, hw, C, D, n_sets): each a distinct tiling of the two GEMMs
SHAPES = [
    (16, 1024, 150, 512, 1),     # bench G-A (32^2): the benchmarked step's call
    (16, 16384, 150, 512, 1),    # bench G-B (128^2): several dV tiles per CTA (row factors fetched a tile ahead), deep split-K
    (3, 200, 19, 512, 1),        # last 128-row tile partial; dT 64-pixel blocks straddling two images
    (1, 256, 847, 512, 1),       # four dT class tiles, 53 dV k-blocks
    (2, 136, 300, 320, 1),       # partial last dV n-tile and dT d-tile; dT classes split in two
    (2, 64, 40, 768, 1),         # three dV n-tiles, six dT d-tiles
    (1, 8, 3, 64, 1),            # smallest accepted
    (4, 1024, 150, 512, 4),      # per-image prompts: per-set k ranges in dT
]
# the two combinations the library's callers make: HeadStep (fp32 G from K2, normalise inside the logits GEMM, 1/N_valid
# on the device, bf16 grad_v) and head.cosine_logits / SegHeadLoss (bf16 G, v_hat); plus the step's call with an fp32
# grad_v, which holds the dV epilogue to fp32 resolution where a CTA owns several tiles (G-A: 256 tiles, G-B: 4096)
COMBOS = {
    "step": dict(g_dtype=torch.float32, raw_v=True, gscale=1.0 / 3000, gv_dtype=torch.bfloat16),
    "step_f32": dict(g_dtype=torch.float32, raw_v=True, gscale=1.0 / 3000, gv_dtype=torch.float32),
    "head": dict(g_dtype=torch.bfloat16, raw_v=False, gscale=None, gv_dtype=torch.bfloat16),
}


@pytest.mark.parametrize("combo", sorted(COMBOS))
@pytest.mark.parametrize("B,hw,C,D,n_sets", SHAPES)
def test_backward_exact_operands(B, hw, C, D, n_sets, combo):
    _run(B, hw, C, D, n_sets=n_sets, seed=hw + C + D, case=f"{combo} B{B} hw{hw} C{C} D{D} sets{n_sets}", **COMBOS[combo])


# every route through the entry on one small shape: (G dtype, normalize, RAW_V) where RAW_V is allowed x grad_v dtype
# x logit_scale x grad_scale
ROUTES = [(torch.float32, True, True), (torch.float32, True, False), (torch.float32, False, False),
          (torch.bfloat16, True, False), (torch.bfloat16, False, False)]


def _name(dt):
    return "f32" if dt == torch.float32 else "bf16"


CROSS = [pytest.param(*r, gv, s, gs, id=f"G{_name(r[0])}-norm{int(r[1])}-raw{int(r[2])}-gv{_name(gv)}-s{s:g}-gs{gs}")
         for r, (gv, s, gs) in itertools.product(ROUTES, itertools.product((torch.float32, torch.bfloat16),
                                                                             (1.0, 14.285714), (None, 0.4)))]


@pytest.mark.parametrize("g_dtype,normalize,raw_v,gv_dtype,scale,gscale", CROSS)
def test_backward_path_cross(g_dtype, normalize, raw_v, gv_dtype, scale, gscale):
    _run(2, 200, 40, 320, g_dtype=g_dtype, normalize=normalize, raw_v=raw_v, gv_dtype=gv_dtype, scale=scale,
         gscale=gscale, seed=1, case=f"cross G{_name(g_dtype)} norm{int(normalize)} raw{int(raw_v)} gv{_name(gv_dtype)} "
                                     f"s{scale:g} gs{gscale}")


@pytest.mark.parametrize("g_dtype,normalize,raw_v", [
    pytest.param(torch.float32, True, True, id="Gf32-raw"), pytest.param(torch.bfloat16, False, False, id="Gbf16-plain"),
    pytest.param(torch.bfloat16, True, False, id="Gbf16-norm")])
def test_grad_t_accumulates(g_dtype, normalize, raw_v):
    """d_grad_t is accumulated into (two micro-batches, or the gradient of an earlier loss): prefill + ref."""
    B, hw, C, D = 2, 1024, 150, 512
    scale = _f32(2.0)
    v, t, G = _inputs(B, hw, C, D, seed=5)
    logits, V, inv_v, t_hat, inv_t = _forward(v, t, C, normalize, scale, raw_v)
    Gk = G if g_dtype == torch.float32 else _bf16_grad(G, C)
    ref = k1b_reference(Gk.cpu(), logits.cpu(), V.cpu(), inv_v.cpu(), t_hat.cpu(), inv_t.cpu(), normalize=normalize,
                        scale=scale, raw_v=raw_v)
    # a prefill of the gradient's own size, so that a result written instead of added shows
    pre = (torch.randn(1, C, D, generator=torch.Generator().manual_seed(9), dtype=torch.float64) *
           float(ref.grad_t.std())).float()
    gt = pre.to(DEV, copy=True)
    gv = torch.full((B, hw, D), float("nan"), device=DEV)
    assert _bwd(Gk, logits, V, inv_v, t_hat, inv_t, C, normalize=normalize, scale=scale, gv=gv, gt=gt,
                flags=BWD_RAW_V if raw_v else 0) == 0, _lib.last_error()
    torch.cuda.synchronize()
    _check("grad_t += ", gt, ref.grad_t, ref.grad_t_A, base=pre)
    _check("grad_v", gv, ref.grad_v, ref.grad_v_A)


@pytest.mark.parametrize("g_dtype,raw_v", [pytest.param(torch.float32, False, id="Gf32"),
                                           pytest.param(torch.float32, True, id="Gf32-raw"),
                                           pytest.param(torch.bfloat16, False, id="Gbf16")])
def test_reuse_prep_two_calls(g_dtype, raw_v):
    """LC2IS_BWD_REUSE_PREP, the two-call data-parallel form of the header: d_grad_t first (d_grad_v = NULL), then d_grad_v
    (d_grad_t = NULL, the flag) from the projections and bf16 operand left in the workspace.  Both outputs meet the
    reference and agree with the one-call result within TAU (not bit for bit: r is summed with float atomics)."""
    B, hw, C, D = 4, 1024, 150, 512
    scale, gsv = _f32(14.285714), 0.4
    v, t, G = _inputs(B, hw, C, D, seed=7)
    logits, V, inv_v, t_hat, inv_t = _forward(v, t, C, True, scale, raw_v)
    Gk = G if g_dtype == torch.float32 else _bf16_grad(G, C)
    gs = torch.tensor([gsv], device=DEV)
    raw = BWD_RAW_V if raw_v else 0
    kw = dict(scale=scale, gscale=gs)
    gv1 = torch.full((B, hw, D), float("nan"), device=DEV)
    gt1 = torch.zeros(1, C, D, device=DEV)
    assert _bwd(Gk, logits, V, inv_v, t_hat, inv_t, C, gv=gv1, gt=gt1, flags=raw, **kw) == 0, _lib.last_error()
    ws = torch.full((int(lib.lc2is_cosine_logits_bwd_workspace(B, hw, D, 1, C)),), 0xFF, dtype=torch.uint8, device=DEV)
    gv2 = torch.full((B, hw, D), float("nan"), device=DEV)
    gt2 = torch.zeros(1, C, D, device=DEV)
    assert _bwd(Gk, logits, V, inv_v, t_hat, inv_t, C, gt=gt2, ws=ws, flags=raw, **kw) == 0, _lib.last_error()
    assert _bwd(Gk, logits, V, inv_v, t_hat, inv_t, C, gv=gv2, ws=ws, flags=raw | BWD_REUSE_PREP, **kw) == 0, \
        _lib.last_error()
    torch.cuda.synchronize()
    ref = k1b_reference(Gk.cpu(), logits.cpu(), V.cpu(), inv_v.cpu(), t_hat.cpu(), inv_t.cpu(), scale=scale,
                        g=float(gs), raw_v=raw_v)
    rv = _check("two-call grad_v", gv2, ref.grad_v, ref.grad_v_A)
    rt = _check("two-call grad_t", gt2, ref.grad_t, ref.grad_t_A)
    _report(f"reuse G{_name(g_dtype)} raw{int(raw_v)}", rv, rt)
    _check("one-call grad_v", gv1, ref.grad_v, ref.grad_v_A)
    _check("one-call grad_t", gt1, ref.grad_t, ref.grad_t_A)
    _check("two-call vs one-call grad_v", gv2, gv1.cpu().double(), ref.grad_v_A)
    _check("two-call vs one-call grad_t", gt2, gt1.cpu().double(), ref.grad_t_A)


@pytest.mark.parametrize("B,C,hw", [(2, 150, 1024), (3, 19, 200), (1, 847, 64), (2, 16, 8)])
def test_grad_to_bf16_bit_exact(B, C, hw):
    """lc2is_grad_to_bf16: bf16_rn(G) bit for bit (ties to even, subnormals kept), and the pad rows C..C_pad-1 exactly +0
    even when the output buffer starts as garbage."""
    g = torch.Generator(device=DEV).manual_seed(C)
    G = torch.randn(B, C, hw, generator=g, device=DEV) * 1e-3
    flat = G.view(-1)
    specials = torch.tensor([1.0 + 2.0 ** -8, 1.0 + 3 * 2.0 ** -8, -(1.0 + 2.0 ** -8), 1e-40, -3e-39, 0.0, -0.0,
                             2.0 ** -130], device=DEV)
    flat[: specials.numel()] = specials
    Cp = _lib.class_pad(C)
    out = torch.randint(-32768, 32767, (B, Cp, hw), dtype=torch.int16, device=DEV, generator=g).view(torch.bfloat16)
    assert lib.lc2is_grad_to_bf16(ptr(G), B, C, hw, ptr(out), stream_ptr()) == 0, _lib.last_error()
    ref = G.cpu().to(torch.bfloat16)
    got = out.cpu()
    assert torch.equal(got[:, :C].view(torch.int16), ref.view(torch.int16))
    assert not bool(got[:, C:].view(torch.int16).any())
    assert torch.equal(ops.grad_to_bf16(G.reshape(B, C, 1, hw)).cpu().view(torch.int16), got.view(torch.int16))


def test_argument_errors_are_returned_before_any_launch():
    B, hw, C, D = 3, 16, 5, 64
    v, t, G = _inputs(B, hw, C, D, seed=2)
    logits, V, inv_v, t_hat, inv_t = _forward(v, t, C, True, 1.0, False)
    Gb = _bf16_grad(G, C)
    gv = torch.zeros(B, hw, D, device=DEV)
    gt = torch.zeros(1, C, D, device=DEV)
    args = (logits, V, inv_v, t_hat, inv_t, C)
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    cases = [
        ("REUSE_PREP with d_grad_t", ERR_ARG, dict(G=G, gv=gv, gt=gt, flags=BWD_REUSE_PREP)),
        ("RAW_V with a bf16 G", ERR_ARG, dict(G=Gb, gv=gv, gt=gt, flags=BWD_RAW_V)),
        ("RAW_V without normalize", ERR_ARG, dict(G=G, gv=gv, gt=gt, flags=BWD_RAW_V, normalize=False)),
        ("hw % 8", ERR_SHAPE, dict(G=G, gv=gv, gt=gt, hw=12)),
        ("D % 64", ERR_SHAPE, dict(G=G, gv=gv, gt=gt, D=96)),
        ("n_sets = 2 with B = 3", ERR_SHAPE, dict(G=G, gv=gv, gt=gt, n_sets=2)),
        ("n_sets = 0", ERR_SHAPE, dict(G=G, gv=gv, gt=gt, n_sets=0)),
    ]
    for what, code, kw in cases:
        Gk = kw.pop("G")
        rc = _bwd(Gk, *args, **kw)
        assert rc == code, (what, rc, _lib.last_error())
        assert _lib.launch_count() == n0, what
    # B = 0: nothing to do, nothing launched, no pointer looked at
    assert _bwd(G, *args, gv=gv, gt=gt, B=0) == 0
    assert lib.lc2is_cosine_logits_bwd_ex(None, F32, None, None, None, None, None, 0, hw, D, 1, C, 1, 1.0, None, None,
                                          F32, None, None, stream_ptr(), 0) == 0
    assert _lib.launch_count() == n0
    assert not bool(gv.any()) and not bool(gt.any())


@pytest.mark.parametrize("v_dtype", [torch.bfloat16, torch.float32], ids=_name)
@pytest.mark.parametrize("per_image", [False, True])
def test_cosine_logits_autograd(v_dtype, per_image):
    """head.cosine_logits (bf16 G from lc2is_grad_to_bf16, v_hat, bf16 grad_v for a bf16 V): .grad against the reference
    built from the module's own forward tensors (ops.proto_normalize / ops.cosine_logits_fwd on the same inputs)."""
    B, h, w, C, D = 2, 16, 16, 150, 512
    n_sets = B if per_image else 1
    scale = _f32(14.285714 if per_image else 1.0)
    v, t, G = _inputs(B, h * w, C, D, n_sets, v_dtype=v_dtype, seed=11 + per_image)
    vd = v.clone().requires_grad_(True)
    td = t.clone().requires_grad_(True)
    out = head.cosine_logits(vd, td, logit_scale=scale, hw_shape=(h, w))
    out.backward(G.reshape(B, C, h, w))
    t_hat, inv_t = ops.proto_normalize(t, True)
    logits, v_hat, inv_v = ops.cosine_logits_fwd(v, t_hat, C, (h, w), True, scale)
    assert torch.equal(logits, out.detach())
    assert vd.grad.dtype == v_dtype and td.grad.shape == t.shape
    Gb = ops.grad_to_bf16(G.reshape(B, C, h, w))
    ref = k1b_reference(Gb.cpu(), logits.cpu(), v_hat.cpu(), inv_v.cpu(), t_hat.cpu(), inv_t.cpu(), scale=scale)
    rv = _check("module grad_v", vd.grad, ref.grad_v, ref.grad_v_A, bf16_out=v_dtype == torch.bfloat16)
    rt = _check("module grad_t", td.grad.reshape(n_sets, C, D), ref.grad_t, ref.grad_t_A)
    _report(f"head.cosine_logits v{_name(v_dtype)} sets{n_sets}", rv, rt)


def test_head_step_backward():
    """The benchmarked step: HeadStep at bench G-A (B = 16, 32^2 -> 512^2, C = 150) on synthetic inputs.  Its grad_v (bf16)
    and grad_t against the reference built from its own buffers: K2's un-scaled fp32 gradient (grad_low, read before the
    next call reuses the block), the logits, the raw V, inv_v, t_hat, inv_t and the 1/N_valid on the device."""
    from lc2is_b200 import synthetic
    from lc2is_b200.step import HeadStep
    B, h, H, C, D = 16, 32, 512, 150, 512
    v = synthetic.make_patch_embeddings(B, h * h, D, dtype=torch.bfloat16).to(DEV)
    t = synthetic.make_prototypes(C, D).to(DEV)
    labels = synthetic.make_labels(B, H, H, C, ignore_frac=0.1).to(DEV)
    step = HeadStep(B, h, h, H, H, C, D, ignore_index=0)
    assert step.fuse_norm and step.fused
    step(v, t, labels)
    torch.cuda.synchronize()
    G = step.grad_low.clone()
    gscale = float(step._blk.gscale)
    assert abs(gscale * int(step.n_valid) - 1) < 1e-6
    ref = k1b_reference(G, step.logits, v.reshape(B * h * h, D), step.inv_v, step.t_hat, step.inv_t, g=gscale, raw_v=True)
    rv = _check("HeadStep grad_v", step.grad_v, ref.grad_v, ref.grad_v_A, bf16_out=True)
    rt = _check("HeadStep grad_t", step.grad_t, ref.grad_t, ref.grad_t_A)
    _report("HeadStep G-A", rv, rt)
