"""K0/K1/K1b parity: cosine-logits tensor-core GEMM (tcgen05/TMEM/TMA) and its backward.

Tolerances:
  v_hat / t_hat : bf16(fp32 normalise) - at most 1 bf16 ulp from the oracle's rounding (fp32 norm
                  summation order differs), on < 0.5 % of the elements
  logits        : vs fp32 matmul of the kernel's OWN bf16 operands: |d| <= 2e-6 * scale (fp32
                  accumulation order only); vs the full-fp32 reference: |d| <= 4e-3 * scale
                  (bf16 unit round-off 2^-9, SURVEY 8c)
  grad_v/grad_t : per element |d| <= 2^-16 * A vs a float64 evaluation of K1b's arithmetic on its OWN operands, A = the
                  abs-sum of the same expression (+ 2^-8 |ref| for a bf16 grad_v): tests/test_gpu_k1b_exact.py; here the
                  second check, rel 2e-2 of max|grad| vs the fp32 autograd oracle (bf16 operands and bf16 dL/dlogits)
"""
import os

import pytest
import torch

from oracle import head_oracle as O
from lc2is_b200 import head, ops, synthetic

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _bf16_ulp_check(got, ref32):
    """got: bf16 tensor; ref32: fp32 values before rounding."""
    ref = ref32.to(torch.bfloat16)
    diff = (got.float() - ref.float()).abs()
    ulp = torch.maximum(ref.float().abs(), torch.tensor(1e-30)) * 2.0 ** -7
    assert bool((diff <= ulp).all())
    assert float((diff > 0).float().mean()) < 5e-3


@pytest.mark.parametrize("B,hw,C,dtype,normalize,scale", [
    (2, 64, 151, torch.float32, True, 1.0),       # golden geometry
    (2, 1024, 150, torch.bfloat16, True, 1.0),    # 32^2 grid
    (1, 16384, 151, torch.bfloat16, True, 14.285714),   # 128^2 grid, temperature 1/0.07
    (3, 200, 19, torch.float32, True, 1.0),       # ragged: hw not a multiple of 128
    (2, 256, 847, torch.bfloat16, True, 1.0),     # open-vocab: 4 N-tiles
    (2, 128, 151, torch.float32, False, 1.0),     # un-normalised (model.py:50)
    (1, 1, 3, torch.float32, True, 1.0),
])
def test_logits(B, hw, C, dtype, normalize, scale):
    D = 512
    v = synthetic.make_patch_embeddings(B, hw, D, dtype=dtype)
    t = synthetic.make_prototypes(C, D)
    t_hat, inv_t = ops.proto_normalize(t.to(DEV), normalize)
    h = int(hw ** 0.5); hw_shape = (h, hw // h) if h * (hw // h) == hw else (1, hw)
    logits, v_hat, inv_v = ops.cosine_logits_fwd(v.to(DEV), t_hat, C, hw_shape, normalize, scale)
    Cp = ops._lib.class_pad(C)
    assert t_hat.shape == (1, Cp, D) and float(t_hat[0, C:].float().abs().max() if Cp > C else 0.0) == 0.0
    v32, t32 = v.float(), t.float()
    if normalize:
        _bf16_ulp_check(v_hat.cpu(), torch.nn.functional.normalize(v32, dim=2).reshape(-1, D))
        _bf16_ulp_check(t_hat[0, :C].cpu(), torch.nn.functional.normalize(t32, dim=1))
        torch.testing.assert_close(inv_v.cpu(), 1 / v32.norm(dim=2).reshape(-1).clamp_min(1e-12), rtol=1e-5, atol=0)
    else:
        assert torch.equal(v_hat.cpu(), v32.to(torch.bfloat16).reshape(-1, D))
    # exact-operand check
    ref_same = scale * torch.einsum("bpd,cd->bcp", v_hat.float().reshape(B, hw, D), t_hat[0, :C].float()).cpu()
    got = logits.reshape(B, C, hw).cpu()
    mag = float(ref_same.abs().max())
    assert float((got - ref_same).abs().max()) <= 2e-6 * max(mag, scale), float((got - ref_same).abs().max())
    # reference (fp32) check
    ref = O.cosine_logits(v32, t32, normalize=normalize, logit_scale=scale, hw_shape=hw_shape).reshape(B, C, hw)
    tol = 4e-3 * (scale if normalize else float(ref.abs().max()))
    assert float((got - ref).abs().max()) <= tol


def test_golden_final_py(golden_dir):
    g = torch.load(os.path.join(golden_dir, "head_final.pt"))
    t = synthetic.load_prototypes()
    low = head.cosine_logits(g["v"].to(DEV), t.to(DEV))
    assert low.shape == g["score_low"].shape
    assert float((low.cpu() - g["score_low"]).abs().max()) <= 4e-3
    raw = head.cosine_logits(g["v"].to(DEV), t.to(DEV), normalize=False)
    assert float((raw.cpu() - g["raw"]).abs().max()) <= 4e-3 * float(g["raw"].abs().max())


def test_per_image_prompts():
    """final.py:129-130: text embeddings differ per image ([B,K,D])."""
    B, hw, C, D = 3, 256, 151, 512
    v = synthetic.make_patch_embeddings(B, hw, D, dtype=torch.float32)
    t = torch.stack([synthetic.make_prototypes(C, D) + 0.3 * i for i in range(B)])
    got = head.cosine_logits(v.to(DEV), t.to(DEV))
    ref = O.cosine_logits(v, t)
    assert float((got.cpu() - ref).abs().max()) <= 4e-3


@pytest.mark.parametrize("B,hw,C,normalize,per_image", [
    (2, 256, 151, True, False),
    (1, 1024, 150, True, False),
    (2, 200, 19, True, False),
    (2, 128, 151, False, False),
    (2, 128, 40, True, True),
    (1, 256, 847, True, False),
])
def test_backward(B, hw, C, normalize, per_image):
    D = 512
    g = torch.Generator().manual_seed(31)
    v = synthetic.make_patch_embeddings(B, hw, D, dtype=torch.float32)
    t = synthetic.make_prototypes(C, D)
    if per_image:
        t = torch.stack([t + 0.2 * i for i in range(B)])
    h = int(hw ** 0.5); hw_shape = (h, hw // h) if h * (hw // h) == hw else (1, hw)
    G = torch.randn(B, C, *hw_shape, generator=g) * 1e-3
    gv_ref, gt_ref = O.cosine_logits_backward(v, t, G, normalize=normalize)
    vd = v.to(DEV).requires_grad_(True)
    td = t.to(DEV).requires_grad_(True)
    out = head.cosine_logits(vd, td, normalize=normalize, hw_shape=hw_shape)
    out.backward(G.to(DEV))
    ev = float((vd.grad.cpu() - gv_ref).abs().max() / gv_ref.abs().max())
    et = float((td.grad.cpu() - gt_ref).abs().max() / gt_ref.abs().max())
    assert ev < 2e-2 and et < 2e-2, (ev, et)


def test_fused_head_loss_matches_oracle():
    B, h, H, C, D = 2, 32, 128, 151, 512
    v = synthetic.make_patch_embeddings(B, h * h, D, dtype=torch.float32)
    t = synthetic.make_prototypes(C, D)
    labels = synthetic.make_labels(B, H, H, C, block=8, ignore_frac=0.1)
    ref = O.head_step(v, t, labels, ignore_index=0, n_cls=C)
    vd = v.to(DEV).requires_grad_(True)
    td = t.to(DEV).requires_grad_(True)
    loss, low, n_valid = head.SegHeadLoss(ignore_index=0)(vd, td, labels.to(DEV))
    (0.4 * loss).backward()
    assert abs(float(loss) - float(ref["loss"])) <= 1e-4 * float(ref["loss"])
    assert int(n_valid) == int((labels != 0).sum())
    ev = float((vd.grad.cpu() - 0.4 * ref["grad_v"]).abs().max() / (0.4 * ref["grad_v"]).abs().max())
    et = float((td.grad.cpu() - 0.4 * ref["grad_t"]).abs().max() / (0.4 * ref["grad_t"]).abs().max())
    assert ev < 3e-2 and et < 3e-2, (ev, et)


@pytest.mark.parametrize("M,K,N,out_dtype", [(300, 768, 512, torch.bfloat16), (1024, 768, 512, torch.float32),
                                              (129, 64, 16, torch.float32), (5000, 384, 272, torch.bfloat16),
                                              (777, 128, 192, torch.float32), (2049, 192, 384, torch.bfloat16),
                                              (64, 64, 48, torch.bfloat16)])
def test_linear_projection_gemm(M, K, N, out_dtype):
    """lc2is_linear_fwd (TextToPatch.visual forward on the tcgen05 pipeline): against an fp32 matmul of the same
    bf16-rounded operands (accumulation order only) and against the fp32 nn.Linear (bf16 operand rounding)."""
    g = torch.Generator().manual_seed(12)
    x = torch.randn(M, K, generator=g)
    w = torch.randn(N, K, generator=g) * K ** -0.5
    b = torch.randn(N, generator=g)
    xb, wb = x.to(torch.bfloat16), w.to(torch.bfloat16)
    y = ops.linear_fwd(xb.to(DEV), wb.to(DEV), b.to(DEV), out_dtype).float().cpu()
    ref_same = xb.float() @ wb.float().t() + b
    ref_fp32 = x @ w.t() + b
    tol = 2e-5 if out_dtype == torch.float32 else 1.0 / 128          # bf16 output rounding
    assert float((y - ref_same).abs().max()) <= tol * float(ref_same.abs().max())
    assert float((y - ref_fp32).abs().max()) <= 2e-2 * float(ref_fp32.abs().max())


@pytest.mark.parametrize("M,K,N,out_dtype", [(32768, 768, 512, torch.bfloat16), (40960, 128, 256, torch.float32),
                                              (38912, 768, 512, torch.float32)])
def test_linear_projection_gemm_two_sm_form(M, K, N, out_dtype):
    """Shapes that take the cta_group::2 kernel on a 148-SM B200 (M % 256 == 0, N % 256 == 0, at least two 256 x 256
    pair tiles per CTA pair: 148); tests/test_gpu_linear_exact.py asserts the route by kernel name.  Same checks as
    above, on the device (the fp32 reference of a 32768 x 768 x 512 product is computed by torch there)."""
    g = torch.Generator(device=DEV).manual_seed(13)
    x = torch.randn(M, K, generator=g, device=DEV)
    w = torch.randn(N, K, generator=g, device=DEV) * K ** -0.5
    b = torch.randn(N, generator=g, device=DEV)
    xb, wb = x.to(torch.bfloat16), w.to(torch.bfloat16)
    y = ops.linear_fwd(xb, wb, b, out_dtype).float()
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        ref_same = xb.float() @ wb.float().t() + b
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old
    tol = 2e-5 if out_dtype == torch.float32 else 1.0 / 128
    err = (y - ref_same).abs()
    assert float(err.max()) <= tol * float(ref_same.abs().max()), (float(err.max()), int(err.argmax()) // N, int(err.argmax()) % N)
    # every row block and channel block written (no tile skipped): per-block error maxima are all small
    blk = err.view(M // 128, 128, N // 128, 128).amax(dim=(1, 3))
    assert float(blk.max()) <= tol * float(ref_same.abs().max())


def test_text_to_patch_module_matches_reference_module(golden_dir):
    """TextToPatch (model/text_patch.py:4-18) with the reference's weights: same parameter names, text first, visual
    projection forward AND backward on the tcgen05 GEMMs (bf16 operands, fp32 accumulation, fp32 weight gradient)."""
    from lc2is_b200.model.text_patch import TextToPatch
    torch.manual_seed(3)
    m = TextToPatch(768, 512, 512, tensor_cores=True).to(DEV)
    assert sorted(k for k, _ in m.named_parameters()) == ["textual.bias", "textual.weight", "visual.bias", "visual.weight"]
    img = torch.randn(2, 64, 768, device=DEV, requires_grad=True)
    text = torch.randn(151, 512, device=DEV)
    t_f, v_f = m(img, text)
    assert t_f.shape == (151, 512) and v_f.shape == (2, 64, 512)
    ref_v = torch.nn.functional.linear(img, m.visual.weight, m.visual.bias)
    assert float((v_f - ref_v).abs().max()) <= 2e-2 * float(ref_v.abs().max())
    v_f.square().mean().backward()
    ref_g = torch.autograd.grad(ref_v.square().mean(), [img, m.visual.weight, m.visual.bias])
    for got, ref in ((img.grad, ref_g[0]), (m.visual.weight.grad, ref_g[1]), (m.visual.bias.grad, ref_g[2])):
        assert float((got - ref).abs().max()) <= 3e-2 * float(ref.abs().max())
    assert m.visual.weight.grad.dtype == torch.float32
    # fp32 inputs without the opt-in keep nn.Linear's fp32 arithmetic; bf16 inputs take the tensor-core path
    m32 = TextToPatch(768, 512, 512).to(DEV)
    m32.load_state_dict(m.state_dict())
    _, v32 = m32(img.detach(), text)
    assert torch.equal(v32, torch.nn.functional.linear(img.detach(), m.visual.weight, m.visual.bias))
    _, vb = m32(img.detach().to(torch.bfloat16), text)
    assert vb.dtype == torch.bfloat16 and float((vb.float() - ref_v).abs().max()) <= 3e-2 * float(ref_v.abs().max())


@pytest.mark.parametrize("M,K,N,gx_dtype", [(300, 768, 512, torch.bfloat16), (4096, 768, 512, torch.float32),
                                              (129, 64, 64, torch.float32), (5000, 384, 192, torch.bfloat16),
                                              (32768, 768, 512, torch.bfloat16), (70000, 128, 256, torch.float32)])
def test_linear_projection_backward(M, K, N, gx_dtype):
    """lc2is_linear_bwd (autograd of text_patch.py:12,17): dX, dW, db against fp32 matmuls of the same bf16-rounded
    operands (accumulation order / split-K reduction order only).  Tolerances: dX 2e-5 (fp32 out) or 2^-7 (bf16 out)
    of max|dX|; dW and db 2e-5 of their maxima (fp32 accumulation over up to 70000 rows)."""
    g = torch.Generator(device=DEV).manual_seed(21)
    x = torch.randn(M, K, generator=g, device=DEV).to(torch.bfloat16)
    w = (torch.randn(N, K, generator=g, device=DEV) * K ** -0.5).to(torch.bfloat16)
    gy = torch.randn(M, N, generator=g, device=DEV).to(torch.bfloat16)
    gx, gw, gb = ops.linear_bwd(gy, x, w, gx_dtype=gx_dtype)
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        ref_gx = gy.float() @ w.float()
        ref_gw = gy.double().t() @ x.double()
        ref_gb = gy.double().sum(0)
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old
    tol = 2e-5 if gx_dtype == torch.float32 else 1.0 / 128
    assert float((gx.float() - ref_gx).abs().max()) <= tol * float(ref_gx.abs().max())
    assert gw.dtype == torch.float32 and float((gw.double() - ref_gw).abs().max()) <= 2e-5 * float(ref_gw.abs().max())
    assert float((gb.double() - ref_gb).abs().max()) <= 2e-5 * float(ref_gb.abs().max())
    # accumulation into caller-owned buffers (two micro-batches) and partial requests
    gw2, gb2 = gw.clone(), gb.clone()
    out = ops.linear_bwd(gy, x, w, need_gx=False, gw=gw2, gb=gb2)
    assert out[0] is None
    assert float((gw2.double() - 2 * ref_gw).abs().max()) <= 4e-5 * float(ref_gw.abs().max())
    assert float((gb2.double() - 2 * ref_gb).abs().max()) <= 4e-5 * float(ref_gb.abs().max())


@pytest.mark.parametrize("B,hw,C,scale", [
    (2, 1024, 150, 1.0),          # 32^2 grid, one tile per SM
    (1, 16384, 151, 14.285714),   # 128^2 grid: several tiles per CTA (double-buffered row factors)
    (3, 200, 19, 1.0),            # ragged: hw not a multiple of 128 (rows of the next image / zero rows in the tile)
    (2, 256, 847, 1.0),           # four N-tiles: the norm is recomputed per N-tile
])
def test_logits_fused_norm(B, hw, C, scale):
    """d_v_hat = NULL: the row normalisation runs inside the GEMM (norm warps + epilogue scaling), no v_hat.
    Operands of the tensor cores are the RAW bf16 V and bf16 t_hat; the fp32 row factor multiplies the accumulator."""
    D = 512
    v = synthetic.make_patch_embeddings(B, hw, D, dtype=torch.bfloat16)
    t = synthetic.make_prototypes(C, D)
    t_hat, _ = ops.proto_normalize(t.to(DEV), True)
    h = int(hw ** 0.5); hw_shape = (h, hw // h) if h * (hw // h) == hw else (1, hw)
    logits, v_hat, inv_v = ops.cosine_logits_fwd(v.to(DEV), t_hat, C, hw_shape, True, scale, fuse_norm=True)
    assert v_hat is None
    v32 = v.float()
    torch.testing.assert_close(inv_v.cpu(), 1 / v32.norm(dim=2).reshape(-1).clamp_min(1e-12), rtol=1e-5, atol=0)
    got = logits.reshape(B, C, hw).cpu()
    ref_same = scale * inv_v.cpu().view(B, 1, hw) * torch.einsum("bpd,cd->bcp", v32, t_hat[0, :C].float().cpu())
    assert float((got - ref_same).abs().max()) <= 2e-6 * max(float(ref_same.abs().max()), scale)
    ref = O.cosine_logits(v32, t.float(), normalize=True, logit_scale=scale, hw_shape=hw_shape).reshape(B, C, hw)
    assert float((got - ref).abs().max()) <= 4e-3 * scale
    # and the legacy two-kernel route agrees within the bf16 rounding of v_hat
    legacy, _, _ = ops.cosine_logits_fwd(v.to(DEV), t_hat, C, hw_shape, True, scale)
    assert float((legacy.reshape(B, C, hw).cpu() - got).abs().max()) <= 4e-3 * scale


@pytest.mark.parametrize("B,hw,C", [(2, 256, 151), (1, 1024, 150), (2, 200, 19), (1, 256, 847)])
def test_backward_raw_v(B, hw, C):
    """LC2IS_BWD_RAW_V: both backward GEMMs on the raw V (the bf16 operand is G * inv||v||, the normalise-backward sits in
    the dV epilogue) against the fp32 autograd oracle and against the v_hat route."""
    D = 512
    g = torch.Generator().manual_seed(33)
    v = synthetic.make_patch_embeddings(B, hw, D, dtype=torch.bfloat16)
    t = synthetic.make_prototypes(C, D)
    h = int(hw ** 0.5); hw_shape = (h, hw // h) if h * (hw // h) == hw else (1, hw)
    G = torch.randn(B, C, *hw_shape, generator=g) * 1e-3
    gv_ref, gt_ref = O.cosine_logits_backward(v.float(), t, G, normalize=True)
    t_hat, inv_t = ops.proto_normalize(t.to(DEV), True)
    vd, Gd = v.to(DEV), G.to(DEV)
    logits, _, inv_v = ops.cosine_logits_fwd(vd, t_hat, C, hw_shape, True, 1.0, fuse_norm=True)
    gv, gt = ops.cosine_logits_bwd(Gd, logits, vd, inv_v, t_hat, inv_t, C, raw_v=True)
    ev = float((gv.cpu() - gv_ref).abs().max() / gv_ref.abs().max())
    et = float((gt[0].cpu() - gt_ref).abs().max() / gt_ref.abs().max())
    assert ev < 2e-2 and et < 2e-2, (ev, et)
    logits2, v_hat, inv_v2 = ops.cosine_logits_fwd(vd, t_hat, C, hw_shape, True, 1.0)
    gv2, gt2 = ops.cosine_logits_bwd(Gd, logits2, v_hat, inv_v2, t_hat, inv_t, C)
    assert float((gv - gv2).abs().max()) <= 2e-2 * float(gv2.abs().max())
    assert float((gt - gt2).abs().max()) <= 2e-2 * float(gt2.abs().max())


# ---- producer of the projection: bicubic x4 of the token-major feature map (model/model.py:42-44) -----------------------
@pytest.mark.parametrize("B,h,w,C,in_dtype,out_dtype", [
    (2, 8, 8, 64, torch.float32, torch.float32), (1, 32, 32, 768, torch.float32, torch.bfloat16),
    (2, 5, 7, 12, torch.float32, torch.float32), (1, 1, 1, 4, torch.float32, torch.float32),
    (2, 6, 4, 32, torch.bfloat16, torch.bfloat16), (1, 2, 9, 8, torch.bfloat16, torch.float32)])
def test_bicubic4_tokens_forward_and_backward(B, h, w, C, in_dtype, out_dtype):
    """lc2is_bicubic4_tokens_fwd / _bwd against the reference lines (oracle.upsample_tokens_bicubic4 = rearrange +
    F.interpolate(bicubic, x4) + rearrange on CPU, and its autograd).  Tolerance: fp32 evaluation order (1e-5 of the maximum)
    or the bf16 rounding of the output (2^-8 relative)."""
    from lc2is_b200 import head
    g = torch.Generator().manual_seed(5)
    x = torch.randn(B, h * w, C, generator=g).to(in_dtype)
    xr = x.float().clone().requires_grad_(True)
    if h == w:
        ref = O.upsample_tokens_bicubic4(xr, h)
    else:                                                    # the reference line needs the grid shape for non-square maps
        t = xr.permute(0, 2, 1).reshape(B, C, h, w)
        ref = torch.nn.functional.interpolate(t, mode="bicubic", scale_factor=4).reshape(B, C, 16 * h * w).permute(0, 2, 1)
    xd = x.to(DEV).requires_grad_(True)
    y = head.upsample_tokens_bicubic4(xd, (h, w), out_dtype)
    assert y.shape == (B, 16 * h * w, C) and y.dtype == out_dtype
    tol = 1e-5 if out_dtype == torch.float32 else 2.0 ** -8
    assert float((y.float().cpu() - ref).abs().max()) <= tol * float(ref.abs().max())
    gy = torch.randn(B, 16 * h * w, C, generator=g).to(torch.bfloat16).float()       # representable in either output dtype
    ref.backward(gy)
    y.backward(gy.to(DEV).to(out_dtype))
    tolg = 1e-5 if in_dtype == torch.float32 else 2.0 ** -7                         # bf16 input: gradient rounded to bf16
    assert xd.grad.dtype == in_dtype
    assert float((xd.grad.float().cpu() - xr.grad).abs().max()) <= tolg * float(xr.grad.abs().max())


def test_bicubic4_tokens_feed_the_projection():
    """The chain of model.py:42-47 on the kernels: tokens -> bicubic x4 (bf16 rows) -> TextToPatch.visual (tcgen05), against
    the reference lines in fp32 (bf16 operand rounding: 2e-2 of the maximum)."""
    from lc2is_b200 import head
    from lc2is_b200.model.text_patch import TextToPatch
    torch.manual_seed(2)
    B, h, C = 2, 8, 768
    m = TextToPatch(C, 512, 512).to(DEV)
    dec = torch.randn(B, h * h, C, device=DEV)
    up = head.upsample_tokens_bicubic4(dec, (h, h))                       # bf16 rows -> tensor-core projection
    _, v = m(up, torch.randn(151, 512, device=DEV))
    ref = torch.nn.functional.linear(O.upsample_tokens_bicubic4(dec.cpu(), h).to(DEV), m.visual.weight, m.visual.bias)
    assert v.shape == (B, 16 * h * h, 512)
    assert float((v.float() - ref).abs().max()) <= 2e-2 * float(ref.abs().max())
