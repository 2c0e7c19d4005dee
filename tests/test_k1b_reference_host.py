"""Host side of the exact-operand K1b tests (no GPU needed): the float64 reference of tests/k1b_reference.py, fed unrounded
float64 operands, against torch.autograd of oracle.cosine_logits in float64 - normalize on / off, shared and per-image
prototypes, s != 1, g != 1 - plus the LC2IS_BWD_RAW_V algebra, the r / rt projection identity, the operand rounding and
check_bound on partial blocks."""
import pytest
import torch
import torch.nn.functional as F

from k1b_reference import TAU, check_bound, gemm_operand, k1b_reference, projections
from oracle import head_oracle as O

f64 = torch.float64


def _operands(B, h, w, C, D, n_sets, normalize, scale, seed=7):
    """Exact float64 forward tensors in the library's layouts: v_hat [B*hw, D], inv_v, t_hat [n_sets, C, D], inv_t, logits
    [B, C, h, w]; plus the raw v / t and a gradient G."""
    g = torch.Generator().manual_seed(seed)
    hw = h * w
    t = torch.randn(*((n_sets,) if n_sets > 1 else ()), C, D, generator=g, dtype=f64)
    v = torch.randn(B, hw, D, generator=g, dtype=f64) * (0.5 + torch.rand(B, hw, 1, generator=g, dtype=f64))
    v = v + 2.0 * t.reshape(-1, C, D)[0, torch.randint(0, C, (B, hw), generator=g)]     # large cosines, like real scores
    if normalize:
        v_hat, t_hat = F.normalize(v, dim=2), F.normalize(t, dim=-1)
        inv_v, inv_t = 1 / v.norm(dim=2), 1 / t.norm(dim=-1)
    else:
        v_hat, t_hat = v, t
        inv_v, inv_t = torch.ones(B, hw, dtype=f64), torch.ones(*t.shape[:-1], dtype=f64)
    t3 = t_hat.reshape(-1, C, D)
    logits = scale * torch.einsum("bpd,bcd->bcp", v_hat, t3.expand(B, -1, -1) if n_sets == 1 else t3)
    G = torch.randn(B, C, h, w, generator=g, dtype=f64) * 1e-3
    return dict(v=v, t=t, v_hat=v_hat.reshape(B * hw, D), inv_v=inv_v.reshape(-1), t_hat=t3,
                inv_t=inv_t.reshape(-1, C), logits=logits.reshape(B, C, h, w), G=G)


def _autograd(v, t, G, normalize, scale, gs):
    v = v.clone().requires_grad_(True)
    t = t.clone().requires_grad_(True)
    out = O.cosine_logits(v, t, normalize=normalize, logit_scale=scale, hw_shape=G.shape[-2:])
    return torch.autograd.grad(out, (v, t), grad_outputs=gs * G)


@pytest.mark.parametrize("normalize", [True, False])
@pytest.mark.parametrize("n_sets", [1, 3])
@pytest.mark.parametrize("scale,gs", [(1.0, 1.0), (14.285714, 0.37)])
def test_reference_equals_autograd_of_the_oracle(normalize, n_sets, scale, gs):
    B, h, w, C, D = 3, 4, 6, 11, 40
    x = _operands(B, h, w, C, D, n_sets, normalize, scale)
    ref = k1b_reference(x["G"], x["logits"], x["v_hat"], x["inv_v"], x["t_hat"], x["inv_t"], normalize=normalize,
                        scale=scale, g=gs)
    gv, gt = _autograd(x["v"], x["t"], x["G"], normalize, scale, gs)
    assert ref.grad_v.dtype == f64 and ref.grad_v.shape == (B, h * w, D) and ref.grad_t.shape == (n_sets, C, D)
    torch.testing.assert_close(ref.grad_v, gv, rtol=0, atol=1e-12 * float(gv.abs().max()))
    torch.testing.assert_close(ref.grad_t, gt.reshape(n_sets, C, D), rtol=0, atol=1e-12 * float(gt.abs().max()))
    # the error scale bounds the value it belongs to, and is not vacuous
    for val, A in ((ref.grad_v, ref.grad_v_A), (ref.grad_t, ref.grad_t_A)):
        assert bool((val.abs() <= A * (1 + 1e-12)).all())
        assert float(A.max()) <= 1e3 * float(val.abs().max())


@pytest.mark.parametrize("n_sets", [1, 2])
def test_raw_v_algebra_equals_the_v_hat_algebra(n_sets):
    """LC2IS_BWD_RAW_V: GEMMs on the raw V with the operand G * inv_v, the normalise-backward folded into the dV epilogue
    (V inv^2 r) - the same numbers as the v_hat form in exact arithmetic."""
    B, h, w, C, D = 2, 5, 4, 9, 24
    scale, gs = 3.5, 0.8
    x = _operands(B, h, w, C, D, n_sets, True, scale, seed=11)
    a = k1b_reference(x["G"], x["logits"], x["v_hat"], x["inv_v"], x["t_hat"], x["inv_t"], scale=scale, g=gs)
    b = k1b_reference(x["G"], x["logits"], x["v"].reshape(B * h * w, D), x["inv_v"], x["t_hat"], x["inv_t"], scale=scale,
                      g=gs, raw_v=True)
    torch.testing.assert_close(b.grad_v, a.grad_v, rtol=0, atol=1e-12 * float(a.grad_v.abs().max()))
    torch.testing.assert_close(b.grad_t, a.grad_t, rtol=0, atol=1e-12 * float(a.grad_t.abs().max()))
    torch.testing.assert_close(b.grad_v_A, a.grad_v_A, rtol=1e-12, atol=0)
    with pytest.raises(ValueError):
        k1b_reference(x["G"], x["logits"], x["v_hat"], x["inv_v"], x["t_hat"], x["inv_t"], normalize=False, raw_v=True)


def test_projection_identity():
    """r[m] = <v_hat_m, dV_hat_m> / g and rt[c] = <t_hat_c, dT_hat_c> / g: the only dot products the normalise-backward
    needs, formed from the logits instead of a second pass over D."""
    B, h, w, C, D, s = 2, 3, 8, 7, 32, 2.5
    x = _operands(B, h, w, C, D, 2, True, s, seed=5)
    G = x["G"].reshape(B, C, h * w)
    vh = x["v_hat"].reshape(B, h * w, D)
    dvh = s * torch.einsum("bcp,bcd->bpd", G, x["t_hat"])
    dth = s * torch.einsum("bcp,bpd->bcd", G, vh)
    r, r_abs, rt, rt_abs = projections(x["G"], x["logits"], 2)
    torch.testing.assert_close(r, (vh * dvh).sum(2), rtol=0, atol=1e-13)
    torch.testing.assert_close(rt, (x["t_hat"] * dth).sum(2), rtol=0, atol=1e-13)
    assert bool((r.abs() <= r_abs).all()) and bool((rt.abs() <= rt_abs).all())
    # shared prototypes: rt sums over every image
    _, _, rt1, _ = projections(x["G"], x["logits"], 1)
    torch.testing.assert_close(rt1[0], rt.sum(0), rtol=0, atol=1e-13)


def test_gemm_operand_rounding():
    """fp32 G -> bf16 round-to-nearest-even; RAW_V: one fp32 multiply by inv_v, then the rounding (not the float64 product
    rounded); a bf16 G [B, C_pad, hw] is its own operand without its pad rows."""
    g = torch.Generator().manual_seed(3)
    B, C, Cp, h, w = 2, 5, 16, 2, 4
    G = torch.randn(B, C, h, w, generator=g)
    inv = torch.rand(B * h * w, generator=g) + 0.5
    op = gemm_operand(G, C)
    assert op.dtype == f64 and op.shape == (B, C, h * w)
    assert torch.equal(op, G.reshape(B, C, -1).to(torch.bfloat16).double())
    raw = gemm_operand(G, C, inv)
    assert torch.equal(raw, (G.reshape(B, C, -1) * inv.reshape(B, 1, -1)).to(torch.bfloat16).double())
    # a product whose fp32 rounding lands exactly on a bf16 tie: fp32 first, then the tie goes to even
    Gt = torch.full((1, 1, 1, 8), 1.0 + 2.0 ** -8 + 2.0 ** -23)
    it = torch.full((8,), 1.0 - 2.0 ** -24)
    assert float(Gt[0, 0, 0, 0]) * float(it[0]) > 1.0 + 2.0 ** -8          # the exact product would round up
    assert float(gemm_operand(Gt, 1, it)[0, 0, 0]) == 1.0
    Gbf = torch.zeros(B, Cp, h * w, dtype=torch.bfloat16)
    Gbf[:, :C] = G.reshape(B, C, -1).to(torch.bfloat16)
    assert torch.equal(gemm_operand(Gbf, C), op)
    with pytest.raises(ValueError):
        gemm_operand(Gbf, C, inv)


def test_check_bound_on_partial_blocks_names_the_block():
    """A [rows, channels] matrix whose sizes are not multiples of the [128 x 64] block: within the bound it passes and
    reports the worst ratio; one element over the bound, or one NaN (an unwritten element), fails and names its block."""
    g = torch.Generator().manual_seed(4)
    R, D = 300, 272
    ref = torch.randn(R, D, generator=g, dtype=f64)
    A = ref.abs() + 1
    worst, use = check_bound("within", ref + 0.5 * TAU * A, ref, A)
    assert abs(worst - 0.5 * TAU) <= 1e-3 * TAU and 0.49 < use <= 0.5 + 1e-9
    bad = ref.clone()
    bad[257, 270] += 2 * TAU * A[257, 270]
    with pytest.raises(AssertionError, match=r"1 of 15 .* rows 256\.\., channels 256\.\."):
        check_bound("over", bad, ref, A)
    bad = ref.clone()
    bad[130, 3] = float("nan")
    with pytest.raises(AssertionError, match=r"rows 128\.\., channels 0\.\."):
        check_bound("unwritten", bad, ref, A)
