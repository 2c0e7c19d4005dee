"""Float64 reference of the cosine-logits backward (K1b, ``lc2is_cosine_logits_bwd[_ex]``) evaluated on the tensors the
kernels actually consume, for the exact-operand K1b tests.  TEST INFRASTRUCTURE ONLY (nothing under lc2is_b200/ imports it).

With logits L = s * <v_hat, t_hat> (the forward's fp32 output), the fp32 gradient G = dL/dlogits and the upstream scalar g:

* GEMM operand  Gb = bf16_rn(G)                       (fp32 G; bf16 G is its own operand)
                Gb = bf16_rn(fp32(G * inv_v[m]))      (LC2IS_BWD_RAW_V: an fp32 multiply, then round to nearest even)
* projections   r[m] = sum_c G L,   rt[set,c] = sum_m G L   from the UNROUNDED G (k1b_prep_f32_kernel; on the bf16-G
                route G is the bf16 tensor itself)
* dV  normalize  inv[m] * (s g sum_c Gb t_hat[c,d] - v_hat[m,d] g r[m])
      RAW_V      s g sum_c Gb t_hat[c,d] - V[m,d] g inv[m]^2 r[m]
      otherwise  s g sum_c Gb t_hat[c,d]
* dT  normalize  inv_t[c] g (s sum_m Gb v_hat[m,d] - t_hat[c,d] rt[c])      (V in place of v_hat under RAW_V)
      otherwise  g s sum_m Gb v_hat[m,d]

Each result comes with an error scale A: the same expression with every factor replaced by its absolute value, i.e. the
float64 abs-sum that bounds the rounding error of the kernels' fp32 accumulations (|fp32 result - exact| <= n u A for a
sum evaluated with n roundings of unit round-off u).  The tests compare per element, |got - ref| <= tau * A.

Everything runs in float64 on the device of the given tensors, one image at a time (so that the 16 x 16384-pixel case
needs a few GB on a GPU, and small shapes can run on the CPU).  A float64 G skips the bf16 rounding of the operand: the
exact algebra, which the host tests compare with torch.autograd.

``check_bound`` asserts a kernel's result against a reference and its A; test_gpu_k1b_exact.py and
test_gpu_step_routes.py share it."""
from __future__ import annotations

from typing import NamedTuple, Optional

import torch
from torch import Tensor

# check_bound's per-element bound |got - ref| <= TAU * A: 2^7 x the fp32 unit round-off (test_gpu_k1b_exact.py says why)
TAU = 2.0 ** -16
BF16_OUT = 2.0 ** -8            # output rounding of a bf16 grad_v: the bf16 unit round-off (half an ulp <= 2^-8 |x|)


class K1bReference(NamedTuple):
    grad_v: Tensor      # float64 [B, hw, D]
    grad_v_A: Tensor    # float64 [B, hw, D] error scale
    grad_t: Tensor      # float64 [n_sets, C, D]
    grad_t_A: Tensor    # float64 [n_sets, C, D] error scale


def _planes(G: Tensor, B: int, C: int, hw: int) -> Tensor:
    """G as [B, C, hw]: an fp32 / float64 [B, C, h, w] gradient, or the bf16 [B, C_pad, hw] operand (pad rows dropped)."""
    return G.reshape(B, G.shape[1], hw)[:, :C]


def gemm_operand(G: Tensor, C: int, inv_v: Optional[Tensor] = None) -> Tensor:
    """The operand of the two backward GEMMs as float64 [B, C, hw]: bf16_rn(G) for fp32 G, bf16_rn(fp32(G * inv_v)) with
    inv_v given (LC2IS_BWD_RAW_V), the values of a bf16 G, and G (times inv_v) unrounded for a float64 G."""
    B = G.shape[0]
    hw = G[0, 0].numel()
    g = _planes(G, B, C, hw)
    if inv_v is not None:
        if g.dtype == torch.bfloat16:
            raise ValueError("LC2IS_BWD_RAW_V takes an fp32 gradient")
        g = g * inv_v.reshape(B, 1, hw).to(g.dtype)        # fp32 * fp32 rounds once, like the kernel's FMUL
    if g.dtype == torch.float32:
        g = g.to(torch.bfloat16)
    return g.double()


def projections(G: Tensor, logits: Tensor, n_sets: int):
    """(r [B, hw], rt [n_sets, C]) and their abs-sums, in float64, from the unrounded G."""
    B, C = logits.shape[:2]
    hw = logits[0, 0].numel()
    p = _planes(G, B, C, hw).double() * logits.reshape(B, C, hw).double()
    r, r_abs = p.sum(1), p.abs().sum(1)
    rt = p.sum(2) if n_sets > 1 else p.sum((0, 2)).unsqueeze(0)
    rt_abs = p.abs().sum(2) if n_sets > 1 else p.abs().sum((0, 2)).unsqueeze(0)
    return r, r_abs, rt, rt_abs


def k1b_reference(G: Tensor, logits: Tensor, v: Tensor, inv_v: Tensor, t_hat: Tensor, inv_t: Optional[Tensor], *,
                  normalize: bool = True, scale: float = 1.0, g: float = 1.0, raw_v: bool = False) -> K1bReference:
    """G: fp32 [B,C,h,w] | bf16 [B,C_pad,hw] | float64 [B,C,h,w];  logits fp32 [B,C,h,w] (the forward's);  v: v_hat bf16
    [B*hw, D] (or the raw bf16 V with raw_v);  inv_v [B*hw];  t_hat [n_sets, C_pad >= C, D];  inv_t [n_sets, C]
    (ignored unless normalize);  scale = logit_scale s;  g = the upstream scalar (the value behind d_grad_scale)."""
    B, C = logits.shape[:2]
    hw = logits[0, 0].numel()
    n_sets, _, D = t_hat.shape
    if raw_v and not normalize:
        raise ValueError("LC2IS_BWD_RAW_V needs normalize")
    f64 = torch.float64
    V = v.reshape(B, hw, D)
    inv = inv_v.reshape(B, hw).double()
    T = t_hat[:, :C].double()
    s, gd = float(scale), float(g)
    sg, sg_abs = s * gd, abs(s * gd)
    gv = torch.empty(B, hw, D, dtype=f64, device=V.device)
    gv_A = torch.empty_like(gv)
    st = torch.zeros(n_sets, C, D, dtype=f64, device=V.device)      # sum_m Gb v
    st_abs = torch.zeros_like(st)
    rt = torch.zeros(n_sets, C, dtype=f64, device=V.device)
    rt_abs = torch.zeros_like(rt)
    for b in range(B):
        k = b if n_sets > 1 else 0
        Gb = gemm_operand(G[b:b + 1], C, inv_v.reshape(B, hw)[b] if raw_v else None)[0]      # [C, hw]
        r, r_abs, rtb, rtb_abs = projections(G[b:b + 1], logits[b:b + 1], 1)
        r, r_abs = r[0], r_abs[0]
        rt[k] += rtb[0]
        rt_abs[k] += rtb_abs[0]
        Vb = V[b].double()                                                               # [hw, D]
        acc = Gb.t() @ T[k]                                                              # [hw, D]
        acc_abs = Gb.abs().t() @ T[k].abs()
        if not normalize:
            gv[b], gv_A[b] = sg * acc, sg_abs * acc_abs
        elif raw_v:
            f = gd * inv[b] * inv[b]
            gv[b] = sg * acc - Vb * (f * r).unsqueeze(1)
            gv_A[b] = sg_abs * acc_abs + Vb.abs() * (abs(gd) * inv[b] * inv[b] * r_abs).unsqueeze(1)
        else:
            ib = inv[b].unsqueeze(1)
            gv[b] = ib * (sg * acc - Vb * (gd * r).unsqueeze(1))
            gv_A[b] = ib.abs() * (sg_abs * acc_abs + Vb.abs() * (abs(gd) * r_abs).unsqueeze(1))
        st[k] += Gb @ Vb
        st_abs[k] += Gb.abs() @ Vb.abs()
    if normalize:
        it = inv_t.reshape(n_sets, C, 1).double()
        gt = it * gd * (s * st - T * rt.unsqueeze(2))
        gt_A = it.abs() * abs(gd) * (abs(s) * st_abs + T.abs() * rt_abs.unsqueeze(2))
    else:
        gt, gt_A = sg * st, sg_abs * st_abs
    return K1bReference(gv, gv_A, gt, gt_A)


def check_bound(name, got, ref, A, bf16_out=False, base=None, tau=TAU):
    """|got - (base + ref)| <= tau * A (+ BF16_OUT |ref|) per element, asserted on the maxima of [128 rows x 64 channels]
    blocks of the [images | sets, rows, D] (or [rows, D]) tensors; the last blocks may be partial.
    -> (worst |got - ref| / A, worst share of the bound used)."""
    got = got.to(ref.device).double().reshape(ref.shape)
    if base is not None:
        got = got - base.to(ref.device).double().reshape(ref.shape)
    err = (got - ref).abs()
    bound = tau * A + (BF16_OUT * ref.abs() if bf16_out else 0.0)
    if base is not None:                           # one fp32 rounding of base + result
        bound = bound + 2.0 ** -24 * (base.to(ref.device).double().reshape(ref.shape) + ref).abs()
    use = torch.where(err == 0, torch.zeros_like(err), err / bound)          # NaN (unwritten) stays NaN
    if use.dim() == 2:
        use = use.unsqueeze(0)
    X, R, D = use.shape
    Rp, Dp = -(-R // 128) * 128, -(-D // 64) * 64
    blocks = torch.nn.functional.pad(use, (0, Dp - D, 0, Rp - R)).view(X, Rp // 128, 128, Dp // 64, 64).amax(dim=(2, 4))
    bad = ~(blocks <= 1)
    if bool(bad.any()):
        worst = torch.nan_to_num(blocks, nan=float("inf")).flatten().argmax()
        x, rt, cb = (int(i) for i in torch.unravel_index(worst, blocks.shape))
        raise AssertionError(f"{name}: {int(bad.sum())} of {blocks.numel()} [128 x 64] blocks exceed the bound; worst: "
                             f"image/set {x}, rows {128 * rt}.., channels {64 * cb}.. at {float(blocks[x, rt, cb]):.3g} "
                             f"x the bound (worst |got-ref|/A overall {float((err / A).nan_to_num(float('inf')).max()):.3g})")
    pos = A > 0
    return float((err[pos] / A[pos]).max()) if bool(pos.any()) else 0.0, float(blocks.max())
