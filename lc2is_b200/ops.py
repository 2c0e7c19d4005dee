"""Tensor-level wrappers over the C ABI.  PyTorch is plumbing only here: it owns device
memory and the current stream; all arithmetic happens in ``liblc2is_b200.so``."""
from __future__ import annotations

from typing import Optional, Tuple

import torch
from torch import Tensor

from . import _lib
from ._lib import BF16, BICUBIC, BILINEAR, F32, check, lib, ptr, stream_ptr

_MODE = {"bilinear": BILINEAR, "bicubic": BICUBIC}


def _req(t: Tensor, dtype, name: str) -> Tensor:
    if not t.is_cuda:
        raise _lib.Lc2isError(f"{name} must be a CUDA tensor (lc2is_b200 has no CPU fallback)")
    if t.dtype != dtype:
        raise _lib.Lc2isError(f"{name} must be {dtype}, got {t.dtype}")
    return t.contiguous()


def _dt(t: Tensor) -> int:
    if t.dtype == torch.float32:
        return F32
    if t.dtype == torch.bfloat16:
        return BF16
    raise _lib.Lc2isError(f"unsupported dtype {t.dtype} (float32 / bfloat16 only)")


def _aligned(t: Tensor) -> Tensor:
    """t, or a copy of it when it does not start on a 16-byte boundary: the projection entries read and write their
    tensors with 16-byte vectors and TMA, and a view into a larger buffer (a bias sliced out of a flat parameter
    buffer, say) may start anywhere."""
    return t if t.data_ptr() % 16 == 0 else t.clone()


# ---- K0 -----------------------------------------------------------------------------------
def proto_normalize(t: Tensor, normalize: bool = True) -> Tuple[Tensor, Tensor]:
    """t [C,D] or [n_sets,C,D] fp32 -> (t_hat bf16 [n_sets,C_pad,D], inv_norm fp32 [n_sets,C])."""
    t = _req(t, torch.float32, "t")
    if t.dim() == 2:
        t = t.unsqueeze(0)
    n_sets, C, D = t.shape
    Cp = _lib.class_pad(C)
    t_hat = torch.empty(n_sets, Cp, D, dtype=torch.bfloat16, device=t.device)
    inv = torch.empty(n_sets, C, dtype=torch.float32, device=t.device)
    check(lib.lc2is_proto_normalize(ptr(t), n_sets, C, D, int(normalize), ptr(t_hat), ptr(inv), stream_ptr()),
          "lc2is_proto_normalize")
    return t_hat, inv


# ---- TextToPatch projection ------------------------------------------------------------------
def linear_fwd(x: Tensor, weight: Tensor, bias: Optional[Tensor] = None, out_dtype=torch.bfloat16) -> Tensor:
    """y = x W^T + b on the tcgen05 pipeline.  x [M,K] bf16, weight [N,K] bf16 (nn.Linear layout), bias fp32 [N]."""
    x = _aligned(_req(x, torch.bfloat16, "x"))
    weight = _aligned(_req(weight, torch.bfloat16, "weight"))
    M, K = x.shape
    N = weight.shape[0]
    if bias is not None:
        bias = _aligned(_req(bias, torch.float32, "bias"))
    y = torch.empty(M, N, dtype=out_dtype, device=x.device)
    check(lib.lc2is_linear_fwd(ptr(x), ptr(weight), ptr(bias), M, N, K, ptr(y), _dt(y), stream_ptr()), "lc2is_linear_fwd")
    return y


def bicubic4_tokens_fwd(x: Tensor, hw_shape: Tuple[int, int], out_dtype=torch.bfloat16) -> Tensor:
    """x [B, h*w, C] fp32/bf16 (token-major) -> [B, 16*h*w, C]: bicubic x4 of model.py:42-44 without the layout changes."""
    if not x.is_cuda:
        raise _lib.Lc2isError("x must be a CUDA tensor (lc2is_b200 has no CPU fallback)")
    if x.dtype not in (torch.float32, torch.bfloat16):
        x = x.float()
    x = x.contiguous()
    B, P, C = x.shape
    h, w = hw_shape
    assert h * w == P
    y = torch.empty(B, 16 * P, C, dtype=out_dtype, device=x.device)
    check(lib.lc2is_bicubic4_tokens_fwd(ptr(x), _dt(x), B, h, w, C, ptr(y), _dt(y), stream_ptr()), "lc2is_bicubic4_tokens_fwd")
    return y


def bicubic4_tokens_bwd(gy: Tensor, hw_shape: Tuple[int, int], out_dtype=torch.float32) -> Tensor:
    """gy [B, 16*h*w, C] -> gx [B, h*w, C]: the transpose of bicubic4_tokens_fwd (two gather passes)."""
    if gy.dtype not in (torch.float32, torch.bfloat16):
        gy = gy.float()
    gy = gy.contiguous()
    B, P16, C = gy.shape
    h, w = hw_shape
    assert 16 * h * w == P16
    gx = torch.empty(B, h * w, C, dtype=out_dtype, device=gy.device)
    ws = torch.empty(int(lib.lc2is_bicubic4_tokens_bwd_workspace(B, h, w, C)), dtype=torch.uint8, device=gy.device)
    check(lib.lc2is_bicubic4_tokens_bwd(ptr(gy), _dt(gy), B, h, w, C, ptr(gx), _dt(gx), ptr(ws), stream_ptr()),
          "lc2is_bicubic4_tokens_bwd")
    return gx


def linear_bwd(gy: Tensor, x: Tensor, weight: Tensor, need_gx: bool = True, need_gw: bool = True, need_gb: bool = True,
               gx_dtype=torch.bfloat16, gw: Optional[Tensor] = None, gb: Optional[Tensor] = None):
    """Backward of y = x W^T + b on tcgen05 (lc2is_linear_bwd).  gy [M,N], x [M,K], weight [N,K]: bf16.
    -> (gx [M,K] gx_dtype | None, gw fp32 [N,K] | None, gb fp32 [N] | None); `gw` / `gb` given: accumulated into
    (a `gw` that is not contiguous or not 16-byte aligned through an aligned copy, written back)."""
    gy = _aligned(_req(gy, torch.bfloat16, "gy"))
    x = _aligned(_req(x, torch.bfloat16, "x"))
    weight = _req(weight, torch.bfloat16, "weight")
    M, N = gy.shape
    K = x.shape[1]
    dev = gy.device
    gx = torch.empty(M, K, dtype=gx_dtype, device=dev) if need_gx else None
    gw_caller = None
    if need_gw and gw is None:
        gw = torch.zeros(N, K, dtype=torch.float32, device=dev)
    elif need_gw and (gw.data_ptr() % 16 or not gw.is_contiguous()):
        gw_caller, gw = gw, gw.clone(memory_format=torch.contiguous_format)
    if need_gb and gb is None:
        gb = torch.zeros(N, dtype=torch.float32, device=dev)
    ws = torch.empty(int(lib.lc2is_linear_bwd_workspace(N, K)), dtype=torch.uint8, device=dev)
    check(lib.lc2is_linear_bwd(ptr(gy), ptr(x), ptr(weight), M, N, K, ptr(gx), _dt(gx) if need_gx else 0,
                               ptr(gw) if need_gw else None, ptr(gb) if need_gb else None, ptr(ws), stream_ptr()),
          "lc2is_linear_bwd")
    if gw_caller is not None:
        gw = gw_caller.copy_(gw)
    return gx, (gw if need_gw else None), (gb if need_gb else None)


# ---- K1 -----------------------------------------------------------------------------------
def cosine_logits_fwd(v: Tensor, t_hat: Tensor, C: int, hw_shape: Tuple[int, int], normalize: bool = True,
                      logit_scale: float = 1.0, fuse_norm: bool = False) -> Tuple[Tensor, Optional[Tensor], Tensor]:
    """v [B,hw,D] fp32/bf16, t_hat from K0 -> (logits fp32 [B,C,h,w], v_hat bf16 [B*hw,D], inv_norm_v).
    fuse_norm (bf16 v, normalize): the row normalisation runs inside the GEMM on the raw V; v_hat is None and the
    backward takes v itself (``cosine_logits_bwd(..., raw_v=True)``)."""
    if not v.is_cuda:
        raise _lib.Lc2isError("v must be a CUDA tensor (lc2is_b200 has no CPU fallback)")
    v = v.contiguous()
    B, hw, D = v.shape
    h, w = hw_shape
    assert h * w == hw
    n_sets = t_hat.shape[0]
    if fuse_norm and not (v.dtype == torch.bfloat16 and normalize):
        raise _lib.Lc2isError("fuse_norm needs bf16 v and normalize=True")
    v_hat = None if fuse_norm else torch.empty(B * hw, D, dtype=torch.bfloat16, device=v.device)
    inv_v = torch.empty(B * hw, dtype=torch.float32, device=v.device)
    logits = torch.empty(B, C, h, w, dtype=torch.float32, device=v.device)
    check(lib.lc2is_cosine_logits_fwd(ptr(v), _dt(v), B, hw, D, ptr(t_hat), n_sets, C, int(normalize),
                                      float(logit_scale), ptr(v_hat), ptr(inv_v), ptr(logits), stream_ptr()),
          "lc2is_cosine_logits_fwd")
    return logits, v_hat, inv_v


def grad_to_bf16(grad: Tensor) -> Tensor:
    """fp32 [B,C,h,w] -> bf16 [B,C_pad,h*w]."""
    grad = _req(grad, torch.float32, "grad")
    B, C = grad.shape[:2]
    hw = grad[0, 0].numel()
    out = torch.empty(B, _lib.class_pad(C), hw, dtype=torch.bfloat16, device=grad.device)
    check(lib.lc2is_grad_to_bf16(ptr(grad), B, C, hw, ptr(out), stream_ptr()), "lc2is_grad_to_bf16")
    return out


def cosine_logits_bwd(grad: Tensor, logits: Tensor, v_hat: Tensor, inv_v: Tensor, t_hat: Tensor,
                      inv_t: Tensor, C: int, normalize: bool = True, logit_scale: float = 1.0,
                      grad_scale: Optional[Tensor] = None, grad_v_dtype=torch.float32,
                      grad_t: Optional[Tensor] = None, raw_v: bool = False) -> Tuple[Tensor, Tensor]:
    """grad: dL/dlogits, bf16 [B,C_pad,hw] or fp32 [B,C,h,w] (converted inside the projection pass).
    raw_v: `v_hat` is the raw bf16 V of a fuse_norm forward (fp32 grad only).
    -> (grad_v [B,hw,D], grad_t fp32 [n_sets,C,D]); grad_t is accumulated into if given."""
    B = logits.shape[0]
    hw = logits[0, 0].numel()
    D = v_hat.shape[-1]
    n_sets = t_hat.shape[0]
    dev = logits.device
    grad = grad.contiguous()
    grad_v = torch.empty(B, hw, D, dtype=grad_v_dtype, device=dev)
    if grad_t is None:
        grad_t = torch.zeros(n_sets, C, D, dtype=torch.float32, device=dev)
    nbytes = int(lib.lc2is_cosine_logits_bwd_workspace(B, hw, D, n_sets, C))
    ws = torch.empty(max(nbytes, 256), dtype=torch.uint8, device=dev)
    check(lib.lc2is_cosine_logits_bwd_ex(ptr(grad), _dt(grad), ptr(logits), ptr(v_hat), ptr(inv_v), ptr(t_hat), ptr(inv_t),
                                         B, hw, D, n_sets, C, int(normalize), float(logit_scale), ptr(grad_scale),
                                         ptr(grad_v), _dt(grad_v), ptr(grad_t), ptr(ws), stream_ptr(),
                                         _lib.BWD_RAW_V if raw_v else 0),
          "lc2is_cosine_logits_bwd")
    return grad_v, grad_t


# ---- K2 -----------------------------------------------------------------------------------
def count_valid(labels: Tensor, n_classes: int, ignore_index: int, out: Optional[Tensor] = None) -> Tensor:
    """#{labels in [0, n_classes) and != ignore_index}: the 'mean' denominator of every CE route."""
    labels = _req(labels, torch.int64, "labels")
    if out is None:
        out = torch.zeros(1, dtype=torch.int64, device=labels.device)
    check(lib.lc2is_count_valid(ptr(labels), labels.numel(), int(n_classes), int(ignore_index), ptr(out), stream_ptr()),
          "lc2is_count_valid")
    return out


def mean_scale(n_valid: Tensor, mult: float = 1.0) -> Tensor:
    out = torch.empty(1, dtype=torch.float32, device=n_valid.device)
    check(lib.lc2is_mean_scale(ptr(n_valid), float(mult), ptr(out), stream_ptr()), "lc2is_mean_scale")
    return out


def finalize_loss(loss_sum: Tensor, n_valid: Tensor) -> Tensor:
    out = torch.empty(1, dtype=torch.float32, device=n_valid.device)
    check(lib.lc2is_finalize_loss(ptr(loss_sum), ptr(n_valid), ptr(out), stream_ptr()), "lc2is_finalize_loss")
    return out


def ce_weight_sum(labels: Tensor, n_classes: int, ignore_index: int, weight: Optional[Tensor] = None,
                  out: Optional[Tensor] = None) -> Tensor:
    """sum of weight[label] over the counted labels (in [0, n_classes), != ignore_index), double[1] on the device: the
    'mean' denominator of the weighted cross-entropy.  weight=None counts them."""
    labels = _req(labels, torch.int64, "labels")
    if weight is not None:
        weight = _class_weight(weight, n_classes)
    if out is None:
        out = torch.zeros(1, dtype=torch.float64, device=labels.device)
    check(lib.lc2is_ce_weight_sum(ptr(labels), labels.numel(), int(n_classes), int(ignore_index), ptr(weight), ptr(out),
                                  stream_ptr()), "lc2is_ce_weight_sum")
    return out


def weighted_mean_loss(loss_sum: Tensor, wsum: Tensor) -> Tensor:
    """loss_sum / wsum as fp32 [1] on the device; NaN when wsum == 0 - torch divides the target and the smoothing parts
    separately, so counted pixels that all have weight 0 give 0/0 even when the smoothing sum is not 0."""
    return torch.where(wsum != 0, loss_sum / wsum, torch.full_like(wsum, float("nan"))).float()


def _class_weight(weight: Tensor, n_classes: int) -> Tensor:
    weight = _req(weight, torch.float32, "weight")
    if weight.dim() != 1 or weight.numel() != n_classes:
        raise _lib.Lc2isError(f"weight must have shape [{n_classes}], got {list(weight.shape)}")
    return weight


def upsample_ce(low: Tensor, labels: Tensor, ignore_index: int = -100, grad_scale: Optional[Tensor] = None,
                want_grad: bool = True, want_bf16: bool = False,
                loss_sum: Optional[Tensor] = None, weight: Optional[Tensor] = None,
                label_smoothing: float = 0.0) -> Tuple[Tensor, Optional[Tensor], Optional[Tensor]]:
    """low [B,C,h,w] fp32, labels [B,H,W] int64 -> (loss_sum double[1], grad_low fp32, grad_low_bf16).
    weight (fp32 [C] on the device) / label_smoothing: the weighted form (lc2is_upsample_ce_fwd_bwd_ex); loss_sum is then
    the sum of the per-pixel losses, to be divided by ce_weight_sum for reduction='mean'."""
    low = _req(low, torch.float32, "low")
    labels = _req(labels, torch.int64, "labels")
    B, C, h, w = low.shape
    Bl, H, W = labels.shape
    if Bl != B:
        raise _lib.Lc2isError("batch mismatch between logits and labels")
    if weight is not None:
        weight = _class_weight(weight, C)
    if loss_sum is None:
        loss_sum = torch.zeros(1, dtype=torch.float64, device=low.device)
    grad = torch.empty_like(low) if (want_grad or want_bf16) else None
    gbf = torch.empty(B, _lib.class_pad(C), h * w, dtype=torch.bfloat16, device=low.device) if want_bf16 else None
    check(lib.lc2is_upsample_ce_fwd_bwd_ex(ptr(low), ptr(labels), B, C, h, w, H, W, int(ignore_index), ptr(weight),
                                           float(label_smoothing), ptr(grad_scale), ptr(loss_sum), ptr(grad), ptr(gbf),
                                           stream_ptr()),
          "lc2is_upsample_ce_fwd_bwd_ex")
    return loss_sum, grad, gbf


def ce_split_supported(h: int, w: int, H: int, W: int) -> bool:
    return bool(lib.lc2is_ce_split_supported(h, w, H, W))


def upsample_ce_split(low: Tensor, labels: Tensor, ignore_index: int = -100, want_grad: bool = True):
    """Split K2 (scale 8 / 16): label prepass + packed-label strip kernel.
    -> (loss_sum double[1], n_valid int64[1], grad_low fp32 UNSCALED | None, labels_packed uint16 [B,H,W])."""
    low = _req(low, torch.float32, "low")
    labels = _req(labels, torch.int64, "labels")
    B, C, h, w = low.shape
    _, H, W = labels.shape
    dev = low.device
    loss_sum = torch.zeros(1, dtype=torch.float64, device=dev)
    n_valid = torch.zeros(1, dtype=torch.int64, device=dev)
    grad = torch.zeros_like(low) if want_grad else None
    packed = torch.empty(B, H, W, dtype=torch.uint16, device=dev)
    st = stream_ptr()
    check(lib.lc2is_ce_labels_prepass(ptr(labels), B, C, h, w, H, W, int(ignore_index), ptr(packed),
                                      ptr(n_valid), ptr(grad), st), "lc2is_ce_labels_prepass")
    check(lib.lc2is_upsample_ce_packed(ptr(low), ptr(packed), B, C, h, w, H, W, ptr(loss_sum), ptr(grad), st),
          "lc2is_upsample_ce_packed")
    return loss_sum, n_valid, grad, packed


# ---- K3 -----------------------------------------------------------------------------------
def argmax_confmat(logits: Tensor, labels: Tensor, confmat: Optional[Tensor] = None, per_image: bool = False,
                   want_pred: bool = False, size: Optional[Tuple[int, int]] = None, mode: Optional[str] = None):
    """logits [N,C,h,w] (fp32/bf16), labels [N,lh,lw] int64.
    size=None: logits are at mask resolution.  size=(H,W)+mode: fused bilinear/bicubic resize.
    Returns (confmat int64 [C,C] (accumulated), per_image int64 [N,3,C] | None, pred int64 [N,H,W] | None)."""
    if not logits.is_cuda:
        raise _lib.Lc2isError("logits must be a CUDA tensor (lc2is_b200 has no CPU fallback)")
    logits = logits.contiguous()
    labels = _req(labels, torch.int64, "labels")
    N, C, h, w = logits.shape
    Nl, lh, lw = labels.shape
    if Nl != N:
        raise _lib.Lc2isError("batch mismatch between logits and labels")
    dev = logits.device
    H, W = (h, w) if size is None else (int(size[0]), int(size[1]))
    if confmat is None:
        confmat = torch.zeros(C, C, dtype=torch.int64, device=dev)
    pi = torch.zeros(N, 3, C, dtype=torch.int64, device=dev) if per_image else None
    pred = torch.empty(N, H, W, dtype=torch.int64, device=dev) if want_pred else None
    if size is None:
        check(lib.lc2is_argmax_confmat(ptr(logits), _dt(logits), N, C, H, W, ptr(labels), lh, lw, ptr(confmat),
                                       ptr(pi), ptr(pred), stream_ptr()), "lc2is_argmax_confmat")
    else:
        logits = _req(logits, torch.float32, "logits")
        check(lib.lc2is_argmax_confmat_lowres(ptr(logits), N, C, h, w, H, W, _MODE[mode], ptr(labels), lh, lw,
                                              ptr(confmat), ptr(pi), ptr(pred), stream_ptr()),
              "lc2is_argmax_confmat_lowres")
    return confmat, pi, pred


def argmax_confmat_packed(low: Tensor, labels_packed: Tensor, size: Tuple[int, int], confmat: Optional[Tensor] = None,
                          per_image: bool = False, want_pred: bool = False):
    """Fused bilinear resize + argmax + confusion matrix from the packed labels of the CE label prepass."""
    low = _req(low, torch.float32, "low")
    N, C, h, w = low.shape
    H, W = int(size[0]), int(size[1])
    dev = low.device
    if confmat is None:
        confmat = torch.zeros(C, C, dtype=torch.int64, device=dev)
    pi = torch.zeros(N, 3, C, dtype=torch.int64, device=dev) if per_image else None
    pred = torch.empty(N, H, W, dtype=torch.int64, device=dev) if want_pred else None
    check(lib.lc2is_argmax_confmat_lowres_packed(ptr(low), N, C, h, w, H, W, ptr(labels_packed), ptr(confmat), ptr(pi),
                                                 ptr(pred), stream_ptr()), "lc2is_argmax_confmat_lowres_packed")
    return confmat, pi, pred


def ragged_descriptors(sizes) -> Tuple[Tensor, int, int]:
    """The descriptor table of lc2is_argmax_confmat_ragged for images of sizes [(H_i, W_i)]: int64 [N,4] rows
    {element offset, H, W, first tile} (a CPU tensor), the total number of tiles and of elements."""
    rows, off, tile = [], 0, 0
    for H, W in sizes:
        H, W = int(H), int(W)
        rows.append((off, H, W, tile))
        off += H * W
        tile += int(lib.lc2is_ragged_tiles(H, W))
    return torch.tensor(rows, dtype=torch.int64).reshape(-1, 4), tile, off


def argmax_confmat_ragged(low: Tensor, sizes, labels_flat: Optional[Tensor] = None, mode: str = "bicubic",
                          confmat: Optional[Tensor] = None, per_image: bool = True, want_pred: bool = False):
    """ONE launch for a ragged batch: low [N,C,h,w] fp32 (CUDA); image i is resized to sizes[i] = (H_i, W_i), argmaxed
    and compared with labels_flat (int64, the images' label maps flattened and concatenated; None = masks only).
    -> (confmat | None, per_image int64 [N,3,C] | None, pred_flat int64 | None, desc (CPU int64 [N,4]))."""
    low = _req(low, torch.float32, "low")
    N, C, h, w = low.shape
    desc, n_tiles, n_elem = ragged_descriptors(sizes)
    if desc.shape[0] != N:
        raise _lib.Lc2isError("one size per image")
    dev = low.device
    d_desc = desc.to(dev, non_blocking=True)
    if labels_flat is not None:
        labels_flat = _req(labels_flat, torch.int64, "labels_flat")
        if labels_flat.numel() != n_elem:
            raise _lib.Lc2isError(f"labels_flat has {labels_flat.numel()} elements, the sizes add up to {n_elem}")
    else:
        per_image, confmat = False, None
    pi = torch.zeros(N, 3, C, dtype=torch.int64, device=dev) if per_image else None
    pred = torch.empty(n_elem, dtype=torch.int64, device=dev) if want_pred else None
    check(lib.lc2is_argmax_confmat_ragged(ptr(low), N, C, h, w, _MODE[mode], ptr(d_desc), n_tiles, ptr(labels_flat),
                                          ptr(confmat), ptr(pi), ptr(pred), stream_ptr()), "lc2is_argmax_confmat_ragged")
    return confmat, pi, pred, desc


def pack_labels(labels: Tensor, C: int, ignore_index: int, n_valid: Optional[Tensor] = None):
    """int64 labels -> (packed uint16 of the same shape, n_valid int64[1] accumulated)."""
    labels = _req(labels, torch.int64, "labels")
    packed = torch.empty(labels.shape, dtype=torch.uint16, device=labels.device)
    if n_valid is None:
        n_valid = torch.zeros(1, dtype=torch.int64, device=labels.device)
    check(lib.lc2is_pack_labels(ptr(labels), labels.numel(), C, int(ignore_index), ptr(packed), ptr(n_valid), stream_ptr()),
          "lc2is_pack_labels")
    return packed, n_valid


def ce_argmax_fused(low: Tensor, labels_packed: Tensor, size: Tuple[int, int], loss_sum: Tensor, grad: Optional[Tensor],
                    confmat: Optional[Tensor] = None, per_image: bool = False, want_pred: bool = False,
                    onehot: bool = False, n_valid: Optional[Tensor] = None):
    """Fused K2 (split form) + K3 for the x16 geometry: accumulates into loss_sum / grad (un-scaled softmax term) /
    confmat.  -> (confmat, per_image | None, pred | None)."""
    low = _req(low, torch.float32, "low")
    N, C, h, w = low.shape
    H, W = int(size[0]), int(size[1])
    dev = low.device
    if confmat is None:
        confmat = torch.zeros(C, C, dtype=torch.int64, device=dev)
    pi = torch.zeros(N, 3, C, dtype=torch.int64, device=dev) if per_image else None
    pred = torch.empty(N, H, W, dtype=torch.int64, device=dev) if want_pred else None
    check(lib.lc2is_ce_argmax_fused_packed(ptr(low), ptr(labels_packed), N, C, h, w, H, W, ptr(loss_sum), ptr(grad),
                                           int(onehot), ptr(n_valid), ptr(confmat), ptr(pi), ptr(pred), stream_ptr()),
          "lc2is_ce_argmax_fused_packed")
    return confmat, pi, pred


def contrastive_fwd(outputs: Tensor, labels: Tensor, ignore_index: int):
    """K4 forward (loss.py:39-64).  outputs [B, h*w, C] fp32, labels [B, h, w] int64.
    -> (loss_sums double[2] = {visual sum, textual sum}, counts int64[2] = {counted pixels, out-of-range labels},
        col_lse [B,w,C], col_adj [B,w,C] = col_lse - ln(#rows of the column labelled c)) - no host sync."""
    outputs = _req(outputs, torch.float32, "outputs")
    labels = _req(labels, torch.int64, "labels")
    B, hw, C = outputs.shape
    _, h, w = labels.shape
    if labels.shape[0] != B or h * w != hw:
        raise ValueError(f"labels {tuple(labels.shape)} do not match outputs {tuple(outputs.shape)}")
    dev = outputs.device
    col = torch.empty(2, B, w, C, dtype=torch.float32, device=dev)
    acc = torch.zeros(4, dtype=torch.int64, device=dev)             # one memset: {sums (as double), counts}
    sums, counts = acc[:2].view(torch.float64), acc[2:]
    check(lib.lc2is_contrastive_fwd(ptr(outputs), ptr(labels), B, h, w, C, int(ignore_index), ptr(col[0]), ptr(col[1]),
                                    ptr(sums), ptr(counts), stream_ptr()), "lc2is_contrastive_fwd")
    return sums, counts, col[0], col[1]


def contrastive_bwd(outputs: Tensor, labels: Tensor, ignore_index: int, col_lse: Tensor, col_adj: Tensor,
                    coef: Tensor) -> Tensor:
    """K4 backward: coef float32[2] (device) = {c_visual, c_textual}; -> grad [B, h*w, C] fp32."""
    outputs = _req(outputs, torch.float32, "outputs")
    labels = _req(labels, torch.int64, "labels")
    coef = _req(coef, torch.float32, "coef")
    B, hw, C = outputs.shape
    _, h, w = labels.shape
    grad = torch.empty_like(outputs)
    check(lib.lc2is_contrastive_bwd(ptr(outputs), ptr(labels), B, h, w, C, int(ignore_index), ptr(col_lse), ptr(col_adj),
                                    ptr(coef), ptr(grad), stream_ptr()), "lc2is_contrastive_bwd")
    return grad


def expand_labels(labels8: Tensor, C: int, ignore_index: int, n_valid: Optional[Tensor] = None) -> Tensor:
    """One-byte host label form (lc2is_pack_labels_host for C <= 254) -> packed uint16 of the same shape;
    n_valid (int64[1]) accumulates the counted labels when given."""
    labels8 = _req(labels8, torch.uint8, "labels8")
    packed = torch.empty(labels8.shape, dtype=torch.uint16, device=labels8.device)
    check(lib.lc2is_expand_labels(ptr(labels8), labels8.numel(), C, int(ignore_index), ptr(packed), ptr(n_valid),
                                  stream_ptr()), "lc2is_expand_labels")
    return packed
