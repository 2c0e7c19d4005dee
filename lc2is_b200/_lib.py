"""ctypes binding of ``liblc2is_b200.so`` (the C ABI in ``include/lc2is_b200.h``).

The library is built in-tree by ``__graft_entry__.build()`` / ``make -C lc2is_b200/csrc``.
There is no fallback: if the shared object is missing the import of any compute module
raises, and every compute call raises :class:`Lc2isError` when no B200 is present.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_float, c_int, c_int64, c_void_p, POINTER

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "liblc2is_b200.so")

F32, BF16 = 0, 1
BILINEAR, BICUBIC = 0, 1
BWD_REUSE_PREP, BWD_RAW_V, BWD_WS_ZEROED = 1, 2, 4      # flags of lc2is_cosine_logits_bwd_ex


class Lc2isError(RuntimeError):
    pass


def _load() -> ctypes.CDLL:
    if not os.path.exists(LIB_PATH):
        raise Lc2isError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -C lc2is_b200/csrc`.  lc2is_b200 has no CPU / PyTorch fallback.")
    return ctypes.CDLL(LIB_PATH)


_lib = _load()

# name -> (restype, argtypes); must list every symbol include/lc2is_b200.h declares
_p = c_void_p
SIGNATURES = {
    "lc2is_last_error": (c_char_p, []),
    "lc2is_abi_version": (c_int, []),
    "lc2is_launch_count": (c_int64, []),
    "lc2is_class_pad": (c_int, [c_int]),
    "lc2is_proto_normalize": (c_int, [_p, c_int, c_int, c_int, c_int, _p, _p, _p]),
    "lc2is_cosine_logits_fwd": (c_int, [_p, c_int, c_int, c_int, c_int, _p, c_int, c_int, c_int, c_float,
                                        _p, _p, _p, _p]),
    "lc2is_linear_fwd": (c_int, [_p, _p, _p, c_int64, c_int, c_int, _p, c_int, _p]),
    "lc2is_bicubic4_tokens_fwd": (c_int, [_p, c_int, c_int, c_int, c_int, c_int, _p, c_int, _p]),
    "lc2is_bicubic4_tokens_bwd_workspace": (c_int64, [c_int, c_int, c_int, c_int]),
    "lc2is_bicubic4_tokens_bwd": (c_int, [_p, c_int, c_int, c_int, c_int, c_int, _p, c_int, _p, _p]),
    "lc2is_linear_bwd_workspace": (c_int64, [c_int, c_int]),
    "lc2is_linear_bwd": (c_int, [_p, _p, _p, c_int64, c_int, c_int, _p, c_int, _p, _p, _p, _p]),
    "lc2is_cosine_logits_bwd_workspace": (c_int64, [c_int, c_int, c_int, c_int, c_int]),
    "lc2is_cosine_logits_bwd_workspace_zeroed": (c_int64, [c_int, c_int, c_int, c_int, c_int]),
    "lc2is_cosine_logits_bwd": (c_int, [_p, c_int, _p, _p, _p, _p, _p, c_int, c_int, c_int, c_int, c_int, c_int,
                                        c_float, _p, _p, c_int, _p, _p, _p]),
    "lc2is_cosine_logits_bwd_ex": (c_int, [_p, c_int, _p, _p, _p, _p, _p, c_int, c_int, c_int, c_int, c_int, c_int,
                                           c_float, _p, _p, c_int, _p, _p, _p, c_int]),
    "lc2is_grad_to_bf16": (c_int, [_p, c_int, c_int, c_int, _p, _p]),
    "lc2is_count_valid": (c_int, [_p, c_int64, c_int, c_int64, _p, _p]),
    "lc2is_mean_scale": (c_int, [_p, c_float, _p, _p]),
    "lc2is_finalize_loss": (c_int, [_p, _p, _p, _p]),
    "lc2is_mean_scale_finalize": (c_int, [_p, c_float, _p, _p, _p, _p]),
    "lc2is_upsample_ce_fwd_bwd": (c_int, [_p, _p, c_int, c_int, c_int, c_int, c_int, c_int, c_int64, _p, _p,
                                          _p, _p, _p]),
    "lc2is_ce_weight_sum": (c_int, [_p, c_int64, c_int, c_int64, _p, _p, _p]),
    "lc2is_upsample_ce_fwd_bwd_ex": (c_int, [_p, _p, c_int, c_int, c_int, c_int, c_int, c_int, c_int64, _p, c_float,
                                             _p, _p, _p, _p, _p]),
    "lc2is_ce_split_supported": (c_int, [c_int, c_int, c_int, c_int]),
    "lc2is_ce_labels_prepass": (c_int, [_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int64, _p, _p, _p, _p]),
    "lc2is_upsample_ce_packed": (c_int, [_p, _p, c_int, c_int, c_int, c_int, c_int, c_int, _p, _p, _p]),
    "lc2is_argmax_confmat": (c_int, [_p, c_int, c_int, c_int, c_int, c_int, _p, c_int, c_int, _p, _p, _p, _p]),
    "lc2is_argmax_confmat_lowres": (c_int, [_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, _p, c_int,
                                            c_int, _p, _p, _p, _p]),
    "lc2is_argmax_confmat_lowres_packed": (c_int, [_p, c_int, c_int, c_int, c_int, c_int, c_int, _p, _p, _p, _p, _p]),
    "lc2is_ragged_tiles": (c_int64, [c_int, c_int]),
    "lc2is_argmax_confmat_ragged": (c_int, [_p, c_int, c_int, c_int, c_int, c_int, _p, c_int64, _p, _p, _p, _p, _p]),
    "lc2is_ce_argmax_fused_supported": (c_int, [c_int, c_int, c_int, c_int, c_int]),
    "lc2is_ce_argmax_fused_packed": (c_int, [_p, _p, c_int, c_int, c_int, c_int, c_int, c_int, _p, _p, c_int, _p, _p, _p, _p, _p]),
    "lc2is_pack_labels": (c_int, [_p, c_int64, c_int, c_int64, _p, _p, _p]),
    "lc2is_step_ce_labels": (c_int, [_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int64, _p, _p, _p, _p]),
    "lc2is_step_ce": (c_int, [_p, _p, _p, c_int, c_int, c_int, c_int, c_int, c_int, c_int64, _p, _p, _p, _p]),
    "lc2is_step_argmax": (c_int, [_p, _p, _p, c_int, c_int, c_int, c_int, c_int, c_int, _p, _p]),
    "lc2is_head_step_workspace": (c_int64, [c_int, c_int, c_int, c_int, c_int, c_int]),
    "lc2is_head_step_host": (c_int, [_p, _p, _p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int64,
                                     c_float, c_int, _p, _p, _p, _p, _p, _p, _p, c_int, c_int]),
    "lc2is_head_step_host_submit": (c_int, [_p, _p, _p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int64,
                                            c_float, c_int, _p, _p, _p, _p, _p, _p, _p, c_int, c_int, POINTER(c_void_p)]),
    "lc2is_head_step_host_wait": (c_int, [_p]),
    "lc2is_ce_labels_prepass_packed": (c_int, [_p, c_int, c_int, c_int, c_int, c_int, c_int, _p, _p, _p]),
    "lc2is_pack_threads": (c_int, []),
    "lc2is_host_label_bytes": (c_int, [c_int]),
    "lc2is_expand_labels": (c_int, [_p, c_int64, c_int, c_int64, _p, _p, _p]),
    "lc2is_contrastive_fwd": (c_int, [_p, _p, c_int, c_int, c_int, c_int, c_int64, _p, _p, _p, _p, _p]),
    "lc2is_contrastive_bwd": (c_int, [_p, _p, c_int, c_int, c_int, c_int, c_int64, _p, _p, _p, _p, _p]),
    "lc2is_pack_labels_host_begin": (c_int, [_p, c_int64, c_int, c_int64, _p, POINTER(c_void_p)]),
    "lc2is_pack_labels_host_end": (c_int, [_p]),
    "lc2is_pack_labels_host": (c_int, [_p, c_int64, c_int, c_int64, _p]),
}
for _name, (_res, _args) in SIGNATURES.items():
    _fn = getattr(_lib, _name)
    _fn.restype = _res
    _fn.argtypes = _args


def last_error() -> str:
    return (_lib.lc2is_last_error() or b"").decode()


def check(code: int, what: str) -> None:
    if code != 0:
        raise Lc2isError(f"{what} failed (code {code}): {last_error()}")


def ptr(t) -> int:
    """Device (or pinned host) pointer of a torch tensor; None -> NULL."""
    if t is None:
        return None
    return t.data_ptr()


def stream_ptr() -> int:
    import torch
    return torch.cuda.current_stream().cuda_stream


def class_pad(C: int) -> int:
    return _lib.lc2is_class_pad(C)


def launch_count() -> int:
    return int(_lib.lc2is_launch_count())


lib = _lib
