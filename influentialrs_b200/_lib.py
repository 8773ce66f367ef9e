"""ctypes binding of libirs_b200.so (include/irs_b200.h).  There is NO fallback: if the library is
missing or a call fails this raises, so a GPU test can never silently pass on another path."""
from __future__ import annotations

import ctypes as C
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "libirs_b200.so")

_p = C.c_void_p
_i = C.c_int
_l = C.c_int64
_f = C.c_float
_z = C.c_size_t

# name -> (restype, argtypes); mirrors include/irs_b200.h one to one
SIGNATURES = {
    "irs_abi_version": (_i, []),
    "irs_error_string": (C.c_char_p, [_i]),
    "irs_launch_count": (C.c_longlong, []),
    "irs_launch_count_reset": (None, []),
    "irs_embed_gather_fwd": (_i, [_p, _p, _p, _f, _p, _l, _i, _i, _l, _p]),
    "irs_embed_scatter_add_bwd": (_i, [_p, _p, _f, _p, _l, _i, _l, _l, _p]),
    "irs_pif_fwd": (_i, [_p, _p, _p, _p, _p, _i, _i, _l, _p]),
    "irs_pim_attn_fwd": (_i, [_p, _p, _p, _l, _l, _l, _p, _p, _f, _f, _i, _p, _p, _i, _i, _i, _i, _i, _i, _f, C.c_uint64, _p]),
    "irs_pim_attn_fwd_blocked": (_i, [_p, _p, _p, _l, _l, _l, _p, _p, _f, _f, _i, _p, _p, _i, _i, _i, _i, _i, _i, _f, C.c_uint64, _p]),
    "irs_pim_attn_tc_supported": (_i, [_i, _i]),
    "irs_pim_attn_fwd_tc": (_i, [_p, _p, _p, _l, _l, _l, _p, _p, _f, _f, _i, _p, _p, _i, _i, _i, _i, _i, _i, _p, _p]),
    "irs_pim_attn_fwd_tc_blocked": (_i, [_p, _p, _p, _l, _l, _l, _p, _p, _f, _f, _i, _p, _p, _i, _i, _i, _i, _i, _i, _p, _p]),
    "irs_pim_attn_img_supported": (_i, [_i, _i]),
    "irs_qkv_images_bytes": (_z, [_i, _i, _i, _i]),
    "irs_qkv_to_images": (_i, [_p, _p, _p, _l, _l, _l, _p, _i, _i, _i, _i, _i, _p]),
    "irs_pim_attn_fwd_img": (_i, [_p, _p, _p, _f, _f, _i, _p, _i, _i, _i, _i, _i, _i, _p, _p]),
    "irs_pim_attn_bwd": (_i, [_p, _p, _p, _l, _l, _l, _p, _p, _f, _f, _i, _p, _p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _f, C.c_uint64, _p]),
    "irs_pim_attn_bwd_blocked": (_i, [_p, _p, _p, _l, _l, _l, _p, _p, _f, _f, _i, _p, _p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _f, C.c_uint64, _p]),
    "irs_residual_layernorm": (_i, [_p, _p, _p, _p, _p, _p, _p, _p, _f, _p, _l, _i, _p]),
    "irs_linear_prepared_bytes": (_z, [_i, _i]),
    "irs_linear_prepare_weights": (_i, [_p, _i, _i, _p, _p]),
    "irs_linear_tc": (_i, [_p, _l, _p, _p, _i, _p, _l, _p, _p, _p, _p, _p, _f, _p, _l, _l, _i, _i, _p, _p]),
    "irs_decoder_chain_supported": (_i, [_i, _i]),
    "irs_decoder_chain_prepared_bytes": (_z, [_i, _i, _i]),
    "irs_decoder_chain_prepare_weights": (_i, [_p, _p, _p, _p, _i, _i, _p, _p]),
    "irs_decoder_chain_tc": (_i, [_p, _p, _p] + [_p] * 11 + [_f, _f, _f, _p, _p, _p, _i, _i, _l, _i, _i, _p, _p]),
    "irs_in_proj_images_tc": (_i, [_p, _p, _p, _p, _i, _i, _l, _i, _p, _p]),
    "irs_sort_exclusions": (_i, [_p, _i, _i, _l, _l, _p, _p, _p]),
    "irs_exclusions_update": (_i, [_p, _p, _p, _l, _p, _i, _i, _l, _l, _p]),
    "irs_score_topk_workspace_bytes": (_z, [_i, _l, _i, _i]),
    "irs_score_topk": (_i, [_p, _l, _p, _p, _l, _p, _p, _i, _i, _p, _p, _i, _l, _i, _p, _z, _p]),
    "irs_scorer_prepared_bytes": (_z, [_l, _i]),
    "irs_scorer_prepare_weights": (_i, [_p, _l, _i, _p, _p]),
    "irs_score_argmax_tc_workspace_bytes": (_z, [_i, _l, _i]),
    "irs_score_argmax_tc": (_i, [_p, _l, _p, _p, _p, _l, _p, _p, _i, _p, _p, _i, _l, _i, _i, _p, _z, _p]),
    "irs_score_argmax_tc_phase1": (_i, [_p, _l, _p, _p, _p, _l, _p, _p, _i, _p, _i, _l, _i, _i, _p, _z, _p]),
    "irs_score_argmax_tc_phase2": (_i, [_p, _l, _p, _p, _p, _l, _p, _p, _i, _p, _p, _p, _i, _l, _i, _i, _p, _z, _p]),
    "irs_score_topk_tc_workspace_bytes": (_z, [_i, _l, _i, _i]),
    "irs_score_topk_tc": (_i, [_p, _l, _p, _p, _p, _l, _p, _p, _i, _i, _p, _p, _i, _l, _i, _p, _z, _p]),
    "irs_score_lse_gather_workspace_bytes": (_z, [_i, _l, _i, _i]),
    "irs_score_lse_gather": (_i, [_p, _l, _p, _p, _l, _p, _i, _p, _p, _i, _l, _i, _p, _z, _p]),
    "irs_score_lse_gather_tc_workspace_bytes": (_z, [_i, _l, _i]),
    "irs_score_lse_gather_tc": (_i, [_p, _l, _p, _p, _p, _l, _p, _i, _p, _p, _i, _l, _i, _p, _z, _p]),
    "irs_score_rank_workspace_bytes": (_z, [_i, _l, _i]),
    "irs_score_rank": (_i, [_p, _l, _p, _p, _l, _p, _p, _p, _i, _p, _i, _l, _i, _p, _z, _p]),
    "irs_score_rank_tc_workspace_bytes": (_z, [_i, _l, _i]),
    "irs_score_rank_tc": (_i, [_p, _l, _p, _p, _p, _l, _p, _p, _p, _i, _p, _i, _l, _i, _p, _z, _p]),
    "irs_score_select": (_i, [_p, _l, _p, _p, _l, _p, _i, _p, _i, _l, _i, _p]),
    "irs_score_count_ahead_workspace_bytes": (_z, [_i, _l, _i]),
    "irs_score_count_ahead": (_i, [_p, _l, _p, _p, _l, _p, _p, _p, _p, _i, _p, _p, _i, _l, _i, _p, _z, _p]),
    "irs_score_count_ahead_tc": (_i, [_p, _l, _p, _p, _p, _l, _p, _p, _p, _p, _i, _p, _p, _i, _l, _i, _p, _z, _p]),
    "irs_score_ce_bwd": (_i, [_p, _l, _p, _p, _p, _p, _f, _p, _p, _p, _i, _l, _i, _p]),
    "irs_score_ce_bwd_tc_workspace_bytes": (_z, [_i, _l, _i]),
    "irs_score_ce_bwd_tc": (_i, [_p, _l, _p, _p, _p, _p, _f, _p, _p, _p, _i, _l, _i, _p, _z, _p]),
    "irs_topk_merge": (_i, [_p, _p, _i, _i, _i, _p, _p, _p]),
    "irs_topk_sample": (_i, [_p, _p, _i, _i, _i, C.c_uint64, _l, _p, _p, _p]),
    "irs_window_shift": (_i, [_p, _p, _p, _i, _i, _i, _i, _p]),
}

_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -m influentialrs_b200.build` "
                "(nvcc, sm_100a).  influentialrs_b200 has no CPU or PyTorch fallback.")
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(l, name)          # AttributeError here = header/library mismatch
            fn.restype = res
            fn.argtypes = args
        if l.irs_abi_version() != 1:
            raise RuntimeError("libirs_b200.so ABI version mismatch")
        _lib = l
    return _lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = lib().irs_error_string(rc).decode()
        raise RuntimeError(f"libirs_b200 {what} failed ({rc}): {msg}")
