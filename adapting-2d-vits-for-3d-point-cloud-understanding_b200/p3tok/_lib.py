"""ctypes binding of libp3tok.so (the C ABI declared in include/p3tok.h).

There is no CPU fallback: if the library is missing this module raises at first use, and every
entry point rejects non-CUDA tensors (BASELINE.json north_star: "no Triton, no multi-backend
dispatch and no CPU fallback").
"""
from __future__ import annotations

import ctypes
import os
import re
from typing import List

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("P3TOK_LIB") or os.path.join(_PKG, "libp3tok.so")   # P3TOK_LIB: A/B builds of the same sources
HEADER_PATH = os.path.join(os.path.dirname(os.path.dirname(_PKG)), "include", "p3tok.h")

OK, ERR_INVALID, ERR_UNSUPPORTED, ERR_CUDA, ERR_WORKSPACE = 0, 1, 2, 3, 4
KNN_APF_SQ, KNN_P4P_CDIST = 0, 1
F32, BF16, I32, I64, BF16X3 = 0, 1, 2, 3, 4
ROWS_APF, ROWS_P4P, ROWS_DIRECT = 0, 1, 2
EW_AXPBY, EW_MUL, EW_GELU, EW_GELU_BWD, EW_RELU, EW_RELU_BWD = 0, 1, 2, 3, 4, 5

_i32, _i64, _vp, _int = ctypes.c_int32, ctypes.c_int64, ctypes.c_void_p, ctypes.c_int


class MlpStruct(ctypes.Structure):
    """struct p3tok_mlp (include/p3tok.h)."""
    _fields_ = [
        ("cin", _i32), ("n_pre", _i32), ("pre_dim", _i32 * 4), ("pre_relu", _i32 * 4),
        ("mid_dim", _i32), ("out_dim", _i32), ("out_relu", _i32), ("wdtype", _i32),
        ("w_pre", _vp * 4), ("b_pre", _vp * 4),
        ("w_mid_g", _vp), ("w_mid_f", _vp), ("b_mid", _vp), ("w_out", _vp), ("b_out", _vp),
    ]


class RowsStruct(ctypes.Structure):
    """struct p3tok_rows (include/p3tok.h)."""
    _fields_ = [
        ("kind", _i32), ("C", _i32), ("D", _i32), ("idx_dtype", _i32),
        ("B", _i64), ("N", _i64), ("G", _i64), ("k", _i64),
        ("x", _vp), ("feats", _vp), ("ctr_idx", _vp), ("knn_idx", _vp), ("perm", _vp),
    ]


class VitLayerStruct(ctypes.Structure):
    """struct p3tok_vit_layer (include/p3tok.h): one APFViTLayer folded by apf_model.fold_vit_layer."""
    _fields_ = [(n, _vp) for n in ("qkv_w", "qkv_b", "proj_w", "proj_b", "fc1d_w", "fc1d_b", "fc2u_w", "fc2u_b")]


_f32 = ctypes.c_float

_SIGNATURES = {
    "p3tok_abi_version": (_int, []),
    "p3tok_last_error": (ctypes.c_char_p, []),
    "p3tok_kernel_launches": (_i64, []),
    "p3tok_fps": (_int, [_vp, _i64, _i64, _i64, _vp, _i64, _vp, _vp]),
    "p3tok_fps_nd": (_int, [_vp, _i64, _i64, _i64, _i64, _vp, _i64, _vp, _vp, _vp]),
    "p3tok_square_distance": (_int, [_vp, _i64, _i64, _vp, _i64, _i64, _vp, _vp]),
    "p3tok_gather_points": (_int, [_vp, _i64, _i64, _i64, _vp, _i64, _vp, _vp]),
    "p3tok_knn": (_int, [_vp, _i64, _i64, _i64, _vp, _i64, _i64, _int, _vp, _int, _vp, _vp]),
    "p3tok_knn_workspace_bytes": (_i64, [_i64, _i64]),
    "p3tok_knn_sorted": (_int, [_vp, _i64, _i64, _i64, _vp, _i64, _i64, _int, _vp, _int, _vp, _vp, _i64, _vp]),
    "p3tok_knn_prepare": (_int, [_vp, _i64, _i64, _i64, _vp, _i64, _vp]),
    "p3tok_knn_query": (_int, [_vp, _i64, _i64, _i64, _vp, _i64, _i64, _int, _vp, _int, _vp, _vp]),
    "p3tok_morton_order": (_int, [_vp, _i64, _i64, _vp, _vp, _vp]),
    "p3tok_apf_group": (_int, [_vp, _i64, _i64, _i64, _vp, _vp, _vp, _i64, _i64, _vp, _vp, _vp]),
    "p3tok_group_gather": (_int, [_vp, _vp, _i64, _i64, _i64, _vp, _i64, _i64, _vp, _vp, _vp]),
    "p3tok_patch_embed_workspace_bytes": (_i64, [ctypes.POINTER(MlpStruct), _i64, _i64, _int]),
    "p3tok_patch_embed": (_int, [ctypes.POINTER(RowsStruct), ctypes.POINTER(MlpStruct), _int, _int, _vp, _i64, _vp, _vp]),
    "p3tok_linear_f32": (_int, [_vp, _i64, _i64, _vp, _i64, _vp, _vp, _i64, _int, _vp, _vp]),
    "p3tok_linear_x3_workspace_bytes": (_i64, [_i64, _i64, _i64]),
    "p3tok_linear_x3_f32": (_int, [_vp, _i64, _i64, _vp, _i64, _vp, _vp, _i64, _int, _vp, _vp, _i64, _vp]),
    "p3tok_linear_bf16": (_int, [_vp, _i64, _i64, _vp, _i64, _vp, _vp, _i64, _int, _vp, _vp, _vp, _vp]),
    "p3tok_token_head_f32": (_int, [_vp, _vp, _i64, _i64, _i64, _i64, _i64] + [_vp] * 12),
    "p3tok_group_max": (_int, [_vp, _i64, _i64, _i64, _vp, _vp]),
    "p3tok_linear_tn_f32": (_int, [_vp, _vp, _i64, _i64, _i64, _vp, _int, _vp]),
    "p3tok_colstats_f32": (_int, [_vp, _i64, _i64, _vp, _vp, _vp]),
    "p3tok_bn_act_f32": (_int, [_vp, _i64, _i64, _vp, _vp, _vp, _vp, _int, _vp, _vp]),
    "p3tok_bn_bwd_stats_f32": (_int, [_vp, _vp, _i64, _i64, _vp, _vp, _vp, _vp, _int, _vp, _vp, _vp]),
    "p3tok_bn_bwd_apply_f32": (_int, [_vp, _vp, _i64, _i64, _i64, _vp, _vp, _vp, _vp, _int, _vp, _vp, _vp, _vp]),
    "p3tok_group_max_arg_f32": (_int, [_vp, _i64, _i64, _i64, _vp, _vp, _vp]),
    "p3tok_group_max_bwd_f32": (_int, [_vp, _vp, _i64, _i64, _i64, _int, _vp, _vp]),
    "p3tok_group_sum_f32": (_int, [_vp, _i64, _i64, _i64, _vp, _vp]),
    "p3tok_scatter_rows_add_f32": (_int, [_vp, _vp, _i64, _i64, _i64, _i64, _i64, _vp, _vp, _vp]),
    "p3tok_build_rows_f32": (_int, [ctypes.POINTER(RowsStruct), _vp, _vp]),
    "p3tok_apf_rows_bwd_f32": (_int, [ctypes.POINTER(RowsStruct), _vp, _vp, _vp]),
    "p3tok_gather_points_bwd_f32": (_int, [_vp, _i64, _i64, _i64, _vp, _i64, _vp, _vp]),
    "p3tok_ln_fwd_f32": (_int, [_vp, _i64, _i64, _vp, _vp, _f32, _vp, _vp, _vp, _vp]),
    "p3tok_ln_bwd_f32": (_int, [_vp, _vp, _i64, _i64, _vp, _vp, _vp, _int, _vp, _vp]),
    "p3tok_ln_param_grad_f32": (_int, [_vp, _vp, _i64, _i64, _vp, _vp, _vp, _vp, _vp]),
    "p3tok_attn_fwd_f32": (_int, [_vp, _i64, _i64, _i64, _i64, _f32, _vp, _vp, _vp]),
    "p3tok_attn_bwd_f32": (_int, [_vp, _vp, _vp, _i64, _i64, _i64, _i64, _f32, _vp, _vp, _vp]),
    "p3tok_ew_f32": (_int, [_int, _vp, _vp, _f32, _f32, _i64, _i64, _vp, _vp]),
    "p3tok_apf_vit_workspace_bytes": (_i64, [_i64, _i64, _i64, _i64, _i64]),
    "p3tok_apf_vit_forward": (_int, [_vp, _i64, _i64, _i64, _i64, _i64, _i64, ctypes.POINTER(VitLayerStruct), _i64, _vp, _vp,
                                     _f32, _vp, _vp, _i64, _vp]),
    "p3tok_vit_forward": (_int, [_vp, _i64, _i64, _i64, _i64, _i64, ctypes.POINTER(VitLayerStruct), _i64, _vp, _vp, _vp, _f32, _vp, _vp,
                                 _i64, _vp, _i64, _vp]),
    "p3tok_layernorm_bf16": (_int, [_vp, _i64, _i64, _f32, _vp, _vp, _vp, _vp]),
    "p3tok_attention_bf16": (_int, [_vp, _i64, _i64, _i64, _i64, _vp, _vp]),
    "p3tok_vit_x3_workspace_bytes": (_i64, [_i64, _i64, _i64, _i64, _i64]),
    "p3tok_apf_vit_forward_x3": (_int, [_vp, _i64, _i64, _i64, _i64, _i64, _i64, ctypes.POINTER(VitLayerStruct), _i64, _vp, _vp,
                                        _f32, _vp, _vp, _i64, _vp]),
    "p3tok_vit_forward_x3": (_int, [_vp, _i64, _i64, _i64, _i64, _i64, ctypes.POINTER(VitLayerStruct), _i64, _vp, _vp, _vp, _f32, _vp,
                                    _vp, _i64, _vp, _i64, _vp]),
    "p3tok_layernorm_split": (_int, [_vp, _i64, _i64, _f32, _vp, _vp, _vp, _vp]),
    "p3tok_attention_x3": (_int, [_vp, _i64, _i64, _i64, _i64, _vp, _vp]),
    "p3tok_linear_bf16_ex": (_int, [_vp, _i64, _i64, _vp, _i64, _vp, _int, _i64, _vp, _f32, _f32, _vp, _vp, _vp]),
}


def declared_symbols() -> List[str]:
    """Every function include/p3tok.h declares (used by the symbol-export test)."""
    with open(HEADER_PATH) as f:
        return sorted(set(re.findall(r"P3TOK_API\s+[\w\s\*]+?\b(p3tok_\w+)\s*\(", f.read())))


_lib = None


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(p3tok has no CPU or eager fallback)")
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        if L.p3tok_abi_version() != 3:
            raise RuntimeError("libp3tok.so ABI version mismatch; rebuild")
        _lib = L
    return _lib


class P3tokError(RuntimeError):
    pass


def check(rc: int, what: str) -> None:
    if rc != OK:
        msg = lib().p3tok_last_error().decode("utf-8", "replace")
        kind = {ERR_INVALID: "invalid argument", ERR_UNSUPPORTED: "unsupported", ERR_CUDA: "CUDA failure",
                ERR_WORKSPACE: "workspace too small"}.get(rc, f"error {rc}")
        raise P3tokError(f"{what}: {kind}: {msg}")
