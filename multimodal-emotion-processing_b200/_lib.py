"""ctypes binding of libmmemo.so (C ABI declared in include/mmemo.h).

The library is built in-tree by ``__graft_entry__.build()`` / ``make -C csrc``.  There is no CPU
fallback: if the shared object is missing or a call fails, this module raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmmemo.so")

_vp, _i64, _i32, _f32, _u64 = C.c_void_p, C.c_int64, C.c_int, C.c_float, C.c_uint64

# name -> argtypes (restype is always int unless noted).  Mirrors include/mmemo.h one to one.
_LINEAR_FWD = [_vp, _i32, _i64, _vp, _i64, _vp, _vp, _i64, _vp, _i64, _i64, _i64, _i64, _i32, _i32, _vp]
_LINEAR_BWD_X = [_vp, _i64, _vp, _i64, _vp, _i64, _vp, _i64, _i64, _i64, _i64, _i32, _vp]
_LINEAR_BWD_W = [_vp, _i64, _vp, _i32, _i64, _vp, _i64, _vp, _i64, _i64, _i64, _i32, _vp]
_ATTN_FWD = [_vp, _i64, _vp, _i64, _vp, _i64, _vp, _i64, _i64, _vp, _vp, _vp, _vp, _i64, _vp,
             _i64, _i64, _i64, _i64, _i64, _vp]
_ATTN_BWD = [_vp, _i64, _vp, _i64, _vp, _i64, _vp, _i64, _vp, _i64, _i64, _vp, _vp, _vp, _vp, _vp,
             _i64, _vp, _vp, _i64, _vp, _i64, _vp, _i64, _vp, _vp, _vp, _i64, _i64, _i64, _i64,
             _i64, _vp]
_LN_FWD = [_vp, _i64, _vp, _i64, _vp, _vp, _vp, _vp, _i64, _vp, _vp, _i64, _i64, _f32, _i32, _vp]
_LN_BWD = [_vp, _i64, _vp, _i64, _vp, _i64, _vp, _vp, _vp, _i64, _vp, _vp, _vp, _i64, _vp, _i64,
           _vp, _vp, _vp, _vp, _i64, _i64, _i32, _vp]
_ROWSUM = [_vp, _i64, _vp, _i64, _i64, _i64, _vp]
_POOL_FWD = [_vp, _vp, _i32, _i32, _i64, _i64, _vp, _vp, _vp]
_POOL_BWD = [_vp, _vp, _vp, _vp, _i32, _i32, _i64, _i64, _vp]
_POOL_FWD_MULTI = [_i32, _vp, _vp, _i32, _i32, _i64, _i64, _vp, _vp]
_POOL_MULTI_ARG = [_i32, _vp, _vp, _i32, _i32, _vp, _i64, _vp, _vp, _vp]
_POOL_BWD_MULTI = [_i32, _vp, _vp, _vp, _vp, _i32, _i32, _vp, _i64, _vp]
_DROPOUT = [_vp, _vp, _i64, _f32, _u64, _vp]
_FOLD_UQ = [_vp, _i64, _i64, _i64] + [_vp] * 6 + [_vp]

class AttnProblem(C.Structure):
    """mmemo_attn_problem of include/mmemo.h (field order and types must match)."""
    _fields_ = [("q", _vp), ("k", _vp), ("v", _vp), ("ldq", _i64), ("ldk", _i64), ("ldv", _i64),
                ("mask", _vp), ("mask_bs", _i64), ("s_prev", _vp), ("c", _vp), ("s_out", _vp),
                ("lds", _i64), ("o", _vp), ("ldo", _i64), ("lse", _vp),
                ("B", _i64), ("H", _i64), ("Lq", _i64), ("Lk", _i64), ("hd", _i64),
                ("d_o", _vp), ("lddo", _i64), ("s", _vp), ("ds_next", _vp),
                ("dq", _vp), ("dk", _vp), ("dv", _vp), ("lddq", _i64), ("lddk", _i64),
                ("lddv", _i64), ("ds_prev", _vp), ("dc", _vp)]


class EnsembleMember(C.Structure):
    """mmemo_ensemble_member of include/mmemo.h (field order and types must match)."""
    _fields_ = [("x0", _vp), ("ld0", _i64), ("x1", _vp), ("ld1", _i64), ("w0", _vp), ("w1", _vp),
                ("b0", _vp), ("ln_gamma", _vp), ("ln_beta", _vp), ("w_out", _vp), ("b_out", _vp),
                ("trans", _vp)]


HEAD_BILINEAR, HEAD_STATE_TRANSFER = 0, 1      # MMEMO_HEAD_* of include/mmemo.h

SIGNATURES = {
    "mmemo_version": [],
    "mmemo_stream_set_workspace": [_vp, _vp, _i64],
    "mmemo_stream_set_sm_budget": [_vp, _i32],
    "mmemo_stream_set_pdl": [_vp, _i32],
    "mmemo_stream_reset": [_vp],
    "mmemo_gemm_uses_tensor_cores": [_i64, _i64, _i64, _i64, _i64, _i64, _i32],
    "mmemo_resattn_uses_tensor_cores": [_i64, _i64, _i64, _i64],
    "mmemo_linear_fwd_f32": _LINEAR_FWD, "mmemo_linear_fwd_bf16": _LINEAR_FWD,
    "mmemo_linear_bwd_x_f32": _LINEAR_BWD_X, "mmemo_linear_bwd_x_bf16": _LINEAR_BWD_X,
    "mmemo_linear_bwd_w_f32": _LINEAR_BWD_W, "mmemo_linear_bwd_w_bf16": _LINEAR_BWD_W,
    "mmemo_linear_fwd_grouped_bf16": [_i32] + [_vp] * 15 + [_vp],
    "mmemo_linear_fwd_grouped_dropout_bf16": [_i32] + [_vp] * 14 + [_f32, _vp, _vp],
    "mmemo_linear_bwd_x_grouped_bf16": [_i32] + [_vp] * 12 + [_vp],
    "mmemo_linear_bwd_w_grouped_bf16": [_i32] + [_vp] * 9 + [_i32, _vp],
    "mmemo_linear_fwd_grouped_f32": [_i32] + [_vp] * 10 + [_vp],
    "mmemo_linear_bwd_x_grouped_f32": [_i32] + [_vp] * 9 + [_vp],
    "mmemo_linear_bwd_w_grouped_f32": [_i32] + [_vp] * 10 + [_vp],
    "mmemo_resattn_fwd_f32": _ATTN_FWD, "mmemo_resattn_fwd_bf16": _ATTN_FWD,
    "mmemo_resattn_bwd_f32": _ATTN_BWD, "mmemo_resattn_bwd_bf16": _ATTN_BWD,
    "mmemo_resattn_fwd_grouped_bf16": [_i32, _vp, _vp],
    "mmemo_resattn_bwd_grouped_bf16": [_i32, _vp, _vp],
    "mmemo_resattn_uses_mma": [_i64, _i64, _i64, _i64, _i32, _i32],
    "mmemo_resattn_kernel_path": [_i64, _i64, _i64, _i64, _i32],
    "mmemo_add_ln_fwd_f32": _LN_FWD, "mmemo_add_ln_fwd_bf16": _LN_FWD,
    "mmemo_add_ln_bwd_f32": _LN_BWD, "mmemo_add_ln_bwd_bf16": _LN_BWD,
    "mmemo_add_ln_fwd_grouped_f32": [_i32] + [_vp] * 9 + [_i64, _f32, _i32, _vp],
    "mmemo_add_ln_fwd_grouped_bf16": [_i32] + [_vp] * 9 + [_i64, _f32, _i32, _vp],
    "mmemo_add_ln_bwd_grouped_f32": [_i32] + [_vp] * 14 + [_i64, _vp],
    "mmemo_add_ln_bwd_grouped_bf16": [_i32] + [_vp] * 14 + [_i64, _vp],
    "mmemo_colsum_grouped_bf16": [_i32, _vp, _vp, _vp, _i64, _vp],
    "mmemo_rowsum_f32": _ROWSUM, "mmemo_rowsum_bf16": _ROWSUM,
    "mmemo_cast_f32_to_bf16": [_vp, _vp, _i64, _vp],
    "mmemo_cast_bf16_to_f32": [_vp, _vp, _i64, _vp],
    "mmemo_cast_f32_to_bf16_multi": [_i32, _vp, _vp, _vp, _vp],
    "mmemo_sqmean_fwd_f32": [_vp, _i64, _vp, _vp], "mmemo_sqmean_fwd_bf16": [_vp, _i64, _vp, _vp],
    "mmemo_sqmean_bwd_f32": [_vp, _vp, _i64, _vp, _vp],
    "mmemo_sqmean_bwd_bf16": [_vp, _vp, _i64, _vp, _vp],
    "mmemo_sum_grouped_f32": [_i32, _vp, _vp, _vp, _vp, _vp],
    "mmemo_sum_grouped_bf16": [_i32, _vp, _vp, _vp, _vp, _vp],
    "mmemo_cast_pad_f32_to_bf16_multi": [_i32] + [_vp] * 6 + [_vp],
    "mmemo_dropout_f32": _DROPOUT, "mmemo_dropout_bf16": _DROPOUT,
    "mmemo_dropout_multi_f32": [_i32, _vp, _vp, _vp, _vp, _f32, _vp, _vp],
    "mmemo_dropout_multi_bf16": [_i32, _vp, _vp, _vp, _vp, _f32, _vp, _vp],
    "mmemo_proj_dropout_bwd_bf16": [_i32] + [_vp] * 6 + [_f32] + [_vp] * 6,
    "mmemo_pool_fwd_f32": _POOL_FWD, "mmemo_pool_fwd_bf16": _POOL_FWD,
    "mmemo_pool_bwd_f32": _POOL_BWD, "mmemo_pool_bwd_bf16": _POOL_BWD,
    "mmemo_pool_fwd_multi_f32": _POOL_FWD_MULTI, "mmemo_pool_fwd_multi_bf16": _POOL_FWD_MULTI,
    "mmemo_pool_fwd_multi_arg_f32": _POOL_MULTI_ARG, "mmemo_pool_fwd_multi_arg_bf16": _POOL_MULTI_ARG,
    "mmemo_pool_bwd_multi_f32": _POOL_BWD_MULTI, "mmemo_pool_bwd_multi_bf16": _POOL_BWD_MULTI,
    "mmemo_ensemble_head_fwd": [_i32, _i32, _vp, _i64, _i64, _i64, _i64, _i64, _f32, _vp, _vp],
    "mmemo_ensemble_head_fwd_members": [_i32, _i32, _vp, _i64, _i64, _i64, _i64, _i64, _f32, _vp,
                                        _vp, _vp],
    "mmemo_fold_uncertainty_f32": _FOLD_UQ, "mmemo_fold_uncertainty_bf16": _FOLD_UQ,
    "mmemo_state_transfer_fwd": [_vp, _vp, _vp, _i64, _i64, _i64, _vp],
    "mmemo_state_transfer_bwd": [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _i64, _vp],
    "mmemo_bilinear_head_fwd": [_vp] * 9 + [_i64, _i64, _f32, _vp],
    "mmemo_bilinear_head_bwd": [_vp] * 15 + [_i64, _i64, _f32, _vp],
    "mmemo_circle_loss_fwd": [_vp, _vp, _vp, _i64, _i64, _vp],
    "mmemo_circle_loss_bwd": [_vp, _vp, _vp, _vp, _i64, _i64, _vp],
    "mmemo_rdrop_kl_fwd": [_vp, _vp, _i64, _i64, _vp],
    "mmemo_rdrop_kl_bwd": [_vp, _vp, _vp, _i64, _i64, _vp],
    "mmemo_state_transfer_fwd_multi": [_i32, _vp, _vp, _vp, _vp, _i64, _i64, _vp],
    "mmemo_state_transfer_bwd_multi": [_i32] + [_vp] * 7 + [_i64, _i64, _vp],
    "mmemo_bilinear_head_fwd_multi": [_i32] + [_vp] * 10 + [_i64, _f32, _vp],
    "mmemo_bilinear_head_bwd_multi": [_i32] + [_vp] * 16 + [_i64, _f32, _vp],
    "mmemo_circle_loss_fwd_multi": [_i32, _vp, _vp, _vp, _vp, _i64, _vp, _vp],
    "mmemo_circle_loss_bwd_multi": [_i32] + [_vp] * 6 + [_i64, _vp],
    "mmemo_rdrop_kl_fwd_multi": [_i32, _vp, _vp, _i64, _vp, _vp],
    "mmemo_rdrop_kl_bwd_multi": [_i32, _vp, _vp, _vp, _vp, _i64, _vp],
    "mmemo_clip_grads_f32": [_i32, _vp, _vp, _vp, _f32, _vp],
    "mmemo_grad_sqnorm_multi_f32": [_i32, _vp, _vp, _vp, _vp, _vp],
    "mmemo_adam_step_multi_f32": [_i32] + [_vp] * 9 + [_f32, _f32, _f32, _i32, _vp, _f32, _vp],
    "mmemo_assemble_batch_f32": [_vp, _vp, _vp, _vp, _vp, _i64, _i64, _i64, _i32, _i32, _f32, _vp],
    "mmemo_assemble_stats_batch_f32": [_vp, _vp, _vp, _vp, _vp, _i64, _i64, _i64, _i32, _i32, _f32,
                                       _vp],
    "mmemo_allreduce_sum_f32": [_vp, _vp, _vp, _i64, _i64, _i64, _i32, _i32, _i32, _vp],
}

_lib = None
ERRORS = {-1: "MMEMO_ERR_ARG", -2: "MMEMO_ERR_SHAPE (unsupported shape)", -3: "MMEMO_ERR_CUDA"}


def load() -> C.CDLL:
    """Load libmmemo.so once and attach prototypes.  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; "
            "g.build()'` (nvcc, sm_100a).  mmemo_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, args in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the .so does not export a declared symbol
        fn.argtypes = args
        fn.restype = C.c_int
    lib.mmemo_last_error.argtypes = []
    lib.mmemo_last_error.restype = C.c_char_p
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        detail = ""
        if rc == -3:
            detail = ": " + (load().mmemo_last_error() or b"").decode()
        raise RuntimeError(f"{what} failed with {ERRORS.get(rc, rc)}{detail}")
