"""ctypes binding of libklab_b200.so (the C ABI declared in include/klab_b200.h).

There is deliberately no fallback: if the shared library is missing it is built with nvcc, and if that is
impossible, or a compute entry is called without an sm_100 device, a RuntimeError is raised.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libklab_b200.so")

F32, BF16 = 0, 1
ACT_NONE, ACT_RELU, ACT_GELU, ACT_RELU_BWD, ACT_GELU_BWD, ACT_GELU_SAVE_GRAD, ACT_MUL_AUX = 0, 1, 2, 3, 4, 5, 6


class GemmEpilogue(C.Structure):
    _fields_ = [
        ("bias", C.c_void_p), ("residual", C.c_void_p), ("aux_in", C.c_void_p), ("aux_out", C.c_void_p),
        ("ldr", C.c_longlong), ("ld_aux_in", C.c_longlong), ("ld_aux_out", C.c_longlong),
        ("alpha", C.c_float), ("act", C.c_int), ("accumulate", C.c_int),
        ("out_dtype", C.c_int), ("res_dtype", C.c_int), ("aux_in_dtype", C.c_int),
        ("dropout_p", C.c_float), ("dropout_seed", C.c_ulonglong), ("dropout_seed_ptr", C.c_void_p),
    ]


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            from .build import build
            build()
        _lib = C.CDLL(LIB_PATH)
        _declare(_lib)
        if _lib.klab_abi_version() != 1:
            raise RuntimeError("libklab_b200.so ABI version mismatch: rebuild with python -m klab_multimodalmodel_b200.build")
    return _lib


def check(rc: int) -> None:
    if rc != 0:
        raise RuntimeError(f"libklab_b200: {lib().klab_last_error().decode()} (status {rc})")


_vp, _i, _ll, _f, _ull, _d = C.c_void_p, C.c_int, C.c_longlong, C.c_float, C.c_ulonglong, C.c_double

# name -> argtypes (restype is int unless listed in _RESTYPES); mirrors include/klab_b200.h
SIGNATURES = {
    "klab_abi_version": [],
    "klab_last_error": [],
    "klab_check_device": [],
    "klab_launch_count": [],
    "klab_set_sm_reserve": [_i],
    "klab_sm_budget": [],
    "klab_set_dynamic_sched": [_i],
    "klab_gemm": [_vp, _i, _i, _i, _i, _vp, _ll, _i, _vp, _ll, _i, _vp, _ll, C.POINTER(GemmEpilogue)],
    "klab_gemm_set_force": [_i, _i, _i],
    "klab_gemm_last_config": [_vp, _vp, _vp],
    "klab_gemm_simt": [_vp, _i, _i, _i, _i, _vp, _ll, _i, _vp, _ll, _i, _vp, _ll, C.POINTER(GemmEpilogue)],
    "klab_rmsnorm_fwd": [_vp, _i, _ll, _i, _vp, _ll, _vp, _f, _vp, _ll, _i, _ll, _vp],
    "klab_rmsnorm_bwd": [_vp, _i, _ll, _i, _vp, _ll, _vp, _ll, _vp, _vp, _vp, _ll, _vp, _ll, _vp, _i, _vp],
    "klab_rmsnorm_bwd_dropout": [_vp, _i, _ll, _i, _vp, _ll, _vp, _ll, _vp, _vp, _vp, _ll, _vp, _ll, _vp, _i, _vp, _vp, _f, _ull, _vp],
    "klab_norm_bwd_workspace_bytes": [_ll, _i],
    "klab_layernorm_fwd": [_vp, _i, _ll, _i, _vp, _ll, _vp, _vp, _f, _vp, _ll, _vp, _ll, _i, _ll, _vp, _vp],
    "klab_layernorm_bwd": [_vp, _i, _ll, _i, _vp, _ll, _i, _ll, _vp, _ll, _vp, _vp, _vp, _vp, _ll, _vp, _ll, _vp, _vp, _i, _vp],
    "klab_colsum": [_vp, _i, _ll, _i, _vp, _ll, _vp, _i, _vp],
    "klab_colsum_workspace_bytes": [_ll, _i],
    "klab_t5_attention_fwd": [_vp, _i, _i, _i, _i, _i, _i, _vp, _ll, _vp, _ll, _vp, _ll, _vp, _ll, _vp, _vp, _i, _i, _i, _i, _vp, _f, _ull, _vp],
    "klab_t5_attention_bwd": [_vp, _i, _i, _i, _i, _i, _i, _vp, _ll, _vp, _ll, _vp, _ll, _vp, _vp, _ll, _vp, _vp, _vp, _vp, _vp,
                              _i, _i, _i, _i, _vp, _vp, _f, _ull, _vp, _vp],
    "klab_t5_attention_bwd_workspace_bytes": [_i, _i, _i, _i],
    "klab_t5_attention_decode_beam": [_vp, _i, _i, _i, _i, _i, _vp, _ll, _vp, _ll, _vp, _ll, _vp, _ll, _i, _vp, _ll, _vp, _vp, _i, _i],
    "klab_swin_attention_fwd": [_vp, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _ll, _vp, _ll, _vp, _vp, _vp],
    "klab_swin_attention_bwd": [_vp, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _ll, _vp, _vp, _ll, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp],
    "klab_swin_cpb_fwd": [_vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp],
    "klab_swin_cpb_bwd": [_vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i],
    "klab_embedding_fwd": [_vp, _i, _i, _i, _vp, _i, _i, _i, _vp, _ll, _i, _vp, _ll, _vp],
    "klab_embedding_bwd": [_vp, _i, _i, _i, _vp, _i, _i, _i, _vp, _ll, _i, _vp, _ll],
    "klab_patchify": [_vp, _i, _i, _i, _i, _i, _i, _vp, _vp, _ll],
    "klab_image_normalize": [_vp, _i, _i, _i, _ll, _vp, _d, _vp, _vp, _i, _vp],
    "klab_patch_merge": [_vp, _i, _i, _i, _i, _vp, _vp, _i],
    "klab_ce_fwd": [_vp, _i, _ll, _i, _vp, _ll, _vp, _vp, _vp, _vp, _vp],
    "klab_ce_bwd": [_vp, _i, _ll, _i, _vp, _ll, _i, _vp, _vp, _vp, _vp],
    "klab_lmhead_ce_workspace_bytes": [_ll, _i],
    "klab_lmhead_ce_fwd": [_vp, _ll, _i, _i, _vp, _ll, _vp, _ll, _f, _vp, _vp, _vp, _vp, _vp],
    "klab_lmhead_ce_bwd_chunk": [_vp, _ll, _i, _vp, _ll, _vp, _ll, _f, _vp, _vp, _vp, _vp, _i, _i, _vp, _ll],
    "klab_cast": [_vp, _i, _i, _ll, _vp, _vp],
    "klab_greedy_step": [_vp, _i, _i, _vp, _ll, _vp, _ll, _i, _vp, _i, _i],
    "klab_beam_topk": [_vp, _i, _i, _i, _vp, _ll, _vp, _vp, _vp],
    "klab_beam_update": [_vp, _i, _i, _i, _i, _i, _i, _f, _i, _vp, _vp, _vp, _vp, _vp, _ll, _vp, _vp, _vp, _vp, _vp, _vp, _vp],
    "klab_dropout_apply": [_vp, _i, _ll, _vp, _vp, _f, _ull, _vp],
    "klab_seed_advance": [_vp, _vp],
    "klab_adam_chunk_elems": [],
    "klab_adam_step": [_vp, _vp, _vp, _i, _d, _d, _d, _d, _d, _ll, _d],
}
_RESTYPES = {"klab_last_error": C.c_char_p, "klab_launch_count": C.c_longlong,
             "klab_norm_bwd_workspace_bytes": C.c_longlong, "klab_colsum_workspace_bytes": C.c_longlong,
             "klab_t5_attention_bwd_workspace_bytes": C.c_longlong, "klab_lmhead_ce_workspace_bytes": C.c_longlong}


def _declare(l: C.CDLL) -> None:
    for name, args in SIGNATURES.items():
        fn = getattr(l, name)
        fn.argtypes = args
        fn.restype = _RESTYPES.get(name, C.c_int)
