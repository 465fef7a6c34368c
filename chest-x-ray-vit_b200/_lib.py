"""ctypes binding of libvitk.so (include/vitk.h).  No fallback: if the library is missing or a
call fails, a RuntimeError is raised with the library's own message."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("VITK_LIB") or os.path.join(_HERE, "libvitk.so")   # VITK_LIB: A/B builds (tools/build_variants.sh)

# enum vitk_epilogue
EPI_STORE_BF16 = 0
EPI_BIAS_BF16 = 1
EPI_BIAS_GELU_BF16 = 2
EPI_BIAS_RESID_F32 = 3
EPI_PATCH_F32 = 4
EPI_DGELU_BF16 = 5
EPI_ACCUM_F32 = 6
EPI_STORE_F32 = 7
EPI_BIAS_GELUG_BF16 = 8
EPI_MUL_BF16 = 9
EPI_UNPATCH_F32 = 10


class GemmArgs(C.Structure):
    _fields_ = [
        ("a", C.c_void_p), ("b", C.c_void_p),
        ("M", C.c_int64), ("N", C.c_int64), ("K", C.c_int64),
        ("lda", C.c_int64), ("ldb", C.c_int64),
        ("a_mn_major", C.c_int32), ("b_mn_major", C.c_int32),
        ("epilogue", C.c_int32), ("split_k", C.c_int32),
        ("d", C.c_void_p), ("ldd", C.c_int64),
        ("d2", C.c_void_p),
        ("bias", C.c_void_p),
        ("aux", C.c_void_p), ("ld_aux", C.c_int64),
        ("rows_in", C.c_int64), ("rows_out", C.c_int64), ("row_off", C.c_int64),
        ("tile_n", C.c_int32), ("max_ctas", C.c_int32), ("variant", C.c_int32),
    ]


_p, _i64, _f, _sz = C.c_void_p, C.c_int64, C.c_float, C.c_size_t
_PROTOS = {
    "vitk_version": (C.c_int, []),
    "vitk_check_device": (C.c_int, [C.c_int]),
    "vitk_last_error": (C.c_char_p, []),
    "vitk_patchify_u8": (C.c_int, [_p, _i64, _i64, _i64, _i64, C.POINTER(C.c_float), C.POINTER(C.c_float), _p, _p]),
    "vitk_patchify_f32": (C.c_int, [_p, _i64, _i64, _i64, _i64, _p, _p]),
    "vitk_hflip_u8": (C.c_int, [_p, _p, _i64, _i64, _i64, _p]),
    "vitk_layernorm_fwd": (C.c_int, [_p, _i64, _p, _p, _f, _i64, _i64, _p, _p, _p, _p]),
    "vitk_layernorm_fwd_rows": (C.c_int, [_p, _i64, _p, _p, _f, _i64, _i64, _i64, _p, _p, _p, _p]),
    "vitk_layernorm_bwd": (C.c_int, [_p, _p, _i64, _p, _p, _p, _p, _i64, _i64, _p, _p, _p, _p, _p]),
    "vitk_layernorm_bwd_rows": (C.c_int, [_p, _p, _i64, _p, _p, _p, _p, _i64, _i64, _i64, _p, _p, _p, _p, _p]),
    "vitk_gemm_bf16": (C.c_int, [C.POINTER(GemmArgs), _p]),
    "vitk_colsum_bf16": (C.c_int, [_p, _i64, _i64, _i64, _p, _p]),
    "vitk_attn_fwd": (C.c_int, [_p, _i64, _i64, _i64, _f, _p, _p, _p]),
    "vitk_attn_probs": (C.c_int, [_p, _p, _i64, _i64, _i64, _f, _p, _p]),
    "vitk_attn_cls_fwd": (C.c_int, [_p, _i64, _i64, _i64, _f, _p, _p, _p]),
    "vitk_attn_cls_bwd": (C.c_int, [_p, _p, _p, _p, _i64, _i64, _i64, _f, _p, _p]),
    "vitk_attn_bwd_workspace_bytes": (_sz, [_i64, _i64, _i64]),
    "vitk_attn_bwd": (C.c_int, [_p, _p, _p, _p, _i64, _i64, _i64, _f, _p, _p, _p]),
    "vitk_embed_cls": (C.c_int, [_p, _p, _i64, _i64, _i64, _p, _p]),
    "vitk_embed_bwd": (C.c_int, [_p, _i64, _i64, _i64, _p, _p, _p, _p, _p]),
    "vitk_head_fwd": (C.c_int, [_p, _i64, _i64, _i64, _i64, _p, _p, _f, _p, _p, _p, _p, _p, _p, _p, _p, _p]),
    "vitk_head_bwd": (C.c_int, [_p, _p, _p, _p, _p, _p, _i64, _i64, _i64, _i64, _p, _p, _p, _p, _p, _p, _p, _p]),
    "vitk_multilabel_counts": (C.c_int, [_p, _p, _i64, _i64, _f, _p, _p]),
    "vitk_cast_f32_bf16": (C.c_int, [_p, _p, _i64, _p]),
    "vitk_fill_zero": (C.c_int, [_p, _sz, _p]),
    "vitk_adamw": (C.c_int, [_p, _p, _p, _p, _p, _i64, _f, _f, _f, _f, _f, _f, _f, _p, C.c_int, _p, _p]),
    "vitk_adamw_tick": (C.c_int, [_p, C.c_int, _f, _f, _p, _p]),
    "vitk_sumsq_f32": (C.c_int, [_p, _i64, _p, _p, _p]),
    "vitk_sumsq_scratch_floats": (C.c_int64, []),
    "vitk_shard_mean": (C.c_int, [_p, _p, _i64, _i64, C.c_int, _f, C.c_int, _p]),
    "vitk_clip_scale": (C.c_int, [_p, _f, _p, _p]),
    "vitk_launch_count": (C.c_int64, []),
    "vitk_gemm_plan": (C.c_int, [C.POINTER(GemmArgs), C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int),
                                 C.POINTER(C.c_int)]),
    "vitk_debug_timeline": (C.c_int, [_p]),
    "vitk_debug_stamp": (C.c_int, [C.c_int64, _p]),
}

_lib = None


def lib() -> C.CDLL:
    """The loaded library; raises if it has not been built (python __graft_entry__.py build)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                               "(there is no CPU or PyTorch fallback for the vitk kernels)")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in _PROTOS.items():
            fn = getattr(L, name)          # AttributeError if the .so is stale
            fn.restype, fn.argtypes = res, args
        _lib = L
    return _lib


def exported_symbols():
    return sorted(_PROTOS)


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = lib().vitk_last_error().decode(errors="replace")
        raise RuntimeError(f"libvitk {what} failed (rc={rc}): {msg}")
