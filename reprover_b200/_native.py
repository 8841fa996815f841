"""ctypes binding of `librpx.so` (the C ABI declared in `include/rpx.h`).

Loading never falls back: if the library is missing, `load()` raises with the
build command; if a compute entry point fails, `check()` raises `RpxError` with
the library's message.  No torch types cross this boundary — callers pass
`tensor.data_ptr()` integers and the raw `cudaStream_t`.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path
from typing import Optional

from ._build import LIB_PATH

RPX_OK = 0
RPX_ERR_INVALID = 1
RPX_ERR_CUDA = 2
RPX_ERR_UNSUPPORTED = 3
RPX_ERR_WORKSPACE = 4
RPX_ERR_MASK = 5

RPX_TOPK_AUTO = 0
RPX_TOPK_FORCE_MMA = 1
RPX_TOPK_FORCE_STREAM = 2
RPX_TOPK_FORCE_EXACT = 4
TOPK_MAX_K = 1024

RPX_DTYPE_BF16 = 0
RPX_DTYPE_F32 = 1
RPX_N_KERNEL_CLASSES = 7
KERNEL_CLASS_NAMES = ("embed", "qkv_gemm", "attention", "oproj_gemm", "ffn_up_gemm", "ffn_down_gemm", "pool")


class RpxError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"rpx error {code}: {msg}")
        self.code = code


class T5Config(C.Structure):
    _fields_ = [
        ("vocab_size", C.c_int32),
        ("d_model", C.c_int32),
        ("d_kv", C.c_int32),
        ("d_ff", C.c_int32),
        ("num_layers", C.c_int32),
        ("num_heads", C.c_int32),
        ("rel_buckets", C.c_int32),
        ("rel_max_distance", C.c_int32),
        ("ln_eps", C.c_float),
    ]


_PP = C.POINTER(C.c_void_p)


class T5Weights(C.Structure):
    _fields_ = [
        ("d_shared", C.c_void_p),
        ("d_rel_bias", C.c_void_p),
        ("d_final_ln", C.c_void_p),
        ("h_q", _PP),
        ("h_k", _PP),
        ("h_v", _PP),
        ("h_o", _PP),
        ("h_ln0", _PP),
        ("h_wi0", _PP),
        ("h_wi1", _PP),
        ("h_wo", _PP),
        ("h_ln1", _PP),
    ]


# name -> (restype, argtypes); mirrors include/rpx.h one to one.
_SIGNATURES = {
    "rpx_last_error": (C.c_char_p, []),
    "rpx_version": (C.c_int, []),
    "rpx_device_check": (C.c_int, []),
    "rpx_encoder_packed_bytes": (C.c_size_t, [C.POINTER(T5Config)]),
    "rpx_encoder_create": (C.c_int, [C.POINTER(T5Config), C.POINTER(T5Weights), C.c_void_p, C.c_size_t,
                                     C.c_void_p, C.POINTER(C.c_void_p)]),
    "rpx_encoder_destroy": (C.c_int, [C.c_void_p]),
    "rpx_encoder_workspace_bytes": (C.c_size_t, [C.c_void_p, C.c_int64, C.c_int64]),
    "rpx_encode_bytes": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_int64), C.c_int32, C.c_int32,
                                   C.c_void_p, C.c_int32, C.c_void_p, C.c_size_t, C.c_void_p]),
    "rpx_encode_ids": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p,
                                 C.c_int32, C.c_void_p, C.c_size_t, C.c_void_p]),
    "rpx_encoder_set_latency_tokens": (C.c_int, [C.c_void_p, C.c_int32]),
    "rpx_t5_relative_bucket": (C.c_int32, [C.c_int32, C.c_int32, C.c_int32]),
    "rpx_encoder_set_debug_hidden": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64]),
    "rpx_encoder_set_profiling": (C.c_int, [C.c_void_p, C.c_int32]),
    "rpx_encoder_read_profile": (C.c_int, [C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_int64)]),
    "rpx_index_state_bytes": (C.c_size_t, []),
    "rpx_index_create": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p)]),
    "rpx_index_destroy": (C.c_int, [C.c_void_p]),
    "rpx_index_stats": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_float),
                                  C.POINTER(C.c_float), C.POINTER(C.c_int64)]),
    "rpx_index_topk_workspace_bytes": (C.c_size_t, [C.c_int64, C.c_int32, C.c_int32, C.c_int32]),
    "rpx_index_topk": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p,
                                 C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p,
                                 C.c_size_t, C.c_void_p]),
    "rpx_sim_topk_workspace_bytes": (C.c_size_t, [C.c_int64, C.c_int32, C.c_int32, C.c_int32]),
    "rpx_sim_topk": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.c_int32, C.c_int32,
                               C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                               C.c_int64, C.c_void_p, C.c_size_t, C.c_void_p]),
    "rpx_topk_merge": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p,
                                 C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "rpx_topk_merge_packed": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_void_p]),
    "rpx_debug_set_timeline": (C.c_int, [C.c_void_p, C.c_int32]),
    "rpx_gemm_bf16_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                    C.c_void_p]),
    "rpx_gemm2_bf16_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                     C.c_void_p]),
    "rpx_t5_attention_bf16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_int32), C.c_int32,
                                        C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib: Optional[C.CDLL] = None


def library_path() -> Path:
    return LIB_PATH


def load() -> C.CDLL:
    """Load librpx.so (once).  Raises if it has not been built — there is no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise RuntimeError(
            f"{LIB_PATH} is missing: the CUDA engine is not built. Run "
            f"`python -c 'import __graft_entry__ as g; g.build()'` (or `python -m reprover_b200._build`). "
            f"There is no CPU / PyTorch fallback for this path."
        )
    lib = C.CDLL(str(LIB_PATH))
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here == header/ABI drift
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error() -> str:
    return load().rpx_last_error().decode("utf-8", "replace")


def check(status: int) -> None:
    if status != RPX_OK:
        raise RpxError(status, last_error())
