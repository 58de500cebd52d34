"""ctypes binding of libalm_b200.so (the C ABI declared in include/alm_b200.h).

There is no fallback: if the library is missing or a call fails, we raise.  The only torch
objects that cross this boundary are raw `data_ptr()`s and the current CUDA stream handle.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

import torch

_PKG = Path(__file__).resolve().parent
LIB_PATH = _PKG / "libalm_b200.so"

P = C.c_void_p
I = C.c_int
L = C.c_int64
F = C.c_float

# name -> argtypes (stream is always last and always a void*)
SIGNATURES: dict[str, list] = {
    "alm_gemm_bf16": [P, I, L, L, P, I, L, L, P, I, L, L, I, I, I, I, F, P, I, I, P],
    "alm_mqa_attn_fwd": [P, L, P, L, L, P, L, L, P, P, L, P, L, P, L, L, I, I, I, I, I, F, P],
    "alm_mqa_attn_bwd": [P, L, P, L, L, P, L, L, P, L, P, P, P, I, P, L, P, L, P, L, P, P, L, L, I, I, I, I, I, F, P],
    "alm_pack_key_mask": [P, P, I, I, P],
    "alm_embed_gather": [P, I, P, P, I, I, P],
    "alm_embed_scatter": [P, I, P, P, I, I, P],
    "alm_attn_delta": [P, L, P, L, P, L, I, I, I, P],
    "alm_kv_append": [P, L, P, P, L, P, I, I, P],
    "alm_gemv_bf16": [P, L, P, L, P, I, L, P, I, I, I, P],
    "alm_gemm_head_ce": [P, L, P, L, P, P, L, I, P, P, P, P, P, P, L, I, I, I, P],
    "alm_ce_finish": [P, I, P, P, L, P, P, I, P],
    "alm_decode_stack_step": [P, I, P, P, P, P, I, L, P, L, P, L, I, I, I, I, I, F, I, P],
    "alm_mqa_attn_decode": [P, L, P, P, L, P, I, P, L, P, L, P, I, I, I, F, P],
    "alm_bias_gather_fwd": [P, P, P, P, I, I, I, L, P],
    "alm_bias_gather_bwd": [P, P, P, P, I, I, I, L, P],
    "alm_hc_pre_fwd": [P] * 12 + [P, P, P, P, P, I, I, I, P],
    "alm_hc_pre_bwd": [P] * 12 + [P, P, P, P, P, P, P, P, P, F] + [P] * 8 + [P, I] + [I, I, I, P],
    "alm_hc_post_fwd": [P, P, P, P, P, P, I, I, I, P],
    "alm_hc_post_bwd": [P, P, P, P, P, P, P, P, P, P, I, I, I, P],
    "alm_geglu_ln_fwd": [P, L, I, P, P, L, P, I, I, I, P],
    "alm_geglu_ln_bwd": [P, L, I, P, P, P, L, P, P, I, I, I, P],
    "alm_ce_fwd_bwd": [P, L, P, L, P, P, L, P, P, I, I, I, P],
    "alm_axpby_bf16": [P, L, F, P, L, F, P, L, L, I, P],
    "alm_cast_pad_bf16": [P, L, P, L, L, I, I, P],
    "alm_cast_pad_multi": [P, I, P],
    "alm_scale_by_scalar_bf16": [P, P, L, P],
    "alm_topk_gumbel_sample": [P, L, P, L, P, I, I, I, F, P],
    "alm_resid_ln_fwd": [P, P, P, P, P, P, P, I, I, P],
    "alm_resid_ln_bwd": [P, P, P, P, P, P, P, P, P, F, I, I, P],
    "alm_residual_unit_fwd": [P, P, P, P, P, P, I, I, I, I, I, P],
    "alm_causal_conv1d_fwd": [P, P, P, P, P, I, I, I, I, I, I, I, I, I, I, P],
    "alm_causal_convT1d_fwd": [P, P, P, P, I, I, I, I, I, P],
    "alm_codec_first_conv": [P, P, P, P, I, I, I, I, I, P],
    "alm_codec_ru_tc": [P, P, P, P, P, I, I, I, I, I, I, P],
    "alm_codec_conv_tc": [P, P, P, P, I, I, I, I, I, I, I, I, I, I, P],
    "alm_codec_pack_c8s": [P, P, I, I, I, P],
    "alm_codec_last_conv": [P, P, P, P, I, I, I, I, I, P],
    "alm_rvq_encode": [P, L, P, P, P, L, P, L, I, I, I, I, P],
    "alm_rvq_pack_codebooks": [P, P, P, L, I, P],
    "alm_rvq_prepare": [P, L, P, P, L, P, I, I, P],
    "alm_rvq_select": [P, L, P, P, P, P, L, P, P, L, I, I, I, I, P],
    "alm_rvq_decode": [P, L, P, P, L, I, I, I, I, P],
}


class AlmError(RuntimeError):
    pass


_lib = None


def load() -> C.CDLL:
    """Load the shared library (building is explicit: `python -m audiolm_pytorch_b200.build`)."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise AlmError(
            f"{LIB_PATH} not found. Build it with `python -m audiolm_pytorch_b200.build` "
            "(there is no CPU / PyTorch fallback for the hot path)."
        )
    lib = C.CDLL(str(LIB_PATH), mode=os.RTLD_LOCAL | os.RTLD_NOW)
    lib.alm_version.restype = I
    lib.alm_status_string.restype = C.c_char_p
    lib.alm_status_string.argtypes = [I]
    lib.alm_launch_count.restype = C.c_ulonglong
    lib.alm_reset_launch_count.restype = None
    lib.alm_decode_stack_scratch_bytes.restype = L
    lib.alm_decode_stack_scratch_bytes.argtypes = [I, I, I, I]
    lib.alm_gemm_head_ce_tiles.restype = I
    lib.alm_gemm_head_ce_tiles.argtypes = [I]
    lib.alm_decode_stack_grid.restype = I
    lib.alm_decode_stack_grid.argtypes = []
    lib.alm_decode_stack_trace_offset.restype = L
    lib.alm_decode_stack_trace_offset.argtypes = [I, I, I, I]
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = I
    _lib = lib
    return lib


def ptr(t) -> int | None:
    if t is None:
        return None
    return t.data_ptr()


def stream_handle() -> int:
    return torch.cuda.current_stream().cuda_stream


def call(name: str, *args) -> None:
    """Invoke `name(*args, current_stream)`; tensors are passed by address."""
    lib = load()
    conv = []
    for a in args:
        if isinstance(a, torch.Tensor):
            if not a.is_cuda:
                raise AlmError(f"{name}: got a {a.device} tensor; the hot path has no CPU implementation")
            conv.append(a.data_ptr())
        else:
            conv.append(a)
    rc = getattr(lib, name)(*conv, stream_handle())
    if rc != 0:
        raise AlmError(f"{name} failed: {lib.alm_status_string(rc).decode()} ({rc})")


def launch_count() -> int:
    return int(load().alm_launch_count())


def reset_launch_count() -> None:
    load().alm_reset_launch_count()
