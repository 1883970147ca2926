"""ctypes binding of libabcgpt.so (C ABI declared in include/abcgpt.h).

The product path has no CPU or PyTorch fallback: if the shared object is missing (or a call fails) the ops
raise.  `lib()` loads lazily so that host-only code (config, checkpoint I/O, CPU tests of the host logic) can
import the package on a machine without the built extension.
"""
from __future__ import annotations

import ctypes
import os
import re
from ctypes import c_char_p, c_float, c_int, c_int64, c_uint32, c_void_p

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libabcgpt.so")
DEBUG_LIB_PATH = os.path.join(HERE, "libabcgpt_debug.so")
HEADER_PATH = os.path.join(os.path.dirname(HERE), "include", "abcgpt.h")
DEBUG_HEADER_PATH = os.path.join(os.path.dirname(HERE), "include", "abcgpt_debug.h")

EPI_BF16, EPI_GELU, EPI_RESID, EPI_DGELU, EPI_F32_RED, EPI_F32 = range(6)
FN_IDS = {"abcgpt_gemm_bf16": 1, "abcgpt_embed_fwd": 2, "abcgpt_layernorm_fwd": 3, "abcgpt_attn_decode": 4, "abcgpt_argmax": 5,
          "abcgpt_sample_topk": 6, "abcgpt_attn_decode_hd": 7, "abcgpt_sample_top_p": 8}
ACT_TANH = 0x100  # OR-ed into EPI_GELU / EPI_DGELU: tanh form of GELU (include/abcgpt.h ABCGPT_ACT_TANH)

_P = c_void_p
_SIGNATURES = {
    "abcgpt_version": (c_int, []),
    "abcgpt_last_error": (c_char_p, []),
    "abcgpt_gemm_bf16": (c_int, [_P, c_int, c_int64, _P, c_int, c_int64, c_int, c_int, c_int, c_int, _P, c_int64, _P,
                                 c_int64, _P, c_int64, _P, c_int, c_int, c_float, c_uint32, _P]),
    "abcgpt_embed_fwd": (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, c_int, c_float, c_uint32, _P]),
    "abcgpt_embed_bwd": (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, c_int, c_float, c_uint32, _P]),
    "abcgpt_add_pos": (c_int, [_P, _P, _P, c_int, c_int, c_int, _P]),
    "abcgpt_set_first_pos": (c_int, [_P, _P, _P, c_int, c_int, c_int, _P]),
    "abcgpt_pos_bwd": (c_int, [_P, _P, c_int, c_int, c_int, _P]),
    "abcgpt_onehot_bf16": (c_int, [_P, _P, c_int, c_int, c_int, _P]),
    "abcgpt_layernorm_fwd": (c_int, [_P, _P, _P, _P, _P, _P, _P, c_int, c_int, _P]),
    "abcgpt_layernorm_fwd_resid": (c_int, [_P, _P, _P, _P, _P, _P, _P, _P, c_int, c_int, c_float, c_uint32, _P]),
    "abcgpt_layernorm_bwd": (c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, c_int, c_int, c_float, c_uint32, _P]),
    "abcgpt_attn_fwd": (c_int, [_P, _P, _P, c_int, c_int, c_int, c_float, c_uint32, _P]),
    "abcgpt_attn_bwd": (c_int, [_P, _P, _P, _P, _P, _P, c_int, c_int, c_int, c_float, c_uint32, _P]),
    "abcgpt_attn_fwd_hd": (c_int, [_P, _P, _P, c_int, c_int, c_int, c_int, c_float, c_uint32, _P]),
    "abcgpt_attn_bwd_hd": (c_int, [_P, _P, _P, _P, _P, _P, c_int, c_int, c_int, c_int, c_float, c_uint32, _P]),
    "abcgpt_ce_fwd": (c_int, [_P, c_int64, _P, _P, c_int, c_int, _P]),
    "abcgpt_ce_finalize": (c_int, [_P, _P, c_int, _P, _P, _P]),
    "abcgpt_ce_bwd": (c_int, [_P, c_int64, _P, _P, _P, _P, c_int, c_int, _P]),
    "abcgpt_sumsq": (c_int, [_P, c_int64, _P, _P, _P]),
    "abcgpt_adamw": (c_int, [_P, _P, _P, _P, _P, c_int64, c_float, c_float, c_float, c_float, c_float, c_int, _P,
                             c_float, _P]),
    "abcgpt_cast_f32_to_bf16": (c_int, [_P, _P, c_int64, _P]),
    "abcgpt_attn_decode": (c_int, [_P, _P, c_int, c_int, c_int, c_int, _P]),
    "abcgpt_attn_decode_hd": (c_int, [_P, _P, _P, c_int, c_int, c_int, c_int, c_int, _P]),
    "abcgpt_sample_batch": (c_int, [_P, c_int, c_int64, _P, _P, _P, c_int, c_int, _P]),
    "abcgpt_colsum_bf16": (c_int, [_P, c_int64, c_int, c_int, _P, _P]),
    "abcgpt_replay": (c_int, [_P, c_int64, c_int64]),
    "abcgpt_set_pdl": (c_int, [c_int]),
    "abcgpt_event_record": (c_int, [c_int, _P]),
    "abcgpt_event_wait": (c_int, [c_int, _P]),
    "abcgpt_nvls_allreduce_sumsq": (c_int, [_P, c_int64, c_int, c_int, c_float, _P, c_int, c_int, _P]),
    "abcgpt_sumsq_partials": (c_int, [_P, c_int, _P, _P]),
    "abcgpt_set_dynamic_tiles": (c_int, [c_int]),
    "abcgpt_argmax": (c_int, [_P, c_int64, c_int, _P, c_int64, c_int, _P]),
    "abcgpt_sample_topk": (c_int, [_P, c_int64, c_int, c_float, c_int, _P, c_int64, _P, c_int64, c_int, _P]),
    "abcgpt_sample_top_p": (c_int, [_P, c_int64, c_int, c_float, c_int, c_float, _P, _P, c_int64, _P, _P, c_int64, c_int, _P]),
}
# include/abcgpt_debug.h: only in libabcgpt_debug.so (tools/)
_DEBUG_SIGNATURES = {
    "abcgpt_debug_gemm_stats": (c_int, [_P]),
    "abcgpt_debug_attn_trace": (c_int, [_P]),
    "abcgpt_debug_attn_cta_trace": (c_int, [_P]),
    "abcgpt_debug_mma_bench": (c_int, [_P, c_int, c_int, c_int, _P]),
    "abcgpt_debug_tmem_ld_bench": (c_int, [_P, c_int, c_int, c_int, _P]),
    "abcgpt_debug_pair_probe": (c_int, [_P, _P, _P, c_int, _P]),
    "abcgpt_debug_mufu_bench": (c_int, [_P, _P, c_int, c_int, c_int, _P]),
    "abcgpt_debug_mufu2_bench": (c_int, [_P, _P, c_int, c_int, c_int, _P]),
    "abcgpt_debug_tmem_mma_bench": (c_int, [_P, c_int, c_int, c_int, c_int, c_int, c_int, _P]),
}

_lib = None
_use_debug = False


class AbcgptError(RuntimeError):
    pass


def declared_symbols(debug: bool = False) -> list[str]:
    """Every function include/abcgpt.h (debug: include/abcgpt_debug.h) declares (used by the CPU-side ABI test)."""
    with open(DEBUG_HEADER_PATH if debug else HEADER_PATH) as f:
        text = f.read()
    return sorted(set(re.findall(r"\b(abcgpt_[a-z0-9_]+)\s*\(", text)))


def use_debug_lib() -> None:
    """tools/ only: route every call of this process through libabcgpt_debug.so (product objects + the instrumentation entry
    points of include/abcgpt_debug.h; built on demand).  Must run before the first call into the library."""
    global _use_debug
    if _lib is not None and not _use_debug:
        raise AbcgptError("use_debug_lib() must be called before the library is first used")
    from . import build as _build
    _build.build(debug=True)
    _use_debug = True


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        # ABCGPT_LIB: experiments only — load another build of the same ABI (A/B timing of two kernel variants on one box)
        path = os.environ.get("ABCGPT_LIB") or (DEBUG_LIB_PATH if _use_debug else LIB_PATH)
        if not os.path.exists(path):
            raise AbcgptError(
                f"{path} is missing: build it with `python -m ai_music_generation_b200.build` "
                "(there is no CPU/PyTorch fallback for the sm_100a kernels)")
        handle = ctypes.CDLL(path)
        sigs = {**_SIGNATURES, **_DEBUG_SIGNATURES} if _use_debug else _SIGNATURES
        for name, (res, args) in sigs.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = lib().abcgpt_last_error()
        raise AbcgptError(f"{what} failed (rc={rc}): {msg.decode() if msg else '?'}")
