"""ctypes binding of libegom2p_b200.so (the C ABI declared in include/egom2p_b200.h).

There is no CPU or eager-PyTorch fallback: if the shared library is missing or a call fails, this
raises. Build it with `python -m egom2p_b200.build` (or `__graft_entry__.build()`)."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libegom2p_b200.so")
MAX_MODS = 8

vp, i32, i64, f32 = C.c_void_p, C.c_int32, C.c_int64, C.c_float


class PlanDesc(C.Structure):
    _fields_ = [("n_mods", i32), ("batch", i32), ("budget", i32), ("is_decoder", i32), ("causal", i32), ("sep", i32),
                ("len", i32 * MAX_MODS), ("mod_id", i32 * MAX_MODS), ("mask", vp * MAX_MODS),
                ("attn_cnt", vp * MAX_MODS), ("ids", vp * MAX_MODS)]


class EmbedDesc(C.Structure):
    _fields_ = [("n_mods", i32), ("dim", i32), ("len", i32 * MAX_MODS), ("vocab", i32 * MAX_MODS),
                ("ids", vp * MAX_MODS), ("token_emb", vp * MAX_MODS), ("pos_emb", vp * MAX_MODS),
                ("mod_emb", vp * MAX_MODS)]


# name -> argtypes (return type int unless listed in _RESTYPES). Must mirror include/egom2p_b200.h exactly;
# tests/test_abi.py checks that every symbol declared in the header is exported and listed here.
SIGNATURES = {
    "egom2p_last_error": [],
    "egom2p_abi_version": [],
    "egom2p_launch_count": [],
    "egom2p_index_plan": [C.POINTER(PlanDesc), vp, vp, vp, vp, vp, vp, vp, vp, vp, vp],
    "egom2p_plan_rows": [vp, i64, C.POINTER(i32), i32, i64, vp, vp, vp],
    "egom2p_embed_gather_fwd": [C.POINTER(EmbedDesc), vp, vp, vp, vp, vp, i64, i32, vp, vp, vp],
    "egom2p_embed_gather_bwd": [C.POINTER(EmbedDesc), vp, vp, vp, vp, vp, vp, i64, i32, vp, vp, vp, vp],
    "egom2p_layernorm_fwd": [vp, vp, i64, i32, f32, vp, vp, vp, vp, vp],
    "egom2p_layernorm_bwd": [vp, vp, vp, vp, vp, vp, vp, i64, i32, vp, vp, vp, vp],
    "egom2p_layernorm_bias_fwd": [vp, vp, vp, i64, i32, f32, vp, vp, vp, vp, vp],
    "egom2p_layernorm_bias_bwd": [vp, vp, vp, vp, vp, vp, vp, i64, i32, vp, vp, vp, vp, vp],
    "egom2p_gemm_bf16": [vp, vp, i32, i32, i32, i64, i64, i32, i32, vp, vp, i64, vp, vp, i64, vp],
    "egom2p_gemm_swiglu_fwd": [vp, vp, i32, i32, i32, i64, i64, vp, i64, vp, i64, vp],
    "egom2p_gemm_swiglu_bwd": [vp, vp, vp, i32, i32, i32, i64, i64, i64, vp, i64, vp],
    "egom2p_gemm_gelu_fwd": [vp, vp, vp, i32, i32, i32, i64, i64, vp, i64, vp, i64, vp],
    "egom2p_gemm_gelu_bwd": [vp, vp, vp, i32, i32, i32, i64, i64, i64, vp, i64, vp],
    "egom2p_ce_partials": [vp, vp, vp, i32, i32, i32, i64, i64, vp, vp, vp, vp],
    "egom2p_ce_finalize": [vp, vp, vp, i32, i32, vp, vp, vp],
    "egom2p_ce_dlogits": [vp, vp, vp, vp, vp, i32, i32, i32, i32, i64, i64, vp, i64, vp],
    "egom2p_attn_lse_stride": [i32],
    "egom2p_attn_ranges_bytes": [i32, i32],
    "egom2p_attn_ranges": [vp, vp, i32, i32, i32, f32, i32, vp, vp],
    "egom2p_attn_fwd": [vp, vp, vp, i32, i32, i32, i32, i64, i64, i64, vp, vp, i64, vp, vp, vp],
    "egom2p_attn_bwd_scratch_bytes": [i32, i32, i32],
    "egom2p_attn_bwd": [vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i64, i64, i64, i64, vp, f32, vp, vp, vp, vp,
                        i64, i64, i64, vp],
    "egom2p_cast_f32_to_bf16": [vp, vp, i64, vp],
    "egom2p_cast_f32_to_bf16_multi": [vp, i32, i64, vp],
    "egom2p_add_f32": [vp, vp, i64, vp, vp, vp],
    "egom2p_sumsq_multi": [vp, i32, i64, vp, vp, vp],
    "egom2p_adamw_multi_steps": [vp, i32, i64, f32, f32, f32, vp, vp, f32, vp],
    "egom2p_image_masks": [vp, C.c_uint64, C.c_uint64, i32, i32, i32, vp, vp, vp, vp, vp, vp],
    "egom2p_sample_rows": [vp, i64, i32, i32, f32, f32, i32, vp, vp, vp, vp, vp],
    "egom2p_cfg_combine_bf16": [vp, vp, i64, f32, vp, vp],
    "egom2p_colsum_f32": [vp, i64, i32, vp, vp],
    "egom2p_colsum_bf16": [vp, i64, i32, i64, vp, vp],
    "egom2p_gather_rows_bf16": [vp, vp, i64, i32, vp, vp],
    "egom2p_scatter_rows_f32": [vp, vp, i64, i32, vp, vp],
}
_RESTYPES = {"egom2p_last_error": C.c_char_p, "egom2p_launch_count": i64, "egom2p_attn_bwd_scratch_bytes": i64, "egom2p_attn_ranges_bytes": i64}

_lib = None


def load() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} not found: the CUDA library is mandatory (no fallback path). "
                               "Run `python -m egom2p_b200.build`.")
        lib = C.CDLL(LIB_PATH)
        for name, args in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.argtypes = args
            fn.restype = _RESTYPES.get(name, C.c_int)
        _lib = lib
    return _lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load().egom2p_last_error()
        raise RuntimeError(f"egom2p_b200 {what} failed (code {rc}): {msg.decode() if msg else '?'}")


def launch_count() -> int:
    return int(load().egom2p_launch_count())
