"""ctypes binding of the C ABI in include/sgpt_b200.h (libsgpt_b200.so, built in-tree by __graft_entry__.build()).

There is no fallback: if the library is missing or a call fails, a RuntimeError is raised.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

_HERE = os.path.dirname(os.path.abspath(__file__))
# SGPT_B200_LIB: explicit path of another build of the SAME library (A/B measurements of two builds on one GPU box); it is
# subject to the same symbol and ABI-version checks — there is still no fallback of any kind
LIB_PATH = os.environ.get("SGPT_B200_LIB") or os.path.join(_HERE, "libsgpt_b200.so")

SGPT_OK = 0
EPI_BF16, EPI_GELU_BF16, EPI_RESID_F32, EPI_RESID_BF16 = 0, 1, 2, 3
POOL_MEAN, POOL_WEIGHTEDMEAN, POOL_LASTTOKEN, POOL_MEANMEAN, POOL_LASTTOKENMEAN = 0, 1, 2, 3, 4
ARCH_GPT_NEO, ARCH_GPTJ, ARCH_BLOOM = 0, 1, 2
ACT_IDENTITY, ACT_TANH, ACT_RELU, ACT_SIGMOID = 0, 1, 2, 3
ELEM_BF16, ELEM_I8 = 0, 1  # element type of a corpus shard (SGPT_ELEM_*)

i32, i64, f32, vp = C.c_int32, C.c_int64, C.c_float, C.c_void_p


class ModelConfigC(C.Structure):
    _fields_ = [("arch", i32), ("n_layer", i32), ("d_model", i32), ("n_head", i32), ("d_ff", i32), ("vocab", i32),
                ("max_pos", i32), ("window", i32), ("rotary_dim", i32), ("ln_eps", f32), ("max_tokens", i32),
                ("max_batch", i32)]


class LayerWeightsC(C.Structure):
    _fields_ = [("ln1_g", vp), ("ln1_b", vp), ("w_qkv", vp), ("b_qkv", vp), ("w_o", vp), ("b_o", vp), ("ln2_g", vp),
                ("ln2_b", vp), ("w_fc", vp), ("b_fc", vp), ("w_proj", vp), ("b_proj", vp), ("local_attention", i32),
                ("_pad", i32)]


class ModelWeightsC(C.Structure):
    _fields_ = [("wte", vp), ("wpe", vp), ("lnf_g", vp), ("lnf_b", vp), ("layers", C.POINTER(LayerWeightsC)),
                ("emb_ln_g", vp), ("emb_ln_b", vp)]


_SIGNATURES = {
    "sgpt_abi_version": (i32, []),
    "sgpt_last_error": (C.c_char_p, []),
    "sgpt_embed_tokens": (i32, [vp, vp, vp, vp, vp, i32, i32, i32, i32, vp]),
    "sgpt_layernorm": (i32, [vp, vp, vp, vp, i32, i32, f32, vp]),
    "sgpt_layernorm_f32_inplace": (i32, [vp, vp, vp, i32, i32, f32, vp]),
    "sgpt_linear_qkv_rotary": (i32, [vp, i64, vp, vp, vp, vp, i32, i32, i32, i32, i32, vp]),
    "sgpt_linear": (i32, [vp, i64, vp, i64, vp, vp, i64, vp, i32, i32, i32, i32, vp]),
    "sgpt_attention": (i32, [vp, vp, vp, i32, i32, i32, i32, f32, i32, i32, vp, i32, vp]),
    "sgpt_pool": (i32, [vp, vp, vp, vp, vp, f32, vp, vp, i32, i32, i32, i32, i32, i32, vp]),
    "sgpt_pool_accumulate": (i32, [vp, vp, vp, vp, vp, f32, vp, vp, i32, i32, i32, i32, i32, i32, i32, f32, vp]),
    "sgpt_pool_ex": (i32, [vp, vp, vp, vp, vp, f32, vp, i32, vp, vp, i32, i32, i32, i32, i32, i32, i32, f32, vp]),
    "sgpt_normalize_rows": (i32, [vp, i32, i32, vp]),
    "sgpt_dense": (i32, [vp, vp, vp, vp, i32, i32, i32, i32, vp]),
    "sgpt_model_set_position_weights": (i32, [vp, vp, i32]),
    "sgpt_layernorm_gather": (i32, [vp, vp, vp, vp, vp, i32, i32, f32, vp]),
    "sgpt_forward": (i32, [vp, vp, vp, vp, i32, i32, i32, vp]),
    "sgpt_lm_logprobs_workspace_bytes": (i64, [i32, i32, i32]),
    "sgpt_lm_logprobs": (i32, [vp, vp, vp, i32, vp, vp, i32, vp, vp, vp, i64, i32, vp]),
    "sgpt_token_logprobs": (i32, [vp, i64, i32, i32, vp, vp, vp, vp, vp]),
    "sgpt_segment_sum": (i32, [vp, vp, i32, vp, vp]),
    "sgpt_model_create": (i32, [C.POINTER(ModelConfigC), C.POINTER(ModelWeightsC), C.POINTER(vp)]),
    "sgpt_model_destroy": (None, [vp]),
    "sgpt_encode": (i32, [vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, i32, vp, vp]),
    "sgpt_model_read_residual": (i32, [vp, vp, i64, C.POINTER(i32), C.POINTER(i32), vp]),
    "sgpt_row_inv_norms": (i32, [vp, vp, i64, i32, vp]),
    "sgpt_f32_to_bf16": (i32, [vp, vp, i64, vp]),
    "sgpt_scores": (i32, [vp, vp, vp, vp, vp, i64, i32, i64, i32, vp]),
    "sgpt_topk_workspace_bytes": (i64, [i32, i64, i32]),
    "sgpt_topk": (i32, [vp, i64, i32, i64, i32, i64, vp, vp, vp, vp]),
    "sgpt_topk_merge": (i32, [vp, vp, i32, i32, i32, vp, vp, vp, vp, vp]),
    "sgpt_search_workspace_bytes": (i64, [i32, i64, i32]),
    "sgpt_profile_enable": (i32, [i32]),
    "sgpt_profile_read": (i32, [vp, vp, vp]),
    "sgpt_profile_gemm_clock": (i32, [vp, vp]),
    "sgpt_debug_topk_timeline": (i32, [vp, i32]),
    "sgpt_search": (i32, [vp, vp, vp, vp, i32, i64, i32, i32, i64, vp, vp, vp, i64, vp]),
    "sgpt_embed_tokens_ex": (i32, [vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, vp]),
    "sgpt_layernorm_ex": (i32, [vp, i32, vp, vp, vp, i32, i32, f32, vp]),
    "sgpt_layernorm_gather_ex": (i32, [vp, i32, vp, vp, vp, vp, i32, i32, f32, vp]),
    "sgpt_pool_ex2": (i32, [vp, i32, vp, vp, vp, vp, f32, vp, i32, vp, vp, i32, i32, i32, i32, i32, i32, i32, f32, vp]),
    "sgpt_bf16_to_f32": (i32, [vp, vp, i64, vp]),
    "sgpt_fold_layernorm": (i32, [vp, vp, vp, vp, vp, vp, vp, i32, i32, vp]),
    "sgpt_resid_stats": (i32, [vp, vp, vp, i32, i32, vp]),
    "sgpt_linear_lnfold": (i32, [vp, i64, vp, i64, vp, vp, vp, i32, f32, vp, i64, i32, i32, i32, i32, vp]),
    "sgpt_linear_qkv_rotary_lnfold": (i32, [vp, i64, vp, vp, vp, vp, i32, f32, vp, vp, vp, i32, i32, i32, i32, i32, vp]),
    "sgpt_linear_resid_ln": (i32, [vp, i64, vp, i64, vp, vp, vp, vp, i32, i32, i32, vp]),
    "sgpt_pool_partials": (i32, [vp, vp, vp, vp, vp, f32, vp, i32, vp, vp, i32, vp, i32, i32, i32, i32, i32, i32, i32, f32, vp]),
    "sgpt_search_packed": (i32, [vp, vp, vp, vp, i32, i64, i32, i32, i64, vp, vp, i64, vp]),
    "sgpt_topk_merge_packed": (i32, [vp, i32, i32, i32, vp, vp, vp, vp]),
    "sgpt_gather_create": (i32, [i32, i32, i32, i32, C.POINTER(vp), vp]),
    "sgpt_gather_connect": (i32, [vp, vp]),
    "sgpt_gather_destroy": (None, [vp]),
    "sgpt_search_gather": (i32, [vp, vp, vp, vp, vp, i32, i64, i32, i32, i64, vp, vp, vp, vp, i64, vp]),
    "sgpt_quantize_rows_i8": (i32, [vp, i32, i64, i32, vp, vp, vp, vp]),
    "sgpt_search_ex": (i32, [vp, vp, vp, vp, i32, i64, i32, i32, i64, vp, vp, vp, i64, i32, vp]),
    "sgpt_search_packed_ex": (i32, [vp, vp, vp, vp, i32, i64, i32, i32, i64, vp, vp, i64, i32, vp]),
    "sgpt_search_gather_ex": (i32, [vp, vp, vp, vp, vp, i32, i64, i32, i32, i64, vp, vp, vp, vp, i64, i32, vp]),
}

ABI_VERSION = 3  # include/sgpt_b200.h SGPT_ABI_VERSION these signatures / struct layouts were written for
IPC_HANDLE_BYTES = 64

_lib: Optional[C.CDLL] = None


def exported_symbols():
    """Every symbol include/sgpt_b200.h declares (used by the CPU test that the library exports all of them)."""
    return sorted(_SIGNATURES)


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} not found: build the CUDA library first (python -c 'import __graft_entry__ as g; g.build()' "
                "or make -C sgpt_b200/csrc). sgpt_b200 has no CPU or PyTorch fallback.")
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(handle, name)  # AttributeError here means the .so is stale: fail loudly
            fn.restype = res
            fn.argtypes = args
        got = handle.sgpt_abi_version()
        if got != ABI_VERSION:  # a stale .so would take these argument lists / struct layouts and corrupt them silently
            raise RuntimeError(f"{LIB_PATH} has ABI version {got}, the Python binding expects {ABI_VERSION}: rebuild "
                               "(python -c 'import __graft_entry__ as g; g.build()')")
        _lib = handle
    return _lib


def check(rc: int, what: str = "") -> None:
    if rc != SGPT_OK:
        msg = lib().sgpt_last_error()
        raise RuntimeError(f"{what or 'sgpt call'} failed (code {rc}): {msg.decode() if msg else '?'}")


def ptr(t) -> Optional[int]:
    """Device (or host) address of a torch tensor; None -> NULL."""
    return None if t is None else t.data_ptr()


def current_stream() -> int:
    import torch

    return torch.cuda.current_stream().cuda_stream
