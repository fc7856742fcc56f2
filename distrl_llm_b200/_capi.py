"""ctypes binding of libb200rl.so (include/b200rl.h): PyTorch tensors in, PyTorch tensors out.

This is the thin shim BASELINE.json's north_star asks for.  There is NO fallback: if the shared
library is missing or a call fails, a RuntimeError is raised (the product path never routes through
the oracle or a torch implementation).
"""
from __future__ import annotations

import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libb200rl.so")

c_void_p, c_int, c_ll, c_float, c_uint = C.c_void_p, C.c_int, C.c_longlong, C.c_float, C.c_uint


class ModelConfig(C.Structure):
    _fields_ = [
        ("vocab", c_int), ("hidden", c_int), ("inter", c_int), ("n_layers", c_int),
        ("n_q_heads", c_int), ("n_kv_heads", c_int), ("head_dim", c_int),
        ("lora_r", c_int), ("lora_scale", c_float), ("rms_eps", c_float), ("rope_theta", c_float),
        ("max_tokens", c_int), ("max_batch", c_int), ("max_seq", c_int), ("max_score_rows", c_int),
    ]


class LossArgs(C.Structure):
    _fields_ = [("nb", c_int), ("grpo", c_int), ("backward", c_int), ("lora_off", c_int),
                ("ref_lp", c_void_p), ("kl_beta", C.c_double), ("old_lp", c_void_p), ("clip_eps", C.c_double)]


class EntropyArgs(C.Structure):
    _fields_ = [("alpha", C.c_double), ("ent_out", c_void_p), ("ent_accum", c_void_p)]


class LayerWeights(C.Structure):
    _fields_ = [
        ("qkv_packed", c_void_p), ("qkv_absmax", c_void_p),
        ("o_packed", c_void_p), ("o_absmax", c_void_p),
        ("gu_packed", c_void_p), ("gu_absmax", c_void_p),
        ("down_packed", c_void_p), ("down_absmax", c_void_p),
        ("qkv_bias", c_void_p), ("ln1_w", c_void_p), ("ln2_w", c_void_p),
    ]


# name -> (restype, argtypes); mirrors include/b200rl.h one to one
SIGNATURES = {
    "b200rl_last_error": (C.c_char_p, []),
    "b200rl_version": (c_int, []),
    "b200rl_check_device": (c_int, []),
    "b200rl_gemm": (c_int, [c_void_p, c_ll, c_void_p, c_ll, c_int, c_void_p, c_ll, c_void_p, c_ll, c_int,
                            c_void_p, c_ll, c_int, c_void_p, c_void_p, c_ll, c_float, c_int, c_int,
                            c_int, c_int, c_ll, c_int, c_int, c_void_p]),
    "b200rl_gemm_set_cta_pair": (c_int, [c_int]),
    "b200rl_gemm_set_tail_split": (c_int, [c_int]),
    "b200rl_gemm_set_wide": (c_int, [c_int]),
    "b200rl_gemm_set_raster": (c_int, [c_int]),
    "b200rl_logprob_slots": (c_int, [c_void_p, c_ll, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, C.c_double, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "b200rl_gemm_set_ext": (c_int, [c_int]),
    "b200rl_gemm_nf4": (c_int, [c_void_p, c_ll, c_void_p, c_void_p, c_int, c_void_p, c_ll, c_void_p, c_ll, c_int, c_void_p, c_ll,
                                c_void_p, c_void_p, c_ll, c_int, c_int, c_int, c_int, c_void_p]),
    "b200rl_gemm_lora": (c_int, [c_void_p, c_ll, c_void_p, c_ll, c_int, c_void_p, c_ll, c_float, c_void_p, c_ll, c_void_p, c_ll,
                                 c_int, c_void_p, c_ll, c_void_p, c_void_p, c_ll, c_int, c_int, c_int, c_int, c_void_p]),
    "b200rl_gemm_dw_grouped": (c_int, [c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int,
                                       c_void_p]),
    "b200rl_gemm_swiglu": (c_int, [c_int, c_void_p, c_ll, c_void_p, c_ll, c_int, c_void_p, c_ll, c_void_p, c_ll, c_int,
                                   c_void_p, c_ll, c_void_p, c_ll, c_int, c_int, c_void_p]),
    "b200rl_embed": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "b200rl_rmsnorm_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_float, c_void_p]),
    "b200rl_rmsnorm_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "b200rl_rope_table": (c_int, [c_void_p, c_int, c_int, c_float, c_void_p]),
    "b200rl_rope": (c_int, [c_void_p, c_void_p, c_int, c_int, c_ll, c_int, c_int, c_int, c_void_p]),
    "b200rl_swiglu_fwd": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "b200rl_swiglu_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "b200rl_gather_rows": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "b200rl_scatter_rows": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "b200rl_attn_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_float, c_void_p]),
    "b200rl_attn_set_prof": (c_int, [c_void_p, c_int]),
    "b200rl_attn_set_tc": (c_int, [c_int]),
    "b200rl_attn_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                c_int, c_int, c_int, c_int, c_int, c_float, c_void_p]),
    "b200rl_attn_seg_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_ll, c_int, c_int, c_float, c_void_p, c_int, c_void_p]),
    "b200rl_attn_seg_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_ll,
                                    c_int, c_int, c_float, c_void_p, c_int, c_void_p, c_int, c_void_p, c_void_p, c_void_p]),
    "b200rl_logprob": (c_int, [c_void_p, c_ll, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "b200rl_loss_coef": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "b200rl_loss_value": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "b200rl_logprob_kl": (c_int, [c_void_p, c_ll, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "b200rl_loss_coef_kl": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, C.c_double, c_void_p, c_int, c_int, c_int, c_void_p]),
    "b200rl_loss_value_kl": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, C.c_double, c_void_p, c_int, c_int, c_int, c_void_p]),
    "b200rl_group_advantage_topk": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "b200rl_nf4_quantize": (c_int, [c_void_p, c_void_p, c_void_p, c_ll, c_void_p]),
    "b200rl_nf4_dequant": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "b200rl_lora_reduce_adamw": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_ll,
                                         c_int, c_float, c_float, c_float, c_float, c_float, c_int, c_void_p]),
    "b200rl_p2p_barrier": (c_int, [c_void_p, c_int, c_int, c_uint, c_void_p]),
    "b200rl_p2p_barrier_timeout": (c_int, [c_void_p, c_int, c_int, c_uint, C.c_double, c_void_p]),
    "b200rl_p2p_status": (c_int, [c_int]),
    "b200rl_p2p_alloc": (c_int, [c_ll, C.POINTER(c_void_p), c_void_p]),
    "b200rl_p2p_open": (c_int, [c_void_p, C.POINTER(c_void_p)]),
    "b200rl_p2p_close": (c_int, [c_void_p]),
    "b200rl_p2p_free": (c_int, [c_void_p]),
    "b200rl_p2p_enable_peer_access": (c_int, [c_int]),
    "b200rl_lora_pack": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "b200rl_lora_grad_accum": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "b200rl_sizeof_pack_desc": (c_int, []),
    "b200rl_sizeof_unpack_desc": (c_int, []),
    "b200rl_model_workspace_bytes": (c_ll, [C.POINTER(ModelConfig)]),
    "b200rl_model_lora_numel": (c_ll, [C.POINTER(ModelConfig)]),
    "b200rl_model_create": (c_int, [C.POINTER(ModelConfig), C.POINTER(LayerWeights), c_void_p, c_void_p, c_void_p,
                                    c_void_p, c_void_p, c_void_p, c_ll, C.POINTER(c_void_p)]),
    "b200rl_model_destroy": (c_int, [c_void_p]),
    "b200rl_model_weight_cache_bytes": (c_ll, [C.POINTER(ModelConfig)]),
    "b200rl_model_set_weight_cache": (c_int, [c_void_p, c_void_p, c_ll]),
    "b200rl_model_set_nf4_inkernel": (c_int, [c_void_p, c_int]),
    "b200rl_model_set_fusion": (c_int, [c_void_p, c_int]),
    "b200rl_model_sync_lora": (c_int, [c_void_p, c_void_p]),
    "b200rl_model_debug_ptr": (c_void_p, [c_void_p, C.c_char_p, c_int]),
    "b200rl_model_microbatch_ex": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                           c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, C.c_double, c_void_p]),
    "b200rl_model_microbatch_packed": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                                               c_void_p, C.c_double, c_void_p]),
    "b200rl_rope_pos": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_ll, c_int, c_int, c_int, c_void_p]),
    "b200rl_gather_rows_idx": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "b200rl_scatter_add_rows": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "b200rl_model_profile": (c_int, [c_void_p, c_int]),
    "b200rl_model_profile_read": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p]),
    "b200rl_launch_count": (c_ll, []),
    "b200rl_set_pdl": (c_int, [c_int]),
    "b200rl_logprob_clip": (c_int, [c_void_p, c_ll, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, C.c_double, c_void_p, c_int,
                                    c_int, c_int, c_void_p]),
    "b200rl_loss_value_clip": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, C.c_double, c_void_p, C.c_double, c_void_p, c_int,
                                       c_int, c_int, c_void_p]),
    "b200rl_model_pass": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int,
                                  c_void_p, c_void_p]),
    "b200rl_model_pass_packed": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "b200rl_logprob_entropy": (c_int, [c_void_p, c_ll, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, C.c_double, c_void_p,
                                       c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, C.c_double,
                                       c_void_p, c_void_p]),
    "b200rl_loss_value_entropy": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, C.c_double, c_void_p, C.c_double, c_void_p,
                                          c_int, c_int, c_int, c_void_p, C.c_double, c_void_p, c_void_p]),
    "b200rl_model_pass_ent": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int,
                                      c_int, c_void_p, c_void_p, c_void_p]),
    "b200rl_model_pass_packed_ent": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "b200rl_model_microbatch": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                        c_int, c_int, c_int, c_int, c_int, c_int, c_void_p]),
}

_lib = None


def load_library() -> C.CDLL:
    """Load libb200rl.so and attach the signatures. Raises if the library was not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python __graft_entry__.py` (nvcc, sm_100a). "
            "distrl_llm_b200 has no CPU or torch fallback."
        )
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def lib() -> C.CDLL:
    return load_library()


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load_library().b200rl_last_error().decode(errors="replace")
        raise RuntimeError(f"libb200rl {what} failed (code {rc}): {msg}")


def ptr(t) -> int | None:
    """Device pointer of a tensor (None -> NULL)."""
    if t is None:
        return None
    return t.data_ptr()


def stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and (not t.is_cuda or not t.is_contiguous()):
            raise RuntimeError("libb200rl needs contiguous CUDA tensors")
