"""ctypes binding of libomniserve_b200.so (the C ABI in include/omniserve_b200.h).

There is no fallback: if the library is missing or a call fails this module raises.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("OB_LIB_PATH") or os.path.join(_HERE, "lib", "libomniserve_b200.so")   # override: instrumented builds

_lib = None

c_p = C.c_void_p
c_i = C.c_int
c_f = C.c_float
c_ll = C.c_longlong


class KV4DecodeArgs(C.Structure):
    _fields_ = [
        ("q", c_p), ("k", c_p), ("v", c_p),
        ("q_batch_stride", c_ll), ("k_batch_stride", c_ll), ("v_batch_stride", c_ll),
        ("out", c_p),
        ("retrieval_kv_pointers", c_p), ("streaming_kv_pointers", c_p),
        ("r_max_pages", c_i), ("s_max_pages", c_i),
        ("length_per_sample", c_p), ("retrieval_head_flags", c_p), ("head_rank_table", c_p),
        ("dynamic_sparse_page_idxes", c_p), ("num_dynamic_sparse_pages", c_i),
        ("batch", c_i), ("num_heads", c_i), ("num_kv_heads", c_i), ("head_dim", c_i), ("tokens_per_block", c_i),
        ("num_retrieval_kv_heads", c_i), ("num_streaming_kv_heads", c_i),
        ("sink_token_num", c_i), ("local_token_num", c_i), ("sink_block_num", c_i), ("local_block_num", c_i),
        ("timestep", c_i),
        ("rotary_embedding_dim", c_i), ("rotary_base", c_f), ("rotary_scale", c_f),
        ("force_split", c_i),
        ("tokens_per_sub_chunk", c_i), ("hidden_dim_per_retrieval_token", c_i),
        ("quant_out", c_p), ("quant_scale", c_p), ("quant_sum", c_p),
        ("history_is_stable", c_i),
        ("kv_scale_quant_orig", c_p), ("kv_scale_orig_quant", c_p),
    ]


class KV4PrefillArgs(C.Structure):
    _fields_ = [
        ("qkv", c_p), ("seq_lens", c_p), ("padding_offset", c_p), ("max_seq_len", c_i),
        ("retrieval_kv_pointers", c_p), ("streaming_kv_pointers", c_p),
        ("r_max_pages", c_i), ("s_max_pages", c_i),
        ("retrieval_head_flags", c_p), ("head_rank_table", c_p),
        ("num_tokens", c_i), ("batch", c_i), ("num_heads", c_i), ("num_kv_heads", c_i),
        ("num_retrieval_kv_heads", c_i), ("num_streaming_kv_heads", c_i),
        ("sink_token_num", c_i), ("local_token_num", c_i), ("sink_block_num", c_i), ("local_block_num", c_i),
        ("rotary_embedding_dim", c_i), ("rotary_base", c_f), ("rotary_scale", c_f),
        ("kv_scale_orig_quant", c_p),
    ]


class PeerCtx(C.Structure):
    _fields_ = [("bufs", c_p * 8), ("flags", c_p * 8), ("epoch", c_p), ("world", c_i), ("rank", c_i), ("max_blocks", c_i)]


class PageSelectorArgs(C.Structure):
    _fields_ = [
        ("q", c_p), ("q_batch_stride", c_ll), ("out", c_p),
        ("retrieval_kv_pointers", c_p), ("r_max_pages", c_i),
        ("length_per_sample", c_p), ("retrieval_head_flags", c_p), ("head_rank_table", c_p),
        ("batch", c_i), ("num_heads", c_i), ("num_kv_heads", c_i), ("head_dim", c_i), ("tokens_per_block", c_i),
        ("size_per_retrieval_token", c_i), ("num_retrieval_kv_heads", c_i),
        ("timestep", c_i),
        ("rotary_embedding_dim", c_i), ("rotary_base", c_f), ("rotary_scale", c_f),
        ("tokens_per_sub_chunk", c_i), ("hidden_dim_per_retrieval_token", c_i),
    ]


class StreamingPrefillArgs(C.Structure):
    _fields_ = [
        ("q", c_p), ("k", c_p), ("v", c_p),
        ("q_row_stride", c_ll), ("k_row_stride", c_ll), ("v_row_stride", c_ll),
        ("out", c_p), ("cu_seqlens", c_p),
        ("batch", c_i), ("num_tokens", c_i), ("num_heads", c_i), ("num_kv_heads", c_i), ("head_dim", c_i),
        ("num_compute_kv_heads", c_i),
        ("kv_heads", c_p), ("sink", c_p), ("local", c_p),
    ]


_SIGS = {
    "ob_version": ([], c_i),
    "ob_error_string": ([c_i], C.c_char_p),
    "ob_w4a8_gemm_per_chn": ([c_p] * 7 + [c_i] * 4 + [c_p], c_i),
    "ob_w4a8_gemm_per_group": ([c_p] * 7 + [c_i] * 4 + [c_p], c_i),
    "ob_w4a8_moe_gemm": ([c_p] * 8 + [c_i] * 5 + [c_p], c_i),
    "ob_w8a8_gemm": ([c_p] * 5 + [c_i] * 4 + [c_p], c_i),
    "ob_w4a8_gemm_ex": ([c_i] + [c_p] * 9 + [c_i] * 7 + [c_p], c_i),
    "ob_debug_w4a8_decode_plan": ([c_i] * 6 + [c_p] * 4, c_i),
    "ob_w4a8_gemm_add_norm_quant": ([c_i] + [c_p] * 9 + [c_i] * 4 + [c_p] * 6 + [c_f] + [c_p], c_i),
    "ob_invoke_quant": ([c_p] * 3 + [c_i] * 2 + [c_p], c_i),
    "ob_invoke_quant_fuse_sum": ([c_p] * 4 + [c_i] * 2 + [c_p], c_i),
    "ob_rms_norm": ([c_p] * 3 + [c_f] + [c_i] * 2 + [c_p], c_i),
    "ob_rms_norm_general": ([c_p] * 4 + [c_f] + [c_i] * 2 + [c_p], c_i),
    "ob_rms_norm_general_fuse_sum": ([c_p] * 5 + [c_f] + [c_i] * 2 + [c_p], c_i),
    "ob_add_rms_norm_general": ([c_p] * 7 + [c_f] + [c_i] * 2 + [c_p], c_i),
    "ob_add_rms_norm": ([c_p] * 4 + [c_f] + [c_i] * 2 + [c_p], c_i),
    "ob_peer_add_rms_norm_general": ([c_p] * 2 + [C.POINTER(PeerCtx)] + [c_p] * 4 + [c_f] + [c_i] * 2 + [c_p], c_i),
    "ob_peer_add_rms_norm": ([c_p] * 2 + [C.POINTER(PeerCtx)] + [c_p] + [c_f] + [c_i] * 2 + [c_p], c_i),
    "ob_silu_and_mul": ([c_p] * 2 + [c_i] * 2 + [c_p], c_i),
    "ob_silu_and_mul_quant": ([c_p] * 4 + [c_i] * 2 + [c_p], c_i),
    "ob_add_f16": ([c_p] * 3 + [c_ll] + [c_p], c_i),
    "ob_kv4_single_query_attention": ([C.POINTER(KV4DecodeArgs), c_p], c_i),
    "ob_kv4_apply_rope_update_kv_cache": ([C.POINTER(KV4PrefillArgs), c_p], c_i),
    "ob_kv4_apply_rope_update_kv_cache_pool": ([C.POINTER(KV4PrefillArgs), c_i, c_p], c_i),
    "ob_compute_padding_offsets": ([c_p] * 2 + [c_i] * 2 + [c_p], c_i),
    "ob_paged_min_max_pool": ([c_p] * 4 + [c_ll] * 2 + [c_i] * 9 + [c_p], c_i),
    "ob_kv4_page_topk": ([c_p] * 2 + [c_i] * 5 + [c_p], c_i),
    "ob_kv4_page_selector": ([C.POINTER(PageSelectorArgs), c_p], c_i),
    "ob_token_streaming_prefill_attention": ([C.POINTER(StreamingPrefillArgs), c_p], c_i),
    "ob_debug_streaming_prefill_plan": ([C.POINTER(StreamingPrefillArgs)] + [c_i] * 3 + [c_p] * 2 + [c_i], c_i),
    "ob_moe_router_logits": ([c_p] * 3 + [c_i] * 3 + [c_p], c_i),
    "ob_moe_topk_sort": ([c_p] * 5 + [c_i] * 3 + [c_p], c_i),
    "ob_moe_expand": ([c_p] * 8 + [c_i] * 3 + [c_p], c_i),
    "ob_moe_finalize": ([c_p] * 4 + [c_i] * 4 + [c_p], c_i),
    "ob_w4a8_moe_gemm_dev": ([c_p] * 8 + [c_i] * 5 + [c_p], c_i),
    "ob_debug_moe_device_plan": ([c_i] * 4 + [c_p, c_i] + [c_p] * 3 + [c_i], c_i),
}
EXPORTS = tuple(_SIGS)


def lib():
    """Load the shared library once.  Raises RuntimeError when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} not found: build it with `python -m omniserve_b200.build` "
                "(there is no CPU / PyTorch fallback for these ops)"
            )
        l = C.CDLL(LIB_PATH)
        for name, (argt, rest) in _SIGS.items():
            fn = getattr(l, name)
            fn.argtypes = argt
            fn.restype = rest
        _lib = l
    return _lib


def check(code: int, what: str):
    if code != 0:
        raise RuntimeError(f"omniserve_b200: {what} failed: {lib().ob_error_string(code).decode()} (code {code})")


def stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def ptr(t):
    return 0 if t is None else t.data_ptr()


def require_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("omniserve_b200 ops need CUDA tensors (no CPU fallback)")


def require_contiguous(*ts):
    """The C ABI takes raw base pointers and dense row pitches: reject strided views instead of reading past them."""
    for t in ts:
        if t is not None and not t.is_contiguous():
            raise RuntimeError("omniserve_b200: this op needs contiguous tensors (got a strided view)")
