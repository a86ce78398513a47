"""Grouped W4A8 per-channel GEMM for mixture-of-experts layers -- the op the reference names but never released
(omniserve/modeling/layers/quantized_linear/w4a8_moe_linear.py:83-94: `mygemm.moe_gemm_forward_cuda_api(x, self.qweight,
self.s1_scales, input_scales, self.s1_szeros, input_sum, problem_sizes)`, forward raises NotImplementedError upstream).
Same argument order; returns the output buffer like the commented-out reference call."""
import ctypes as C

import torch

from .. import _lib as L


def moe_gemm_forward_cuda_api(x, qweight, s1_scales, input_scales, s1_szeros, input_sum, problem_sizes, out=None):
    """x int8 [T, K], rows sorted by expert; qweight int8 [E, N, K/2]; s1_scales / s1_szeros fp16 [E, N]; input_scales /
    input_sum fp16 [T]; problem_sizes: rows per expert (sequence of ints, or an int tensor -- a CUDA tensor is read back to
    the host, which synchronises).  Returns fp16 [T, N]."""
    L.require_cuda(x, qweight, s1_scales, input_scales, s1_szeros, input_sum)
    L.require_contiguous(x, qweight, s1_scales, input_scales, s1_szeros, input_sum)
    sizes = problem_sizes.tolist() if torch.is_tensor(problem_sizes) else list(problem_sizes)
    E, N, K2 = qweight.shape
    T, K = x.shape
    if K2 * 2 != K or len(sizes) != E or tuple(s1_scales.shape) != (E, N) or tuple(s1_szeros.shape) != (E, N):
        raise RuntimeError("moe_gemm_forward_cuda_api: inconsistent shapes")
    if sum(sizes) != T:
        raise RuntimeError("moe_gemm_forward_cuda_api: problem_sizes must sum to the number of token rows")
    if out is None:
        out = torch.empty((T, N), dtype=torch.float16, device=x.device)
    arr = (C.c_int * E)(*[int(v) for v in sizes])
    L.check(L.lib().ob_w4a8_moe_gemm(L.ptr(x), L.ptr(qweight), L.ptr(s1_scales), L.ptr(input_scales), L.ptr(s1_szeros),
                                     L.ptr(input_sum), L.ptr(out), arr, E, T, N, K, out.stride(0), L.stream()),
            "moe_gemm_forward_cuda_api")
    return out


MAX_DEV_TOKENS = 64


def moe_gemm_forward_cuda_api_dev(x, qweight, s1_scales, input_scales, s1_szeros, input_sum, expert_offsets, num_tokens, out=None):
    """The same grouped GEMM with the expert row ranges in DEVICE memory: expert e owns rows [expert_offsets[e],
    expert_offsets[e + 1]) of x (int32 [E + 1], e.g. moe_helpers.moe_topk_gating_softmax(..., out_offsets=)).  Nothing is read
    back to the host, so the call is asynchronous and capturable in a CUDA graph.  The kernel serves at most 64 rows per
    expert, which holds whenever the layer has num_tokens <= 64 tokens (a token routes to distinct experts); larger layers
    raise ValueError -- use moe_gemm_forward_cuda_api or per-expert dense GEMMs there.  Returns fp16 [rows of x, N]."""
    if int(num_tokens) > MAX_DEV_TOKENS:
        raise ValueError(f"moe_gemm_forward_cuda_api_dev: {num_tokens} tokens; the device-offset GEMM serves <= {MAX_DEV_TOKENS}")
    E, N, K2 = qweight.shape
    T, K = x.shape
    if expert_offsets.dtype != torch.int32 or expert_offsets.numel() != E + 1:
        raise ValueError("moe_gemm_forward_cuda_api_dev: expert_offsets must be int32 [E + 1]")
    if K2 * 2 != K or tuple(s1_scales.shape) != (E, N) or tuple(s1_szeros.shape) != (E, N):
        raise ValueError("moe_gemm_forward_cuda_api_dev: inconsistent shapes")
    L.require_cuda(x, qweight, s1_scales, input_scales, s1_szeros, input_sum, expert_offsets, out)
    L.require_contiguous(x, qweight, s1_scales, input_scales, s1_szeros, input_sum, expert_offsets)
    if out is None:
        out = torch.empty((T, N), dtype=torch.float16, device=x.device)
    L.check(L.lib().ob_w4a8_moe_gemm_dev(L.ptr(x), L.ptr(qweight), L.ptr(s1_scales), L.ptr(input_scales), L.ptr(s1_szeros),
                                         L.ptr(input_sum), L.ptr(out), L.ptr(expert_offsets), E, T, N, K, out.stride(0),
                                         L.stream()), "moe_gemm_forward_cuda_api_dev")
    return out
