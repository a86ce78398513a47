"""Prefill (context-stage) attention.

In the reference this is third-party FP16 FlashAttention (`flash_attn_varlen_func` / `block_sparse_attn`,
omniserve/modeling/layers/ctx_attn/ctx_attn_func.py:40-87).
  * Dense heads: `make()` calls PyTorch's fused causal SDPA, which is library code in the same sense (SURVEY.md section 2b).
  * LServe's streaming heads: `token_streaming_attn_func` (the reference's `block_sparse_attn.token_streaming_attn_func`,
    ctx_attn_func.py:62-73) sends them to this project's own kernel (csrc/prefill_attention.cu), whose work per query is
    bounded by sink + local instead of growing with the prompt.  Query position i attends key j iff
    j <= i and (j < sink or i - j < local) -- the window the streaming-head decode attention keeps, so a prompt prefilled
    and then decoded sees one consistent window.  Dense heads of the same call go to `make()`.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Sequence

import torch
import torch.nn.functional as F

from . import _lib as L

HEAD_DIM = 128


def make(cu_seqlens: torch.Tensor, max_len: int, hq: int, hkv: int, dh: int):
    lens = (cu_seqlens[1:] - cu_seqlens[:-1]).tolist()
    offs = cu_seqlens.tolist()
    uniform = len(set(lens)) == 1
    g = hq // hkv

    def attn(q, k, v):  # q [T,hq,dh], k/v [T,hkv,dh] (strided views) -> [T,hq,dh]
        T = q.shape[0]
        if uniform:
            B, L = len(lens), lens[0]
            qq = q.reshape(B, L, hq, dh).transpose(1, 2)
            kk = k.reshape(B, L, hkv, dh).transpose(1, 2)
            vv = v.reshape(B, L, hkv, dh).transpose(1, 2)
            o = F.scaled_dot_product_attention(qq, kk, vv, is_causal=True, enable_gqa=(g > 1))
            return o.transpose(1, 2).reshape(T, hq, dh)
        out = torch.empty((T, hq, dh), dtype=q.dtype, device=q.device)
        for b, L in enumerate(lens):
            s = offs[b]
            qq = q[s:s + L].transpose(0, 1).unsqueeze(0)
            kk = k[s:s + L].transpose(0, 1).unsqueeze(0)
            vv = v[s:s + L].transpose(0, 1).unsqueeze(0)
            o = F.scaled_dot_product_attention(qq, kk, vv, is_causal=True, enable_gqa=(g > 1))
            out[s:s + L] = o.squeeze(0).transpose(0, 1)
        return out

    return attn


# ---------------------------------------------------------------------------------------------- streaming heads
def split_heads(head_mask_type, streaming_info, hq: int, hkv: int):
    """Validate the reference's per-q-head masks (ctx_attn_init.py:30-45: -1 = streaming, 0 = dense; streaming_info =
    (sink, local) per q-head, repeated over each GQA group) and reduce them to kv groups.
    -> (streaming kv heads, their sinks, their locals, dense kv heads)."""
    if hq <= 0 or hkv <= 0 or hq % hkv:
        raise ValueError(f"{hq} query heads cannot be grouped over {hkv} kv heads")
    g = hq // hkv
    mt = [int(x) for x in (head_mask_type.tolist() if torch.is_tensor(head_mask_type) else head_mask_type)]
    si = [int(x) for x in (streaming_info.reshape(-1).tolist() if torch.is_tensor(streaming_info) else streaming_info)]
    if len(mt) != hq:
        raise ValueError(f"head_mask_type has {len(mt)} entries for {hq} query heads")
    if any(x not in (0, -1) for x in mt):
        raise ValueError("head_mask_type entries must be 0 (dense) or -1 (streaming); block-sparse heads are not supported")
    if len(si) != 2 * hq:
        raise ValueError(f"streaming_info has {len(si)} entries, expected (sink, local) for each of {hq} query heads")
    s_kv, sinks, locals_, d_kv = [], [], [], []
    for h in range(hkv):
        grp = range(h * g, (h + 1) * g)
        if len({mt[i] for i in grp}) != 1 or len({(si[2 * i], si[2 * i + 1]) for i in grp}) != 1:
            raise ValueError(f"head_mask_type / streaming_info differ within the GQA group of kv head {h}")
        sink, local = si[2 * h * g], si[2 * h * g + 1]
        if mt[h * g] == -1:
            if sink < 0 or local < 1:
                raise ValueError(f"kv head {h}: sink must be >= 0 and local >= 1 (got {sink}, {local})")
            s_kv.append(h); sinks.append(sink); locals_.append(local)
        else:
            d_kv.append(h)
    return s_kv, sinks, locals_, d_kv


def _args(q, k, v, out, cu: Sequence[int], hq: int, hkv: int, kv_heads, sinks, locals_):
    i32 = C.c_int32
    keep = [(i32 * len(cu))(*cu), (i32 * max(len(kv_heads), 1))(*kv_heads), (i32 * max(len(sinks), 1))(*sinks),
            (i32 * max(len(locals_), 1))(*locals_)]
    a = L.StreamingPrefillArgs()
    a.q, a.k, a.v, a.out = L.ptr(q), L.ptr(k), L.ptr(v), L.ptr(out)
    a.q_row_stride = q.stride(0) if q is not None else 0
    a.k_row_stride = k.stride(0) if k is not None else 0
    a.v_row_stride = v.stride(0) if v is not None else 0
    a.cu_seqlens = C.cast(keep[0], C.c_void_p)
    a.batch, a.num_tokens, a.num_heads, a.num_kv_heads, a.head_dim = len(cu) - 1, cu[-1], hq, hkv, HEAD_DIM
    a.num_compute_kv_heads = len(kv_heads)
    a.kv_heads, a.sink, a.local = (C.cast(x, C.c_void_p) for x in keep[1:])
    return a, keep


def streaming_prefill_attention(q, k, v, cu_seqlens, kv_heads: List[int], sinks: List[int], locals_: List[int], out=None):
    """The kernel alone: token-streaming attention of the q-heads of `kv_heads` (each with its group's sink / local).
    q [T, Hq, 128], k / v [T, Hkv, 128] fp16 views with head stride 128 (e.g. cut from the qkv activation); cu_seqlens
    int32 [B + 1] (device or host).  out fp16 [T, Hq, 128] contiguous (allocated if None); only those heads' slots are
    written."""
    L.require_cuda(q, k, v, out)
    T, hq, dh = q.shape
    hkv = k.shape[1]
    if dh != HEAD_DIM or k.shape[2] != HEAD_DIM or v.shape[2] != HEAD_DIM:
        raise ValueError("token-streaming attention needs head_dim 128")
    for name, x in (("q", q), ("k", k), ("v", v)):
        if x.dtype != torch.float16:
            raise ValueError(f"{name} must be fp16")
        if x.stride(2) != 1 or x.stride(1) != HEAD_DIM:
            raise ValueError(f"{name} must have unit inner stride and head stride 128")
    if out is None:
        out = torch.empty((T, hq, HEAD_DIM), dtype=torch.float16, device=q.device)
    elif out.shape != (T, hq, HEAD_DIM) or out.dtype != torch.float16 or not out.is_contiguous():
        raise ValueError("out must be a contiguous fp16 [T, Hq, 128] tensor")
    cu = [int(x) for x in (cu_seqlens.tolist() if torch.is_tensor(cu_seqlens) else cu_seqlens)]
    a, keep = _args(q, k, v, out, cu, hq, hkv, kv_heads, sinks, locals_)
    L.check(L.lib().ob_token_streaming_prefill_attention(C.byref(a), L.stream()), "token_streaming_prefill_attention")
    return out


def streaming_prefill_plan(cu_seqlens: Sequence[int], hq: int, hkv: int, kv_heads, sinks, locals_):
    """Host-only (no GPU): the launch plan of `streaming_prefill_attention`, one dict per CTA:
    launch, cta (x, y), seq, q_lo, q_hi (positions within the sequence), kv_head, key_tiles (64-key tile indices)."""
    cu = [int(x) for x in cu_seqlens]
    a, keep = _args(None, None, None, None, cu, hq, hkv, kv_heads, sinks, locals_)
    lib = L.lib()
    out = (C.c_int * 8)()
    cap = 1 << 16
    tiles = (C.c_int * cap)()
    L.check(lib.ob_debug_streaming_prefill_plan(C.byref(a), 0, 0, 0, out, tiles, cap), "streaming_prefill_plan")
    ctas = []
    for launch in range(out[0]):
        L.check(lib.ob_debug_streaming_prefill_plan(C.byref(a), launch, 0, 0, out, tiles, cap), "streaming_prefill_plan")
        gx, gy = out[1], out[2]
        for y in range(gy):
            for x in range(gx):
                L.check(lib.ob_debug_streaming_prefill_plan(C.byref(a), launch, x, y, out, tiles, cap), "streaming_prefill_plan")
                ctas.append(dict(launch=launch, cta=(x, y), seq=out[3], q_lo=out[4], q_hi=out[5], kv_head=out[6],
                                 key_tiles=list(tiles[:min(out[7], cap)])))
    return ctas


def _fused_sdpa():
    """Long-context SDPA must not fall back to the math backend (it would materialise L x L scores)."""
    from torch.nn.attention import SDPBackend, sdpa_kernel
    return sdpa_kernel([SDPBackend.FLASH_ATTENTION, SDPBackend.CUDNN_ATTENTION, SDPBackend.EFFICIENT_ATTENTION])


def token_streaming_attn_func(q, k, v, cu_seqlens_q, cu_seqlens_k, head_mask_type, streaming_info, max_seqlen_q,
                              max_seqlen_k):
    """block_sparse_attn.token_streaming_attn_func with the reference caller's positional order (ctx_attn_func.py:68-73).
    q [T, Hq, 128], k / v [T, Hkv, 128] fp16 (views into the qkv activation are fine); head_mask_type int [Hq] (-1 streaming,
    0 dense); streaming_info int [2 * Hq] = (sink, local) per q-head.  Streaming heads run this project's kernel, dense heads
    fused causal SDPA on their gathered GQA groups.  -> fp16 [T, Hq, 128] contiguous."""
    if q.dim() != 3 or k.dim() != 3 or v.dim() != 3:
        raise ValueError("q, k, v must be [T, heads, head_dim]")
    T, hq, dh = q.shape
    hkv = k.shape[1]
    if dh != HEAD_DIM or k.shape[2] != HEAD_DIM or v.shape[2] != HEAD_DIM:
        raise ValueError(f"token-streaming attention needs head_dim 128 (got {dh})")
    if k.shape[0] != T or v.shape != k.shape:
        raise ValueError("k / v must be [T, Hkv, 128] with the same T as q")
    cu_q = [int(x) for x in (cu_seqlens_q.tolist() if torch.is_tensor(cu_seqlens_q) else cu_seqlens_q)]
    cu_k = [int(x) for x in (cu_seqlens_k.tolist() if torch.is_tensor(cu_seqlens_k) else cu_seqlens_k)]
    if cu_q != cu_k:
        raise ValueError("cu_seqlens_q must equal cu_seqlens_k (prefill with a cached prefix is not supported)")
    if len(cu_q) < 2 or cu_q[0] != 0 or cu_q[-1] != T or any(b < a for a, b in zip(cu_q, cu_q[1:])):
        raise ValueError("cu_seqlens must start at 0, be non-decreasing and end at T")
    s_kv, sinks, locals_, d_kv = split_heads(head_mask_type, streaming_info, hq, hkv)
    L.require_cuda(q, k, v)
    L.lib()
    g = hq // hkv
    cu_dev = torch.tensor(cu_q, dtype=torch.int32, device=q.device)
    max_len = max(b - a for a, b in zip(cu_q, cu_q[1:]))
    if not s_kv:          # all dense: the reference's flash_attn_varlen_func branch
        with _fused_sdpa():
            return make(cu_dev, max_len, hq, hkv, dh)(q, k, v)
    out = torch.empty((T, hq, HEAD_DIM), dtype=torch.float16, device=q.device)
    streaming_prefill_attention(q, k, v, cu_q, s_kv, sinks, locals_, out)
    if d_kv:
        qh = [h * g + i for h in d_kv for i in range(g)]
        idx_q = torch.tensor(qh, device=q.device)
        idx_kv = torch.tensor(d_kv, device=q.device)
        with _fused_sdpa():
            o = make(cu_dev, max_len, len(qh), len(d_kv), dh)(q.index_select(1, idx_q), k.index_select(1, idx_kv),
                                                              v.index_select(1, idx_kv))
        out.index_copy_(1, idx_q, o)
    return out
