"""Oracle of LServe's token-streaming ("Lambda"-masked) prefill attention -- test infrastructure only.

Mask: query position i of a sequence attends key position j iff  j <= i  and  (j < sink  or  i - j < local).
  * head_mask_type -1 = streaming head with (sink, local) from streaming_info, 0 = dense causal head
    (reference omniserve/modeling/layers/ctx_attn/ctx_attn_init.py:11-52, repeated per GQA group);
  * the window is the one the streaming-head decode attention keeps: the sink plus the last `local` tokens, the current
    token included (reference .../sparse_attention/decoderMaskedMultiheadAttentionTemplate.hpp:1570-1584;
    tests/test_gpu_lserve.py `positions()`: min(sink + local - 1, cached) cached tokens + the new one).
Exact attention is computed in float64 for selected rows.
"""
from __future__ import annotations

import numpy as np


def attends(i, j, sink: int, local: int):
    """Elementwise mask (numpy broadcasting)."""
    i, j = np.asarray(i), np.asarray(j)
    return (j <= i) & ((j < sink) | (i - j < local))


def mask(L: int, sink: int, local: int) -> np.ndarray:
    """bool [L, L]: row = query position, column = key position."""
    i = np.arange(L)[:, None]
    j = np.arange(L)[None, :]
    return attends(i, j, sink, local)


def attended_positions(i: int, sink: int, local: int) -> np.ndarray:
    """Key positions query position i attends, ascending."""
    j = np.arange(i + 1)
    return j[attends(i, j, sink, local)]


def attention_rows(q, k, v, cu_seqlens, kv_head: int, sink: int, local: int, rows=None) -> dict:
    """Exact (float64) token-streaming attention of the g q-heads of `kv_head`.
    q [T, Hq, Dh], k / v [T, Hkv, Dh] (numpy, any float dtype), cu_seqlens [B + 1].  rows: global token indices to compute
    (default: all).  -> {row: float64 [g, Dh]}."""
    T, hq, dh = q.shape
    g = hq // k.shape[1]
    cu = np.asarray(cu_seqlens, np.int64)
    rows = range(T) if rows is None else rows
    out = {}
    scale = 1.0 / np.sqrt(dh)
    for t in rows:
        b = int(np.searchsorted(cu, t, side="right")) - 1
        s0 = int(cu[b])
        pos = attended_positions(t - s0, sink, local) + s0
        kk = k[pos, kv_head].astype(np.float64)
        vv = v[pos, kv_head].astype(np.float64)
        qq = q[t, kv_head * g:(kv_head + 1) * g].astype(np.float64)
        s = qq @ kk.T * scale
        s -= s.max(axis=1, keepdims=True)
        p = np.exp(s)
        out[t] = (p @ vv) / p.sum(axis=1, keepdims=True)
    return out
