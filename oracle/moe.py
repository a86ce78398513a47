"""CPU definition of the Mixtral mixture-of-experts block of the W4A8 stack.

TEST INFRASTRUCTURE -- see oracle/__init__.py.  numpy only.

The reference calls these ops but never released them: MixtralSparseMoeBlockOurs.forward
(omniserve/modeling/models/mixtral_w4a8_unpad.py:300-395) raises NotImplementedError before
`moe_helpers.moe_topk_gating_softmax` (:315), `moe_expand_inputs_and_scales` (:345), the `w1_w3` / `w2`
grouped GEMMs (:354,382), `SiluAndMulQuant` (:376) and `moe_finalize_routing` (:388).  So this module is the
definition the CUDA ops (omniserve_b200/csrc/moe_ops.cu) are held to.
"""
from __future__ import annotations

import numpy as np

from . import act, w4a8

f32 = np.float32
f16 = np.float16


def router_logits(x_f16, gate_f16) -> np.ndarray:
    """``router_logits = self.gate(hidden_states).float()`` (:277,305): an fp16 nn.Linear without bias, i.e. the dot product
    of the fp16 normed row and the fp16 gate row accumulated in fp32 and rounded once to fp16; returned as fp32 [T, E].
    The dot product is evaluated exactly here (fp64); the kernel's fp32 accumulation differs only below the fp16 rounding."""
    x = np.asarray(x_f16, f16).astype(np.float64)
    g = np.asarray(gate_f16, f16).astype(np.float64)
    return (x @ g.T).astype(f16).astype(f32)


def softmax_f32(logits) -> np.ndarray:
    """``p = softmax(float(logits))`` over the experts, in fp32."""
    l = np.asarray(logits, f32)
    e = np.exp(l - l.max(axis=1, keepdims=True), dtype=f32)
    return (e / e.sum(axis=1, keepdims=True, dtype=f32)).astype(f32)


def topk_gating_softmax(logits, k: int):
    """moe_helpers.moe_topk_gating_softmax(router_logits, top_k) (:315), routing part.

    Selection: the k experts of largest p; ties go to the lower expert index; the k slots of a token are ordered by
    descending p, then ascending index.  Weights: Mixtral's renormalisation ``w = p_sel / sum(p_sel)`` in fp32 (the
    Hugging Face MixtralSparseMoeBlock definition) -- the chosen definition, since the reference never shipped its own.
    Returns (routing_weights fp32 [T, k], expert_indices int32 [T * k], token-major as the caller's torch.bincount (:320)
    expects)."""
    p = softmax_f32(logits)
    T, E = p.shape
    if not 1 <= k <= E:
        raise ValueError("need 1 <= k <= E")
    idx = np.empty((T, k), np.int32)
    w = np.empty((T, k), f32)
    for t in range(T):
        order = sorted(range(E), key=lambda e: (-float(p[t, e]), e))[:k]
        idx[t] = order
        sel = p[t, order].astype(f32)
        s = f32(0.0)
        for v in sel:
            s = f32(s + v)
        w[t] = sel / s
    return w, idx.reshape(-1)


def permutation(expert_indices, num_experts: int):
    """Routed rows sorted by expert; within an expert by flat position t * k + j ascending (a stable sort).  Returns
    (permuted_loc_to_unpermuted_loc int32 [T * k], expert_offsets int32 [E + 1]): expert e owns permuted rows
    [offsets[e], offsets[e + 1])."""
    ei = np.asarray(expert_indices, np.int64)
    perm = np.argsort(ei, kind="stable").astype(np.int32)
    counts = np.bincount(ei, minlength=num_experts)
    offsets = np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)
    return perm, offsets


def expand(q, ssums, scales, perm, k: int):
    """moe_helpers.moe_expand_inputs_and_scales (:345): row r of the expanded INT8 rows / sums / scales is token
    perm[r] // k.  Returns (q_out, ssums_out, scales_out, unpermuted_loc_to_permuted_loc)."""
    perm = np.asarray(perm, np.int64)
    tok = perm // k
    inv = np.empty(perm.shape[0], np.int32)
    inv[perm] = np.arange(perm.shape[0], dtype=np.int32)
    return np.asarray(q)[tok], np.asarray(ssums)[tok], np.asarray(scales)[tok], inv


def finalize(y_f16, weights, inv, num_tokens: int):
    """moe_helpers.moe_finalize_routing (:388): ``out[t] = fp16(sum_j w[t, j] * float(y[inv[t * k + j]]))``, fp32, j
    ascending (a product and a sum per step, each rounded to fp32)."""
    y = np.asarray(y_f16, f16).astype(f32)
    w = np.asarray(weights, f32)
    k = w.shape[1]
    inv = np.asarray(inv, np.int64).reshape(num_tokens, k)
    acc = np.zeros((num_tokens, y.shape[1]), f32)
    for j in range(k):
        acc = (acc + (w[:, j:j + 1] * y[inv[:, j]]).astype(f32)).astype(f32)
    return acc.astype(f16)


def moe_block(x_f16, gate_f16, w13, w2, k: int, logits=None):
    """The block of :300-395 on the fp16 post_attention_layernorm output x [T, H]: router, routing, per-token INT8 quant with
    the row sums (invoke_quant_fuse_sum, :334), expand, w1_w3 grouped GEMM (per-channel W4A8, [gate | up] halves as in the
    dense MLP), silu * mul -> INT8 quant with sums, w2 grouped GEMM, combine.  w13 / w2 = (qweight [E, N, K/2], s1_scales
    [E, N], s1_szeros [E, N]).  `logits` overrides the router (for tests that pin the routing).  Returns (out fp16 [T, H],
    dict of the intermediates)."""
    x = np.asarray(x_f16, f16)
    T = x.shape[0]
    E = np.asarray(gate_f16).shape[0]
    lg = router_logits(x, gate_f16) if logits is None else np.asarray(logits, f32)
    w, ei = topk_gating_softmax(lg, k)
    perm, offsets = permutation(ei, E)
    q, sc, ss = act.quant_fuse_sum(x)
    qe, sse, sce, inv = expand(q, ss, sc, perm, k)
    sizes = np.diff(offsets)
    gu = w4a8.moe_gemm_per_chn(qe, w13[0], w13[1], sce, w13[2], sse, sizes)
    qm, sc2, ss2 = act.quant_fuse_sum(act.silu_and_mul(gu))
    y = w4a8.moe_gemm_per_chn(qm, w2[0], w2[1], sc2, w2[2], ss2, sizes)
    out = finalize(y, w, inv, T)
    return out, dict(logits=lg, weights=w, expert_indices=ei, perm=perm, offsets=offsets, inv=inv, gate_up=gu, y=y)
