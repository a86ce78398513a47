"""moe_helpers: the routing, permutation and combine ops of the reference's Mixtral block, which it calls but never released
(omniserve/modeling/models/mixtral_w4a8_unpad.py:300-395; semantics pinned by oracle/moe.py).  Same functions and positional
argument order as the caller (:315, :345, :388); the device `expert_offsets` the grouped GEMM consumes comes out through the
extension keyword `out_offsets=`, since the caller unpacks exactly three values.  Every op is asynchronous and capturable in a
CUDA graph (no host read-back)."""
import torch

from .. import _lib as L

MAX_EXPERTS = 64
MAX_TOP_K = 8


def _check_routing(num_experts: int, top_k: int):
    if not 1 <= num_experts <= MAX_EXPERTS:
        raise ValueError(f"moe routing: {num_experts} experts (supported: 1..{MAX_EXPERTS})")
    if not 1 <= top_k <= min(num_experts, MAX_TOP_K):
        raise ValueError(f"moe routing: top_k {top_k} (supported: 1..min(E, {MAX_TOP_K}))")


def moe_router_logits(hidden_states, gate_weight, out=None):
    """`self.gate(hidden_states).float()` (:277,305): fp16 x [T, H] . gate_weight fp16 [E, H]^T -> fp32 [T, E] holding the
    fp16-rounded dot products.  A row's logits do not depend on the other rows of the batch (fixed reduction order)."""
    if hidden_states.dim() != 2 or gate_weight.dim() != 2 or hidden_states.shape[1] != gate_weight.shape[1]:
        raise ValueError("moe_router_logits: need x [T, H] and gate_weight [E, H]")
    if hidden_states.dtype != torch.float16 or gate_weight.dtype != torch.float16:
        raise ValueError("moe_router_logits: x and gate_weight must be fp16")
    T, H = hidden_states.shape
    E = gate_weight.shape[0]
    if not 1 <= E <= MAX_EXPERTS or H % 8:
        raise ValueError(f"moe_router_logits: E must be in 1..{MAX_EXPERTS} and H a multiple of 8")
    L.require_cuda(hidden_states, gate_weight, out)
    L.require_contiguous(hidden_states, gate_weight, out)
    if out is None:
        out = torch.empty((T, E), dtype=torch.float32, device=hidden_states.device)
    L.check(L.lib().ob_moe_router_logits(L.ptr(hidden_states), L.ptr(gate_weight), L.ptr(out), T, H, E, L.stream()),
            "moe_router_logits")
    return out


def moe_topk_gating_softmax(router_logits, top_k, out_offsets=None):
    """router_logits fp32 [T, E] -> (routing_weights fp32 [T, k], expert_indices int32 [T * k] token-major,
    permuted_loc_to_unpermuted_loc int32 [T * k]).  Softmax in fp32, the k most probable experts (ties: lower index; slots in
    descending p), weights renormalised over the k; rows sorted by expert, stably by (token, slot).  out_offsets: int32
    [E + 1] device tensor that receives expert_offsets (expert e owns permuted rows [off[e], off[e + 1]))."""
    if not torch.is_tensor(router_logits) or router_logits.dim() != 2:
        raise ValueError("moe_topk_gating_softmax: router_logits must be a [T, E] tensor")
    if router_logits.dtype != torch.float32:
        raise ValueError("moe_topk_gating_softmax: router_logits must be fp32 (`self.gate(x).float()`)")
    T, E = router_logits.shape
    _check_routing(E, int(top_k))
    k = int(top_k)
    if out_offsets is not None and (out_offsets.dtype != torch.int32 or out_offsets.numel() != E + 1):
        raise ValueError("moe_topk_gating_softmax: out_offsets must be int32 [E + 1]")
    L.require_cuda(router_logits, out_offsets)
    L.require_contiguous(router_logits, out_offsets)
    dev = router_logits.device
    weights = torch.empty((T, k), dtype=torch.float32, device=dev)
    idx = torch.empty((T * k,), dtype=torch.int32, device=dev)
    perm = torch.empty((T * k,), dtype=torch.int32, device=dev)
    offsets = out_offsets if out_offsets is not None else torch.empty((E + 1,), dtype=torch.int32, device=dev)
    L.check(L.lib().ob_moe_topk_sort(L.ptr(router_logits), L.ptr(weights), L.ptr(idx), L.ptr(perm), L.ptr(offsets), T, E, k,
                                     L.stream()), "moe_topk_gating_softmax")
    return weights, idx, perm


def moe_expand_inputs_and_scales(q_hidden_states, q_input_ssums, q_input_scales, permuted_loc_to_unpermuted_loc, out=None):
    """Gather the per-token INT8 rows [T, H] and their sums / scales fp16 [T] into permuted order (row r = token
    perm[r] // k).  Returns (q_moe_input_feats int8 [T * k, H], moe_input_ssums, moe_input_scales fp16 [T * k],
    unpermuted_loc_to_permuted_loc int32 [T * k]).  q_input_ssums may be None (then the second value is None).  out: an
    optional 4-tuple of preallocated outputs."""
    perm = permuted_loc_to_unpermuted_loc
    if q_hidden_states.dim() != 2 or q_hidden_states.dtype != torch.int8 or perm.dtype != torch.int32:
        raise ValueError("moe_expand_inputs_and_scales: need int8 [T, H] rows and an int32 permutation")
    T, H = q_hidden_states.shape
    n = perm.numel()
    if T == 0 or n % T or not 1 <= n // T <= MAX_TOP_K or H % 16:
        raise ValueError("moe_expand_inputs_and_scales: permutation length must be k * T (k <= 8), H a multiple of 16")
    k = n // T
    L.require_cuda(q_hidden_states, q_input_ssums, q_input_scales, perm)
    L.require_contiguous(q_hidden_states, q_input_ssums, q_input_scales, perm)
    dev = q_hidden_states.device
    if out is None:
        out = (torch.empty((n, H), dtype=torch.int8, device=dev),
               None if q_input_ssums is None else torch.empty((n,), dtype=torch.float16, device=dev),
               torch.empty((n,), dtype=torch.float16, device=dev), torch.empty((n,), dtype=torch.int32, device=dev))
    q_out, s_out, sc_out, inv = out
    L.check(L.lib().ob_moe_expand(L.ptr(q_hidden_states), L.ptr(q_input_ssums), L.ptr(q_input_scales), L.ptr(perm), L.ptr(q_out),
                                  L.ptr(s_out), L.ptr(sc_out), L.ptr(inv), T, k, H, L.stream()), "moe_expand_inputs_and_scales")
    return q_out, s_out, sc_out, inv


def moe_finalize_routing(q_w2_out, routing_weights, unpermuted_loc_to_permuted_loc, num_tokens, out=None):
    """out fp16 [T, H] = fp16(sum_j routing_weights[t, j] * q_w2_out[unpermuted_loc_to_permuted_loc[t * k + j]]) in fp32,
    j ascending.  q_w2_out fp16 [T * k, H] (expert outputs in permuted order)."""
    T = int(num_tokens)
    if routing_weights.dim() != 2 or routing_weights.shape[0] != T or routing_weights.dtype != torch.float32:
        raise ValueError("moe_finalize_routing: routing_weights must be fp32 [num_tokens, k]")
    k = routing_weights.shape[1]
    if not 1 <= k <= MAX_TOP_K or q_w2_out.dim() != 2 or q_w2_out.shape[0] != T * k or q_w2_out.dtype != torch.float16:
        raise ValueError("moe_finalize_routing: q_w2_out must be fp16 [num_tokens * k, H]")
    H = q_w2_out.shape[1]
    L.require_cuda(q_w2_out, routing_weights, unpermuted_loc_to_permuted_loc, out)
    L.require_contiguous(routing_weights, unpermuted_loc_to_permuted_loc, out)
    if q_w2_out.stride(1) != 1:
        raise RuntimeError("moe_finalize_routing: q_w2_out rows must be contiguous")
    if out is None:
        out = torch.empty((T, H), dtype=torch.float16, device=q_w2_out.device)
    L.check(L.lib().ob_moe_finalize(L.ptr(q_w2_out), L.ptr(routing_weights), L.ptr(unpermuted_loc_to_permuted_loc), L.ptr(out), T,
                                    k, H, q_w2_out.stride(0), L.stream()), "moe_finalize_routing")
    return out
