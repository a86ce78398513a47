"""Mixtral-style W4A8KV4 mixture-of-experts decoder stack (single GPU): a real batched prefill and a CUDA-graph decode step.

Mirrors the reference's unreleased Mixtral model (omniserve/modeling/models/mixtral_w4a8_unpad.py):
  * MixtralDecoderLayer.forward      :441-463 -- input_layernorm (RMSNormGeneral -> INT8 + sum), KV4 attention,
                                      residual add, post_attention_layernorm (plain RMSNorm, fp16), MoE block, residual add
  * MixtralSparseMoeBlockOurs        :269-395 -- router, top-k routing, per-token quant, expand, w1_w3 grouped GEMM,
                                      silu * mul -> quant, w2 grouped GEMM, combine (semantics: oracle/moe.py)
  * MoEW4A8OF16LinearDynamicInputScale  (w4a8_moe_linear.py) -- per-channel expert weights [E, N, K/2], s1_scales / s1_szeros [E, N]
The attention half is the dense stack's (omniserve_b200/model.py): the same ops, PagedKVCache and fused attention + quant.
The residual add after the MoE block is folded into the next layer's input norm, as in LlamaW4A8._layer.

Decode (<= 64 tokens) runs the grouped GEMMs with device-resident expert offsets and never synchronises the host, so
model.DecodeGraph captures it unchanged.  Prefill reads the expert offsets to the host once per layer and runs each expert's
contiguous rows through the dense per-channel GEMM (the persistent tcgen05 kernel for large groups), which streams an
expert's weights once instead of once per 64 rows.
"""
from __future__ import annotations

import math
from dataclasses import dataclass

import torch

from . import _lib as L
from .model import ActivationBuffer, LlamaConfig, LlamaW4A8, Ops, PagedKVCache, W4A8Linear, TOKENS_PER_BLOCK

MAX_DECODE_TOKENS = 64   # the device-offset grouped GEMM serves <= 64 rows per expert


@dataclass
class MixtralConfig(LlamaConfig):
    vocab_size: int = 32000
    rope_theta: float = 1e6
    num_local_experts: int = 8
    num_experts_per_tok: int = 2

    @staticmethod
    def mixtral_8x7b(**kw):
        """Mixtral-8x7B: hidden 4096, intermediate 14336, 32 layers, 32 / 8 heads of 128, vocab 32000, rope_theta 1e6,
        rms eps 1e-5, 8 experts, top-2, per-channel W4A8."""
        return MixtralConfig(**kw)

    @staticmethod
    def tiny(**kw):
        d = dict(hidden_size=256, intermediate_size=512, num_hidden_layers=2, num_attention_heads=4, num_key_value_heads=2,
                 vocab_size=1024, num_local_experts=4, num_experts_per_tok=2)
        d.update(kw)
        return MixtralConfig(**d)


class MoEW4A8Linear:
    """Buffers of MoEW4A8OF16LinearDynamicInputScale, per-channel: qweight int8 [E, N, K/2] (each expert in the
    w4a8_linear.py:297-327 tile layout), s1_scales / s1_szeros fp16 [E, N]."""

    def __init__(self, num_experts: int, in_features: int, out_features: int, device):
        assert in_features % 128 == 0 and out_features % 128 == 0
        self.num_experts, self.in_features, self.out_features = num_experts, in_features, out_features
        self.qweight = torch.zeros((num_experts, out_features, in_features // 2), dtype=torch.int8, device=device)
        self.s1_scales = torch.zeros((num_experts, out_features), dtype=torch.float16, device=device)
        self.s1_szeros = torch.zeros((num_experts, out_features), dtype=torch.float16, device=device)

    def random_init_(self, gen: torch.Generator, std: float = 0.02):
        """W4A8Linear.random_init_ per expert -- random packed-u4 bytes, s1 = U(0.75, 1.25) * std / 4.6 -- except that the
        zero point is 7.5 * s1 (W4A8Linear: 8 * s1), so the synthetic weights (q - 7.5) * s1 have zero mean.  The router
        input is a plain RMSNorm output whose rows do not sum to zero (the dense stack's norm subtracts the mean), and with
        a -0.5 * s1 mean weight the gate and up halves share a bias that drives the fp16 row sums of silu * up past 65504
        at the Mixtral-8x7B shape.  `gen` may be a CPU or a device generator; a device generator fills the weights where
        they live (the full Mixtral shape holds 22.5 GB of expert weights)."""
        dev = self.qweight.device
        on_dev = gen.device.type != "cpu"
        E, N = self.num_experts, self.out_features
        for e in range(E):
            q = torch.randint(0, 256, self.qweight[e].shape, generator=gen, dtype=torch.uint8,
                              device=gen.device if on_dev else "cpu")
            self.qweight[e].view(torch.uint8).copy_(q)
        s1 = (torch.rand((E, N), generator=gen, device=gen.device if on_dev else "cpu") * 0.5 + 0.75) * (std / 4.6)
        self.s1_scales.copy_(s1.half().to(dev))
        self.s1_szeros.copy_((s1.half().float() * 7.5).half().to(dev))
        return self


class MoEBuffers:
    """Activation arena of the MoE block for T tokens (T * k routed rows)."""

    def __init__(self, T: int, k: int, E: int, hidden: int, inter: int, device):
        n = T * k
        f16, i8, i32 = torch.float16, torch.int8, torch.int32
        self.normed = torch.empty((T, hidden), dtype=f16, device=device)
        self.logits = torch.empty((T, E), dtype=torch.float32, device=device)
        self.offsets = torch.zeros((E + 1,), dtype=i32, device=device)
        self.q_in = torch.empty((n, hidden), dtype=i8, device=device)
        self.sum_in = torch.empty((n,), dtype=f16, device=device)
        self.scale_in = torch.empty((n,), dtype=f16, device=device)
        self.inv = torch.empty((n,), dtype=i32, device=device)
        self.gate_up = torch.empty((n, 2 * inter), dtype=f16, device=device)
        self.q_act = torch.empty((n, inter), dtype=i8, device=device)
        self.sum_act = torch.empty((n,), dtype=f16, device=device)
        self.scale_act = torch.empty((n,), dtype=f16, device=device)
        self.y = torch.empty((n, hidden), dtype=f16, device=device)
        self.out = torch.empty((T, hidden), dtype=f16, device=device)


def _add_f16(out, a, b):
    L.check(L.lib().ob_add_f16(L.ptr(out), L.ptr(a), L.ptr(b), a.numel(), L.stream()), "add_f16")


class MixtralW4A8(LlamaW4A8):
    """Mixtral decoder stack over the W4A8KV4 ops.  alloc / prefill / decode_step have LlamaW4A8's meanings; there are no
    dense-MLP weights.  device_init=True draws the expert weights with a seeded generator on the device."""

    def __init__(self, cfg: MixtralConfig, device="cuda", seed: int = 0, device_init: bool = False, ops: Ops = None):
        if cfg.group_size != -1:
            raise ValueError("MixtralW4A8: per-channel experts only (group_size = -1)")
        self.ops = ops or Ops()
        from .backend import activation_ops, moe_helpers, qgemm_w4a8_moe
        self.moe_helpers, self.moe_gemm, self.activation_ops = moe_helpers, qgemm_w4a8_moe, activation_ops
        self.cfg, self.device, self.tp_rank, self.tp_size, self.pg = cfg, device, 0, 1, None
        E, k = cfg.num_local_experts, cfg.num_experts_per_tok
        if not 1 <= E <= moe_helpers.MAX_EXPERTS or not 1 <= k <= min(E, moe_helpers.MAX_TOP_K):
            raise ValueError(f"MixtralW4A8: {E} experts, top-{k} (supported: E <= 64, 1 <= k <= min(E, 8))")
        self.hq, self.hkv = cfg.num_attention_heads, cfg.num_key_value_heads
        self.q_size, self.kv_size = self.hq * cfg.head_dim, self.hkv * cfg.head_dim
        self.inter = cfg.intermediate_size
        self.fuse_silu_quant = True
        self.fuse_add_norm = hasattr(self.ops.layernorm_ops, "add_rms_norm_general")
        self.fuse_attn_quant = hasattr(self.ops.fused_attention_pure_dense, "single_query_attention_quant")
        self.fuse_gemm_norm = False
        self.act_sum = True
        gen = torch.Generator().manual_seed(seed * 1000)
        gen_rep = torch.Generator().manual_seed(seed * 1000 + 999)
        gen_dev = torch.Generator(device=device).manual_seed(seed * 1000 + 7) if device_init else None
        H = cfg.hidden_size
        self.layers = []
        for _ in range(cfg.num_hidden_layers):
            ly = {
                "qkv_proj": W4A8Linear(H, self.q_size + 2 * self.kv_size, -1, device, self.ops).random_init_(gen),
                "o_proj": W4A8Linear(self.q_size, H, -1, device, self.ops).random_init_(gen),
                "gate": (torch.randn((E, H), generator=gen) / math.sqrt(H)).half().to(device),
                "w1_w3": MoEW4A8Linear(E, H, 2 * self.inter, device).random_init_(gen_dev or gen),
                "w2": MoEW4A8Linear(E, self.inter, H, device).random_init_(gen_dev or gen),
                "input_layernorm": (1.0 + 0.05 * torch.randn(H, generator=gen_rep)).half().to(device),
                "post_attention_layernorm": (1.0 + 0.05 * torch.randn(H, generator=gen_rep)).half().to(device),
            }
            self.layers.append(ly)
        self.norm_weight = (1.0 + 0.05 * torch.randn(H, generator=gen_rep)).half().to(device)
        self.embed_tokens = (torch.randn(cfg.vocab_size, H, generator=gen_rep) * 0.5).half().to(device)
        self.vocab_local = cfg.vocab_size
        self.lm_head = (torch.randn(cfg.vocab_size, H, generator=torch.Generator().manual_seed(seed * 1000 + 500)) * 0.02).half().to(device)
        self.kv = None
        self.buf = None
        self.moe_buf = None
        self.peer = False
        self.record_moe_inputs = None   # a list: every MoE block appends (layer, normed input) -- for tests
        self._flags = torch.ones(self.hkv, dtype=torch.int32, device=device)
        self._rank = torch.arange(self.hkv, dtype=torch.int32, device=device)

    def weight_bytes(self) -> int:
        n = 0
        for ly in self.layers:
            n += ly["qkv_proj"].qweight.numel() + ly["o_proj"].qweight.numel()
            n += ly["w1_w3"].qweight.numel() + ly["w2"].qweight.numel()
        return n

    def alloc(self, batch: int, max_ctx: int, max_tokens: int):
        cfg = self.cfg
        self.kv = PagedKVCache(cfg, self.hkv, batch, max_ctx, self.device)
        self.buf = ActivationBuffer(max_tokens, cfg.hidden_size, 0, self.q_size + 2 * self.kv_size, self.q_size, self.device)
        self.moe_buf = MoEBuffers(max_tokens, cfg.num_experts_per_tok, cfg.num_local_experts, cfg.hidden_size, self.inter,
                                  self.device)
        self.batch, self.max_ctx = batch, max_ctx
        self.context_lens = torch.zeros((batch,), dtype=torch.int32, device=self.device)

    # ------------------------------------------------------------------ the MoE block
    def _experts(self, lin: MoEW4A8Linear, x, scales, sums, out, T: int, offsets_host):
        """One grouped W4A8 GEMM over the routed rows.  Device offsets (<= 64 tokens, no host sync) or, with the host copy
        of the offsets, the dense per-channel GEMM on each expert's contiguous rows."""
        if offsets_host is None:
            self.moe_gemm.moe_gemm_forward_cuda_api_dev(x, lin.qweight, lin.s1_scales, scales, lin.s1_szeros, sums,
                                                        self.moe_buf.offsets, T, out=out)
            return
        gemm = self.ops.qgemm_w4a8_per_chn.gemm_forward_cuda
        for e in range(lin.num_experts):
            r0, r1 = offsets_host[e], offsets_host[e + 1]
            if r1 > r0:
                gemm(x[r0:r1], lin.qweight[e], lin.s1_scales[e], scales[r0:r1], lin.s1_szeros[e], sums[r0:r1], out[r0:r1])

    def moe_block(self, li: int, x, device_offsets: bool):
        """mixtral_w4a8_unpad.py:300-395 on the fp16 post_attention_layernorm output x [T, H]; returns fp16 [T, H] (a view of
        the arena).  device_offsets=True: no host synchronisation (T <= 64)."""
        cfg, ly, m, b = self.cfg, self.layers[li], self.moe_buf, self.buf
        T = x.shape[0]
        k = cfg.num_experts_per_tok
        n = T * k
        if device_offsets and T > MAX_DECODE_TOKENS:
            raise ValueError(f"MixtralW4A8: {T} tokens; the device-offset MoE path serves <= {MAX_DECODE_TOKENS}")
        if self.record_moe_inputs is not None:
            self.record_moe_inputs.append((li, x.clone()))
        mh = self.moe_helpers
        logits = mh.moe_router_logits(x, ly["gate"], out=m.logits[:T])
        weights, _, perm = mh.moe_topk_gating_softmax(logits, k, out_offsets=m.offsets)
        qh, sc, sm = b.quantized_hidden_states_buffer[:T], b.quantized_scale_buffer[:T], b.quantized_sum_buffer[:T]
        self.ops.fused_kernels.invoke_quant_fuse_sum(qh, x, sm, sc)
        qe, se, sce, inv = mh.moe_expand_inputs_and_scales(qh, sm, sc, perm, out=(m.q_in[:n], m.sum_in[:n], m.scale_in[:n], m.inv[:n]))
        offsets_host = None if device_offsets else m.offsets.tolist()   # prefill: one host read-back per layer
        gu = m.gate_up[:n]
        self._experts(ly["w1_w3"], qe, sce, se, gu, T, offsets_host)
        qm, sm2, sc2 = m.q_act[:n], m.sum_act[:n], m.scale_act[:n]
        self.activation_ops.silu_and_mul_quant(qm, gu, sm2, sc2)
        y = m.y[:n]
        self._experts(ly["w2"], qm, sc2, sm2, y, T, offsets_host)
        return mh.moe_finalize_routing(y, weights, inv, T, out=m.out[:T])

    # ------------------------------------------------------------------ one decoder layer
    def _layer(self, li: int, hidden, delta, T: int, is_prompt: bool, meta):
        """hidden (+ delta, the previous layer's not-yet-added MoE output) -> (hidden', delta').  The attention half is
        LlamaW4A8._layer's (steps 1-5); then residual add, plain RMSNorm and the MoE block (mixtral_w4a8_unpad.py:455-462)."""
        cfg, ly, b = self.cfg, self.layers[li], self.buf
        fused_attention_fine_grained_dense = self.ops.fused_attention_fine_grained_dense
        fused_attention_pure_dense = self.ops.fused_attention_pure_dense
        qh = b.quantized_hidden_states_buffer[:T]
        sc, sm = b.quantized_scale_buffer[:T], b.quantized_sum_buffer[:T]
        qkv = b.qkv_proj_act_buffer[:T]
        od = b.out_down_proj_act_buffer[:T]
        ha, hb = b.hidden_a[:T], b.hidden_b[:T]
        # 1. (residual add of the previous MoE output +) input_layernorm -> int8 + sum
        h1 = self._norm_quant(qh, hidden, delta, ha, ly["input_layernorm"], sm, sc)
        # 2. qkv_proj
        ly["qkv_proj"](qh, sc, sm, qkv)
        q3 = qkv[:, : self.q_size].view(T, self.hq, cfg.head_dim)
        k3 = qkv[:, self.q_size: self.q_size + self.kv_size].view(T, self.hkv, cfg.head_dim)
        v3 = qkv[:, self.q_size + self.kv_size:].view(T, self.hkv, cfg.head_dim)
        qa = b.quantized_attn_buffer[:T]
        if is_prompt:
            # 3a. RoPE in place + KV4 page write, then fp16 attention; 4. quant + sum
            fused_attention_fine_grained_dense.apply_bias_rope_update_kv_cache(
                qkv, meta["seq_lens"], None, meta["padding_offset"], self.kv.tables[li], None, meta["flags"],
                meta["rank"], self.hq, self.hkv, meta["max_seq_len"], TOKENS_PER_BLOCK, self.kv_size // 2, 0, 0, 0, 0,
                0, self.hkv, 0, cfg.head_dim, cfg.rope_theta, 1.0, 8192, True, True, True)
            attn = meta["prefill_attn"](q3, k3, v3).reshape(T, self.q_size)
            self.ops.fused_kernels.invoke_quant_fuse_sum(qa, attn, sm, sc)
        elif self.fuse_attn_quant:
            # 3b. KV4 decode attention with the quant of step 4 fused in
            fused_attention_pure_dense.single_query_attention_quant(
                q3, k3, v3, self.kv.tables[li], meta["context_lens"], None, self.max_ctx, TOKENS_PER_BLOCK,
                self.kv_size // 2, meta["timestep"], cfg.head_dim, cfg.rope_theta, True, True, True,
                qa, sm, sc, history_is_stable=True)
        else:
            attn = fused_attention_pure_dense.single_query_attention(
                q3, k3, v3, self.kv.tables[li], meta["context_lens"], None, self.max_ctx, TOKENS_PER_BLOCK,
                self.kv_size // 2, meta["timestep"], cfg.head_dim, cfg.rope_theta, True, True, True).reshape(T, self.q_size)
            self.ops.fused_kernels.invoke_quant_fuse_sum(qa, attn, sm, sc)
        # 5. o_proj
        ly["o_proj"](qa, sc, sm, od)
        # 6. residual add + post_attention_layernorm (plain RMSNorm, fp16 out: the router reads it)
        _add_f16(hb, h1, od)
        xn = self.moe_buf.normed[:T]
        self.ops.layernorm_ops.rms_norm(xn, hb, ly["post_attention_layernorm"], cfg.rms_norm_eps)
        # 7. MoE block; its residual add is folded into the next norm
        return hb, self.moe_block(li, xn, device_offsets=not is_prompt)

    @torch.no_grad()
    def decode_step(self, tokens: torch.Tensor, timestep: int):
        """As LlamaW4A8.decode_step; batches of more than 64 tokens raise ValueError (the device-offset grouped GEMM)."""
        if tokens.numel() > MAX_DECODE_TOKENS:
            raise ValueError(f"MixtralW4A8.decode_step: batch {tokens.numel()} > {MAX_DECODE_TOKENS}")
        return super().decode_step(tokens, timestep)
