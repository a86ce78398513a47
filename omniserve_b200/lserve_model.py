"""LServe long-context sparse decode of a Llama W4A8KV4 stack (BASELINE config 3: Llama-3-8B-Instruct-Gradient-1048k,
256K context, bs = 1) on top of the `omniserve_backend`-compatible ops.

Mirrors, per layer, the reference's decode path with static + dynamic sparsity switched on
(omniserve/modeling/models/llama_w4a8_unpad.py:326-361 -> DecodingAttentionWrapper.forward_w_dynamic_sparse_fine_grained,
omniserve/modeling/layers/decoding_attention.py:88-143,236-304):
  * every KV head is a RETRIEVAL head (full history in a retrieval page pool that also carries the kmax / kmin page statistics)
    or a STREAMING head (sink + local ring pool); the split comes from the model's attn_patterns file at a static sparsity
    (omniserve/attn_config.py:113-150, head tables ctx_attn_init.py:52-76);
  * retrieval q-heads attend `dynamic_sparse_token_budget / 64` pages chosen by the page selector, re-chosen every
    `selector_update_interval` steps (the cached choice is reused in between);
  * everything else (norms, W4A8 GEMMs, quant, SiLU) is the dense layer of omniserve_b200/model.py.
The prompt (context) stage, `LServeDecoder.prefill`, mirrors the reference's prompt path of the same layers
(llama_w4a8_unpad.py:83-111,265-325; ctx_attn_func.py:9-31,62-73): the fused KV4 page write fills the retrieval pool with its
kmax / kmin statistics and the streaming pool's sink + local ring, streaming heads attend through the token-streaming
prefill kernel (ctx sink / local window) and dense heads through fused SDPA, and the MLP runs in chunks of
`chunk_prefill_size` rows.  `fill_random` instead fills the pages with valid random KV4 data and statistics, which is what the
decode kernels' cost depends on (the C3 benchmark).  CUDA graphs: one graph for steps that run the selector, one for steps
that reuse the choice.
"""
from __future__ import annotations

from typing import List, Optional

import torch

from . import lserve, prefill_attention
from .model import TOKENS_PER_BLOCK, ActivationBuffer, LlamaConfig, LlamaW4A8


class LServeDecoder:
    def __init__(self, cfg: LlamaConfig, retrieval_head_flags: List[List[int]], device="cuda", sink_tokens: int = 128,
                 local_tokens: int = 256, token_budget: int = 4096, selector_interval: int = 4, seed: int = 0,
                 ctx_sink_tokens: int = 128, ctx_local_tokens: int = 8192, chunk_prefill_size: int = 32000):
        assert len(retrieval_head_flags) == cfg.num_hidden_layers
        self.cfg, self.device = cfg, device
        self.m = LlamaW4A8(cfg, device, seed=seed)               # weights, small ops, lm_head
        self.sink, self.local = sink_tokens, local_tokens
        # prompt stage (omniserve/engine/arg_utils.py:82-88): streaming heads' prefill window and the MLP row chunk
        self.ctx_sink, self.ctx_local, self.chunk_prefill_size = ctx_sink_tokens, ctx_local_tokens, chunk_prefill_size
        self.sink_blk = (sink_tokens + TOKENS_PER_BLOCK - 1) // TOKENS_PER_BLOCK
        self.local_blk = (local_tokens + TOKENS_PER_BLOCK - 1) // TOKENS_PER_BLOCK + 1   # ring: one spare page (block_table_utils)
        self.sp = lserve.SparseDecodeConfig(dynamic_sparse_token_budget=token_budget, selector_update_interval=selector_interval,
                                            rotary_base=cfg.rope_theta)
        self.flags, self.rank, self.hr, self.hs, self.flags_host = [], [], [], [], []
        for fl in retrieval_head_flags:
            f = torch.tensor(fl, dtype=torch.int32)
            r = torch.zeros_like(f)
            r[f == 1] = torch.arange(int((f == 1).sum()), dtype=torch.int32)
            r[f == 0] = torch.arange(int((f == 0).sum()), dtype=torch.int32)
            self.flags.append(f.to(device)); self.rank.append(r.to(device)); self.flags_host.append(list(fl))
            self.hr.append(int(f.sum())); self.hs.append(int(len(fl) - f.sum()))

    def alloc(self, max_ctx: int):
        cfg, dev = self.cfg, self.device
        self.max_ctx = max_ctx
        self.pages = (max_ctx + TOKENS_PER_BLOCK - 1) // TOKENS_PER_BLOCK
        self.r_k, self.r_v, self.s_k, self.s_v, self.r_tab, self.s_tab = [], [], [], [], [], []
        g = torch.Generator().manual_seed(7)
        for li in range(cfg.num_hidden_layers):
            hr, hs = self.hr[li], self.hs[li]
            kb = hr * (64 * 64 + 64 * 4 + 2 * 4 * 128 * 2)          # nibbles + scales/zeros + kmax/kmin of 4 sub-chunks
            vb = hr * (64 * 64 + 64 * 4)
            rk = torch.zeros((self.pages, max(kb, 16)), dtype=torch.uint8, device=dev)
            rv = torch.zeros((self.pages, max(vb, 16)), dtype=torch.uint8, device=dev)
            perm = torch.randperm(self.pages, generator=g)
            tab = torch.empty((1, 2, self.pages), dtype=torch.int64)
            tab[0, 0] = rk.data_ptr() + perm * rk.shape[1]
            tab[0, 1] = rv.data_ptr() + perm * rv.shape[1]
            sp = self.sink_blk + self.local_blk
            sb = max(hs, 1) * (64 * 64 + 64 * 4)
            sk = torch.zeros((sp, sb), dtype=torch.uint8, device=dev)
            sv = torch.zeros((sp, sb), dtype=torch.uint8, device=dev)
            stab = torch.empty((1, 2, sp), dtype=torch.int64)
            stab[0, 0] = sk.data_ptr() + torch.arange(sp) * sb
            stab[0, 1] = sv.data_ptr() + torch.arange(sp) * sb
            self.r_k.append(rk); self.r_v.append(rv); self.s_k.append(sk); self.s_v.append(sv)
            self.r_tab.append(tab.to(dev) if hr else None); self.s_tab.append(stab.to(dev) if hs else None)
        m = self.m
        m.buf = ActivationBuffer(1, cfg.hidden_size, m.inter, m.q_size + 2 * m.kv_size, m.q_size, dev)
        m.batch = 1
        self.context_lens = torch.zeros((1,), dtype=torch.int32, device=dev)
        P = max(3, self.sp.dynamic_sparse_token_budget // TOKENS_PER_BLOCK)
        self.dyn = [torch.zeros((1, m.hq, P), dtype=torch.int32, device=dev) for _ in range(cfg.num_hidden_layers)]
        self.page_choice_valid = True     # False after a prefill: the next decode step must run the selector

    def kv_bytes(self) -> int:
        return sum(t.numel() for lst in (self.r_k, self.r_v, self.s_k, self.s_v) for t in lst)

    def fill_random(self, ctx: int):
        """Valid random pages for `ctx` cached tokens: any nibbles, positive scales, mid-range zero points, N(0,1) statistics."""
        for li in range(self.cfg.num_hidden_layers):
            for pool, h, stats in ((self.r_k[li], self.hr[li], True), (self.r_v[li], self.hr[li], False),
                                   (self.s_k[li], self.hs[li], False), (self.s_v[li], self.hs[li], False)):
                if h == 0:
                    continue
                pool.random_(0, 256)
                sz = pool[:, h * 4096: h * 4096 + h * 256].view(torch.float16)
                sz[:, : h * 64] = 0.1
                sz[:, h * 64:] = 7.5
                if stats:
                    pool[:, h * 4096 + h * 256:].view(torch.float16).normal_()
        self.context_lens.fill_(ctx)

    # ------------------------------------------------------------------ one decode step (bs = 1)
    @torch.no_grad()
    def decode_step(self, tokens: torch.Tensor, timestep: int, run_selector: bool):
        """`timestep` = cached tokens (host int baked into the launch configuration); the appended token goes to position
        `timestep`.  run_selector False reuses the page choice stored by the last selector step."""
        m, cfg = self.m, self.cfg
        b, ops = m.buf, m.ops
        if not run_selector and not self.page_choice_valid:
            raise RuntimeError("decode_step(run_selector=False) after prefill: no page choice for the new context yet")
        self.page_choice_valid = True
        self.context_lens.add_(1)
        hidden = m.embed_tokens[tokens]
        delta = None
        qh, sc, sm = b.quantized_hidden_states_buffer[:1], b.quantized_scale_buffer[:1], b.quantized_sum_buffer[:1]
        qkv, od = b.qkv_proj_act_buffer[:1], b.out_down_proj_act_buffer[:1]
        ha, hb = b.hidden_a[:1], b.hidden_b[:1]
        sparse = ops_sparse()
        for li, ly in enumerate(m.layers):
            h1 = m._norm_quant(qh, hidden, delta, ha, ly["input_layernorm"], sm, sc)
            ly["qkv_proj"](qh, sc, sm, qkv)
            q3 = qkv[:, : m.q_size].view(1, m.hq, cfg.head_dim)
            k3 = qkv[:, m.q_size: m.q_size + m.kv_size].view(1, m.hkv, cfg.head_dim)
            v3 = qkv[:, m.q_size + m.kv_size:].view(1, m.hkv, cfg.head_dim)
            hr, hs = self.hr[li], self.hs[li]
            args = (q3, k3, v3, self.r_tab[li], self.s_tab[li], self.flags[li], self.rank[li], self.context_lens, self.sink,
                    self.local, self.sink_blk, self.local_blk, hr, hs, timestep, self.sp)
            if run_selector and hr:
                sel = lserve.dynamic_select_topk_pages(*args)
                if sel.shape == self.dyn[li].shape:
                    self.dyn[li].copy_(sel)
                else:   # context within the token budget: every page, fewer than the budget's (eager steps only)
                    self.dyn[li] = sel
            attn = sparse.single_query_attention(
                q3, k3, v3, self.r_tab[li], self.s_tab[li], self.flags[li], self.rank[li], self.dyn[li] if hr else None,
                self.context_lens, None, self.sp.memory_max_len, TOKENS_PER_BLOCK, hr * cfg.head_dim // 2, hs * cfg.head_dim // 2,
                self.sink, self.local, self.sink_blk, self.local_blk, hr, hs, timestep, cfg.head_dim, cfg.rope_theta, 1.0, True, True,
                True, self.sp.sub_chunk_size, hr * cfg.head_dim, self.sp.multiblock_switch).reshape(1, m.q_size)
            qa = b.quantized_attn_buffer[:1]
            ops.fused_kernels.invoke_quant_fuse_sum(qa, attn, sm, sc)
            ly["o_proj"](qa, sc, sm, od)
            h2 = m._norm_quant(qh, h1, od, hb, ly["post_attention_layernorm"], sm, sc)
            gu = b.gate_up_proj_act_buffer[:1]
            ly["gate_up_proj"](qh, sc, sm, gu)
            qm = b.quantized_mlp_act_buffer[:1]
            ops.activation_ops.silu_and_mul_quant(qm, gu, sm, sc)
            ly["down_proj"](qm, sc, sm, od)
            hidden, delta = h2, od
        self.last_decode_state = (hidden, delta)
        return m._sample(hidden, delta)

    # ------------------------------------------------------------------ prompt (context) stage, bs = 1
    @torch.no_grad()
    def prefill(self, tokens: torch.Tensor, sparse_prefill: bool = True):
        """Run the prompt `tokens` (int64 [L], L <= max_ctx) through every layer, fill both page pools and return the next
        token.  sparse_prefill False gives every head the dense causal prefill mask (the reference's sparse_prefill_mode
        off); the pools are written the same way either way.  The activations are allocated for this call (L rows; the
        MLP intermediates `chunk_prefill_size` rows) and released after it."""
        from .backend import fused_attention_fine_grained_dense as wr
        m, cfg = self.m, self.cfg
        ops, dev = m.ops, self.device
        T = int(tokens.numel())
        if not 0 < T <= self.max_ctx:
            raise ValueError(f"prompt of {T} tokens: must be 1 .. max_ctx = {self.max_ctx}")
        Dh, H = cfg.head_dim, cfg.hidden_size
        C = max(1, min(self.chunk_prefill_size, T))
        f16, i8 = torch.float16, torch.int8
        qh = torch.empty((T, H), dtype=i8, device=dev)
        sc = torch.empty((T,), dtype=f16, device=dev)
        sm = torch.empty((T,), dtype=f16, device=dev)
        qkv = torch.empty((T, m.q_size + 2 * m.kv_size), dtype=f16, device=dev)
        qa = torch.empty((T, m.q_size), dtype=i8, device=dev)
        od = torch.empty((T, H), dtype=f16, device=dev)
        ha = torch.empty((T, H), dtype=f16, device=dev)
        hb = torch.empty((T, H), dtype=f16, device=dev)
        gu = torch.empty((C, 2 * m.inter), dtype=f16, device=dev)
        qm = torch.empty((C, m.inter), dtype=i8, device=dev)
        sl = torch.tensor([T], dtype=torch.int32, device=dev)
        cu = torch.tensor([0, T], dtype=torch.int32, device=dev)
        pad = wr.compute_padding_offsets(cu, T, T)
        g = m.hq // m.hkv
        sinfo = [self.ctx_sink, self.ctx_local] * m.hq
        hidden, delta = m.embed_tokens[tokens], None
        for li, ly in enumerate(m.layers):
            hr, hs = self.hr[li], self.hs[li]
            h1 = m._norm_quant(qh, hidden, delta, ha, ly["input_layernorm"], sm, sc)
            ly["qkv_proj"](qh, sc, sm, qkv)
            # RoPE in place + KV4 pages of both pools (streaming ring with the DECODE sink / local, as the reference) + kmax / kmin
            wr.apply_bias_rope_update_kv_cache_pool(
                qkv, sl, sl if hs else None, pad, self.r_tab[li], self.s_tab[li], self.flags[li], self.rank[li], m.hq, m.hkv, T,
                TOKENS_PER_BLOCK, hr * Dh // 2, hs * Dh // 2, self.sink, self.local, self.sink_blk, self.local_blk, hr, hs, Dh,
                cfg.rope_theta, 1.0, 8192, True, True, True, tokens_per_sub_chunk=self.sp.sub_chunk_size)
            q3 = qkv[:, : m.q_size].view(T, m.hq, Dh)
            k3 = qkv[:, m.q_size: m.q_size + m.kv_size].view(T, m.hkv, Dh)
            v3 = qkv[:, m.q_size + m.kv_size:].view(T, m.hkv, Dh)
            if sparse_prefill and hs:
                mask = [-1 if int(f) == 0 else 0 for f in self.flags_host[li] for _ in range(g)]
                attn = prefill_attention.token_streaming_attn_func(q3, k3, v3, cu, cu, mask, sinfo, T, T)
            else:   # the reference's head_mask_type=None branch: dense causal attention for every head
                with prefill_attention._fused_sdpa():
                    attn = prefill_attention.make(cu, T, m.hq, m.hkv, Dh)(q3, k3, v3)
            attn = attn.reshape(T, m.q_size)
            if m.act_sum:
                ops.fused_kernels.invoke_quant_fuse_sum(qa, attn, sm, sc)
            else:
                ops.fused_kernels.invoke_quant(qa, attn, sc)
            del attn
            ly["o_proj"](qa, sc, sm, od)
            h2 = m._norm_quant(qh, h1, od, hb, ly["post_attention_layernorm"], sm, sc)
            for c0 in range(0, T, C):      # llama_w4a8_unpad.py:89-111: the MLP in chunks of chunk_prefill_size rows
                c1 = min(T, c0 + C)
                n = c1 - c0
                ly["gate_up_proj"](qh[c0:c1], sc[c0:c1], sm[c0:c1], gu[:n])
                ops.activation_ops.silu_and_mul_quant(qm[:n], gu[:n], sm[c0:c1] if m.act_sum else None, sc[c0:c1])
                ly["down_proj"](qm[:n], sc[c0:c1], sm[c0:c1], od[c0:c1])
            hidden, delta = h2, od
        self.last_hidden = torch.add(hidden[T - 1:], delta[T - 1:])     # hidden state of the last prompt row
        nxt = m._sample(self.last_hidden)
        self.context_lens.fill_(T)
        self.page_choice_valid = False     # llama_w4a8_unpad.py:278-281: the first decode step re-runs the selector
        return nxt


def ops_sparse():
    from .backend import fused_attention_fine_grained_sparse
    return fused_attention_fine_grained_sparse


class LServeDecodeGraphs:
    """Two CUDA graphs: a step that runs the page selector and a step that reuses the cached choice (timestep is baked into
    launch configurations, so the graphs are captured at the bench's context length)."""

    def __init__(self, dec: LServeDecoder, timestep: int):
        self.dec = dec
        dev = dec.device
        self.tokens = torch.zeros((1,), dtype=torch.int64, device=dev)
        self.out = torch.zeros((1,), dtype=torch.int64, device=dev)
        saved = dec.context_lens.clone()
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            for sel in (True, False):
                self.out.copy_(dec.decode_step(self.tokens.clone(), timestep, sel))
                dec.context_lens.copy_(saved)
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        self.graphs = {}
        for sel in (True, False):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                nxt = dec.decode_step(self.tokens, timestep, sel)
                self.out.copy_(nxt)
                self.tokens.copy_(nxt)
                dec.context_lens.copy_(saved)      # the bench re-runs the same position: keep the context length fixed
            self.graphs[sel] = g
        torch.cuda.synchronize()

    def step(self, run_selector: bool):
        self.graphs[run_selector].replay()
        return self.out
