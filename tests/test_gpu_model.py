"""-m gpu: the host-side model runner (call order of llama_w4a8_unpad.py) over the C ABI ops."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _mk(ops=None, fuse=True, group=-1):
    from omniserve_b200.model import LlamaConfig, LlamaW4A8
    cfg = LlamaConfig.tiny(group_size=group)
    m = LlamaW4A8(cfg, "cuda", ops=ops, fuse_silu_quant=fuse)
    m.alloc(batch=3, max_ctx=192, max_tokens=3 * 70)
    return cfg, m


def _prompts(cfg):
    g = torch.Generator().manual_seed(1)
    return torch.randint(0, cfg.vocab_size, (70 + 33 + 64,), generator=g).cuda(), [70, 33, 64]


@pytest.mark.parametrize("group", [-1, 128])
def test_graph_replay_equals_eager(group):
    from omniserve_b200.model import DecodeGraph
    cfg, m1 = _mk(group=group)
    toks, lens = _prompts(cfg)
    f1 = m1.prefill(toks, lens)
    m1.prepare_decode()
    eager = []
    t = f1.clone()
    for _ in range(4):
        t = m1.decode_step(t, 192)
        eager.append(t.clone())
    cfg, m2 = _mk(group=group)
    f2 = m2.prefill(toks, lens)
    assert torch.equal(f1, f2)
    g = DecodeGraph(m2, 192)
    g.tokens.copy_(f2)
    for i in range(4):
        g.step()
        torch.cuda.synchronize()
        assert torch.equal(g.out, eager[i]), f"step {i}"
    assert m2.context_lens.tolist() == [74, 37, 68]
    for a, b in zip(m1.kv.k_pools, m2.kv.k_pools):
        assert torch.equal(a, b)


def test_fused_silu_quant_equals_two_kernel_chain():
    cfg, m1 = _mk(fuse=True)
    cfg, m2 = _mk(fuse=False)
    toks, lens = _prompts(cfg)
    assert torch.equal(m1.prefill(toks, lens), m2.prefill(toks, lens))
    assert torch.equal(m1.last_hidden, m2.last_hidden)


def test_whole_stack_vs_reference_kernels():
    """Same weights, same prompts through the reference's rebuilt kernels (oracle/_ref, or their recorded outputs) and
    ours."""
    from tests.gpu_util import ref_module, reference_outputs
    from omniserve_b200.model import Ops
    cfg, ours = _mk(fuse=False)
    toks, lens = _prompts(cfg)
    a = ours.prefill(toks, lens)

    def run():
        cfg, ref = _mk(ops=Ops(ref_module), fuse=False)
        ref.prefill(toks, lens)
        res = {"prefill_hidden": ref.last_hidden.float(), "v_pages_layer0": ref.kv.v_pools[0].clone()}   # before decode appends
        ref.prepare_decode()
        ref.decode_step(a.clone(), 192)
        res["decode_hidden"] = ref.last_decode_state[0].float() + ref.last_decode_state[1].float()
        return res
    r = reference_outputs("model_tiny_prefill_decode", ref_module("qgemm_w4a8_per_chn") is not None, run,
                          whole=("v_pages_layer0",))
    x, y = r.pair("prefill_hidden", ours.last_hidden.float())
    assert np.abs(x - y).max() <= 2e-2 * r.absmax("prefill_hidden")      # two layers of fp16 / int8-rounding drift
    # V pages byte-identical would need identical hidden states; compare the first layer's pages instead
    x, y = r.pair("v_pages_layer0", ours.kv.v_pools[0])
    assert (x != y).mean() < 2e-3
    ours.prepare_decode()
    ours.decode_step(a.clone(), 192)
    ho = ours.last_decode_state[0].float() + ours.last_decode_state[1].float()
    x, y = r.pair("decode_hidden", ho)
    assert np.abs(x - y).max() <= 3e-2 * r.absmax("decode_hidden")


def test_reference_op_chain_equals_fused_production_path_bit_for_bit():
    """GPU half of the boundary proof (tests/test_ref_callers_cpu.py is the CPU half): model.py restricted to the
    reference's op set issues the call sequence recorded from the reference's own LlamaDecoderLayer
    (tests/golden/ref_layer_trace.json), and its results -- prefill hidden states, sampled ids, KV pages, decode hidden
    states -- equal the fused production path (add+norm+quant, silu*mul+quant, attention+quant in one launch each) bit for bit."""
    import json
    import os
    from omniserve_b200 import _lib as L
    from tests.ref_trace_worker import ReferenceOpsOnly
    cfg, fused = _mk()
    cfg, plain = _mk(ops=ReferenceOpsOnly(), fuse=False)
    assert fused.fuse_add_norm and fused.fuse_attn_quant and not plain.fuse_add_norm and not plain.fuse_attn_quant
    toks, lens = _prompts(cfg)
    # record the C-ABI entry points the unfused path goes through (pass-through wrapper around the real library)
    real, names = L.lib(), []

    class Tap:
        def __getattr__(self, n):
            f = getattr(real, n)
            if not n.startswith("ob_"):
                return f

            def g(*a):
                names.append(n)
                return f(*a)
            return g
    saved = L.lib
    L.lib = lambda: Tap()
    try:
        b = plain.prefill(toks, lens)
        n_prefill = len(names)
        plain.prepare_decode()
        tb = plain.decode_step(b.clone(), 192)
    finally:
        L.lib = saved
    a = fused.prefill(toks, lens)
    assert torch.equal(a, b) and torch.equal(fused.last_hidden, plain.last_hidden)
    fused.prepare_decode()
    ta = fused.decode_step(a.clone(), 192)
    torch.cuda.synchronize()
    assert torch.equal(ta, tb)
    ha = fused.last_decode_state[0].float() + fused.last_decode_state[1].float()
    hb = plain.last_decode_state[0].float() + plain.last_decode_state[1].float()
    assert torch.equal(ha, hb)
    for x, y in zip(fused.kv.k_pools + fused.kv.v_pools, plain.kv.k_pools + plain.kv.v_pools):
        assert torch.equal(x, y)
    # per layer, the unfused path's entry points are those of the reference's own layer, in order
    fx = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_layer_trace.json")))["traces"]
    per_layer_prefill = [c[0] for c in fx["prefill"]["calls"]]
    per_layer_decode = [c[0] for c in fx["decode"]["calls"]]
    L_ = cfg.num_hidden_layers
    pre = [n for n in names[:n_prefill] if n not in ("ob_compute_padding_offsets", "ob_rms_norm")]
    dec = [n for n in names[n_prefill:] if n != "ob_rms_norm"]
    assert pre == per_layer_prefill * L_, pre
    assert dec == per_layer_decode * L_, dec
