"""-m gpu: the Mixtral mixture-of-experts stack -- routing, permutation and combine kernels against oracle/moe.py, the
device-offset grouped GEMM against the host-table one, CUDA-graph capture of the MoE block, batch independence, and the
tiny / Mixtral-8x7B-shape model (omniserve_b200/moe_model.py)."""
import numpy as np
import pytest
import torch

from tests.gpu_util import t

pytestmark = pytest.mark.gpu


def _distinct_logits(rng, T, E):
    """fp32 logits whose values within a row are distinct multiples of 1/16: every softmax gap is far above fp32 rounding."""
    grid = np.arange(-4 * E, 4 * E, dtype=np.float32) / 16.0
    return np.stack([rng.permutation(grid)[:E] for _ in range(T)]).astype(np.float32)


@pytest.mark.parametrize("T,E,k", [(37, 8, 2), (300, 8, 2), (5000, 64, 8), (1, 4, 4), (2100, 16, 1)])
def test_topk_sort_matches_oracle(T, E, k):
    from omniserve_b200.backend import moe_helpers as mh
    from oracle import moe
    rng = np.random.default_rng(T + E + k)
    lg = _distinct_logits(rng, T, E)
    off = torch.full((E + 1,), -7, dtype=torch.int32, device="cuda")
    w, ei, perm = mh.moe_topk_gating_softmax(t(lg), k, out_offsets=off)
    torch.cuda.synchronize()
    rw, rei = moe.topk_gating_softmax(lg, k)
    rperm, roff = moe.permutation(rei, E)
    np.testing.assert_array_equal(ei.cpu().numpy(), rei)
    np.testing.assert_allclose(w.cpu().numpy(), rw, rtol=2e-6, atol=1e-7)
    np.testing.assert_array_equal(perm.cpu().numpy(), rperm)
    np.testing.assert_array_equal(off.cpu().numpy(), roff)


def test_topk_exact_ties_go_to_the_lower_index():
    from omniserve_b200.backend import moe_helpers as mh
    lg = np.array([[1, 1, 1, 0, 0, 0, 0, 0], [0, 2, 0, 2, 0, 0, 0, 2], [0] * 8, [3, 0, 0, 0, 0, 0, 0, 3]], np.float32)
    w, ei, perm = mh.moe_topk_gating_softmax(t(lg), 2)
    torch.cuda.synchronize()
    assert ei.view(4, 2).tolist() == [[0, 1], [1, 3], [0, 1], [0, 7]]
    assert torch.equal(w.cpu(), torch.full((4, 2), 0.5))
    # stable within an expert: expert 0 holds (t0, s0), (t2, s0), (t3, s0) in that order
    assert perm.tolist()[:3] == [0, 4, 6]


def test_router_logits_match_oracle_and_are_row_independent():
    from omniserve_b200.backend import moe_helpers as mh
    from oracle import moe
    rng = np.random.default_rng(3)
    T, H, E = 97, 4096, 8
    x = rng.standard_normal((T, H)).astype(np.float16)
    g = (rng.standard_normal((E, H)) / 64).astype(np.float16)
    lg = mh.moe_router_logits(t(x), t(g))
    one = mh.moe_router_logits(t(x[40:41]), t(g))
    torch.cuda.synchronize()
    got = lg.cpu().numpy()
    ref = moe.router_logits(x, g)
    assert np.all(got == got.astype(np.float16).astype(np.float32))    # fp16-rounded values
    ulp = np.spacing(np.abs(ref).astype(np.float16)).astype(np.float32)
    assert np.all(np.abs(got - ref) <= ulp)
    assert (got == ref).mean() > 0.98
    np.testing.assert_array_equal(one.cpu().numpy(), got[40:41])


def test_expand_bit_exact_and_finalize_within_one_ulp():
    from omniserve_b200.backend import moe_helpers as mh
    from oracle import moe
    rng = np.random.default_rng(5)
    T, E, k, H = 45, 8, 2, 512
    lg = _distinct_logits(rng, T, E)
    w, ei, perm = mh.moe_topk_gating_softmax(t(lg), k)
    q = rng.integers(-128, 128, (T, H), dtype=np.int8)
    ss = rng.standard_normal(T).astype(np.float16)
    sc = rng.uniform(0.01, 0.05, T).astype(np.float16)
    qo, sso, sco, inv = mh.moe_expand_inputs_and_scales(t(q), t(ss), t(sc), perm)
    y = (rng.standard_normal((T * k, H)) * 3).astype(np.float16)
    out = mh.moe_finalize_routing(t(y), w, inv, T)
    torch.cuda.synchronize()
    rq, rss, rsc, rinv = moe.expand(q, ss, sc, perm.cpu().numpy(), k)
    np.testing.assert_array_equal(qo.cpu().numpy(), rq)
    np.testing.assert_array_equal(sso.cpu().numpy(), rss)
    np.testing.assert_array_equal(sco.cpu().numpy(), rsc)
    np.testing.assert_array_equal(inv.cpu().numpy(), rinv)
    ref = moe.finalize(y, w.cpu().numpy(), rinv, T).astype(np.float32)
    got = out.cpu().numpy().astype(np.float32)
    ulp = np.spacing(np.abs(ref).astype(np.float16)).astype(np.float32)
    assert np.all(np.abs(got - ref) <= ulp)


def _gemm_case(E, N, K, sizes, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    rows = sum(sizes)
    qw = torch.randint(-128, 128, (E, N, K // 2), generator=g, device="cuda", dtype=torch.int8)
    x = torch.randint(-127, 128, (rows, K), generator=g, device="cuda", dtype=torch.int8)
    s1 = (torch.rand((E, N), generator=g, device="cuda") * 0.01 + 0.005).half()
    szs = (s1.float() * 8).half()
    sa = (torch.rand(rows, generator=g, device="cuda") * 0.02 + 0.01).half()
    ss = torch.randn(rows, generator=g, device="cuda").half()
    off = torch.tensor([0] + list(np.cumsum(sizes)), dtype=torch.int32, device="cuda")
    return qw, x, s1, szs, sa, ss, off


@pytest.mark.parametrize("N,K", [(28672, 4096), (4096, 14336)])
@pytest.mark.parametrize("sizes,tokens", [((9, 7, 8, 6, 10, 8, 11, 5), 32),     # bs 32, top-2, every expert used
                                           ((20, 0, 0, 16, 0, 28, 0, 0), 32),    # empty experts
                                           ((64, 64, 0, 0, 0, 0, 0, 0), 64),     # skewed: two experts take all 64 tokens
                                           ((0, 0, 1, 0, 0, 1, 0, 0), 1)])       # one token
def test_device_offset_gemm_bit_identical_to_host_table(N, K, sizes, tokens):
    from omniserve_b200.backend import qgemm_w4a8_moe as op
    E = 8
    qw, x, s1, szs, sa, ss, off = _gemm_case(E, N, K, sizes, seed=N + sum(sizes))
    ref = op.moe_gemm_forward_cuda_api(x, qw, s1, sa, szs, ss, list(sizes))
    got = torch.full_like(ref, float("nan"))
    op.moe_gemm_forward_cuda_api_dev(x, qw, s1, sa, szs, ss, off, tokens, out=got)
    torch.cuda.synchronize()
    assert torch.equal(got, ref)


def _tiny_model(seed=0, **kw):
    from omniserve_b200.moe_model import MixtralConfig, MixtralW4A8
    return MixtralW4A8(MixtralConfig.tiny(**kw), "cuda", seed=seed)


def test_moe_block_graph_replay_equals_eager_under_changing_routing():
    m = _tiny_model()
    T = 32
    m.alloc(T, 256, T)
    H = m.cfg.hidden_size
    x = torch.empty((T, H), dtype=torch.float16, device="cuda")
    gen = torch.Generator(device="cuda").manual_seed(1)
    x.copy_(torch.randn((T, H), generator=gen, device="cuda").half())
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        m.moe_block(0, x, True)   # warm-up: tensor maps, launch attributes
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out_g = m.moe_block(0, x, True)
    seen = []
    for i in range(3):
        x.copy_((torch.randn((T, H), generator=gen, device="cuda") * (1 + i)).half())
        graph.replay()
        got = out_g.clone()
        offs = m.moe_buf.offsets.clone()
        eager = m.moe_block(0, x, True).clone()
        torch.cuda.synchronize()
        assert torch.equal(m.moe_buf.offsets, offs)
        assert torch.equal(got, eager)
        seen.append(tuple(offs.tolist()))
    assert len(set(seen)) > 1, "the replays did not see different routings"


def test_moe_block_is_batch_independent():
    m = _tiny_model(seed=2)
    T = 32
    m.alloc(T, 256, T)
    x = torch.randn((T, m.cfg.hidden_size), generator=torch.Generator(device="cuda").manual_seed(3), device="cuda").half()
    full = m.moe_block(1, x, True).clone()
    for i in (0, 13, 31):
        one = m.moe_block(1, x[i:i + 1].contiguous(), True).clone()
        torch.cuda.synchronize()
        assert torch.equal(one[0], full[i])


def test_moe_block_matches_oracle_on_the_models_own_inputs():
    """The block on the normed rows a real prefill fed it: routing, permutation and expand exact; each grouped GEMM within
    the GEMM tolerance of test_gpu_moe.py on its own inputs; silu * mul -> quant and the combine as the oracle chain.  The
    end to end bound is looser: the oracle's exact expf / division moves an INT8 activation code by one step here and there
    (oracle/act.py), and the second GEMM carries that into the output."""
    from oracle import act, moe, w4a8
    m = _tiny_model(seed=4)
    m.alloc(2, 256, 256)
    m.record_moe_inputs = []
    toks = torch.randint(0, m.cfg.vocab_size, (200,), generator=torch.Generator().manual_seed(4)).cuda()
    m.prefill(toks, [120, 80])
    torch.cuda.synchronize()
    recorded, m.record_moe_inputs = m.record_moe_inputs, None
    assert len(recorded) == m.cfg.num_hidden_layers
    k = m.cfg.num_experts_per_tok
    for dev_off in (False, True):
        for li, xn in recorded:
            xs = xn[:64] if dev_off else xn       # the device-offset path serves <= 64 tokens
            T = xs.shape[0]
            ly, mb = m.layers[li], m.moe_buf
            x = xs.cpu().numpy()
            out = m.moe_block(li, xs, dev_off).cpu().numpy().astype(np.float32)
            lg = mb.logits[:T].cpu().numpy()
            ref_lg = moe.router_logits(x, ly["gate"].cpu().numpy())
            assert np.all(np.abs(lg - ref_lg) <= np.spacing(np.abs(ref_lg).astype(np.float16)).astype(np.float32))
            w13 = tuple(a.cpu().numpy() for a in (ly["w1_w3"].qweight, ly["w1_w3"].s1_scales, ly["w1_w3"].s1_szeros))
            w2 = tuple(a.cpu().numpy() for a in (ly["w2"].qweight, ly["w2"].s1_scales, ly["w2"].s1_szeros))
            ref, st = moe.moe_block(x, ly["gate"].cpu().numpy(), w13, w2, k, logits=lg)
            n = T * k
            np.testing.assert_array_equal(mb.offsets.cpu().numpy(), st["offsets"])
            np.testing.assert_array_equal(mb.inv[:n].cpu().numpy(), st["inv"])
            q, sc, ss = (a[:n].cpu().numpy() for a in (mb.q_in, mb.scale_in, mb.sum_in))
            sizes = np.diff(st["offsets"])
            for got, (xq, xsc, xss), w in ((mb.gate_up[:n], (q, sc, ss), w13),
                                           (mb.y[:n], tuple(a[:n].cpu().numpy() for a in (mb.q_act, mb.scale_act, mb.sum_act)), w2)):
                r = w4a8.moe_gemm_per_chn(xq, w[0], w[1], xsc, w[2], xss, sizes)
                g = got.cpu().numpy()
                assert np.abs(g.astype(np.float32) - r.astype(np.float32)).max() <= 1e-3 * np.abs(r.astype(np.float32)).max()
                assert (g == r).mean() > 0.999
            qa, sa, _ = act.quant_fuse_sum(act.silu_and_mul(mb.gate_up[:n].cpu().numpy()))
            assert (np.abs(qa.astype(np.int32) - mb.q_act[:n].cpu().numpy()) <= 1).all()
            fin = moe.finalize(mb.y[:n].cpu().numpy(), st["weights"], st["inv"], T).astype(np.float32)
            assert np.all(np.abs(out - fin) <= np.spacing(np.abs(fin).astype(np.float16)).astype(np.float32))
            ref = ref.astype(np.float32)
            err = np.abs(out - ref).max()
            print(f"\nlayer {li} ({'device' if dev_off else 'host'} offsets): max |moe block - oracle| {err:.3e} of "
                  f"{np.abs(ref).max():.3e}")
            assert err <= 2e-2 * np.abs(ref).max()


def test_tiny_model_graph_decode_equals_eager_decode():
    from omniserve_b200.model import DecodeGraph
    B, L = 4, 40
    a, b = _tiny_model(seed=5), _tiny_model(seed=5)
    toks = torch.randint(0, 1024, (B * L,), generator=torch.Generator().manual_seed(5)).cuda()
    for m in (a, b):
        m.alloc(B, 256, B * L)
    ta = a.prefill(toks, [L] * B)
    tb = b.prefill(toks, [L] * B)
    assert torch.equal(ta, tb)
    g = DecodeGraph(a, max_timestep=L + 8)
    g.tokens.copy_(ta)
    tok = tb
    for _ in range(4):
        out = g.step().clone()
        ha, da = a.last_decode_state
        tok = b.decode_step(tok, L + 8)
        hb, db = b.last_decode_state
        torch.cuda.synchronize()
        assert torch.equal(out, tok)
        assert torch.equal(ha, hb) and torch.equal(da, db)
    assert torch.equal(a.context_lens, b.context_lens)


def test_tiny_model_prefill_then_decode_matches_longer_prefill():
    n = 300
    toks = torch.randint(0, 1024, (n + 1,), generator=torch.Generator().manual_seed(6)).cuda()
    a, b = _tiny_model(seed=6), _tiny_model(seed=6)
    a.alloc(1, 512, 512)
    b.alloc(1, 512, 512)
    a.prefill(toks[:n], [n])
    a.decode_step(toks[n:n + 1], n)
    h, d = a.last_decode_state
    dec_h = (h.float() + d.float())[0]
    b.prefill(toks, [n + 1])
    torch.cuda.synchronize()
    ref = b.last_hidden.float()[n]
    err, scale = (dec_h - ref).abs().max().item(), ref.abs().max().item()
    print(f"\nprefill(n)+decode vs prefill(n+1): {err:.3e} of {scale:.3e}")
    assert int(a.context_lens[0]) == n + 1
    assert err <= 3e-2 * scale


def test_decode_batch_over_64_raises():
    m = _tiny_model()
    m.alloc(65, 128, 65)
    with pytest.raises(ValueError):
        m.decode_step(torch.zeros(65, dtype=torch.int64, device="cuda"), 1)


def test_mixtral_8x7b_shape_prefill_and_graph_decode_smoke():
    from omniserve_b200.model import DecodeGraph
    from omniserve_b200.moe_model import MixtralConfig, MixtralW4A8
    cfg = MixtralConfig.mixtral_8x7b()
    B, L = 32, 1024
    m = MixtralW4A8(cfg, "cuda", seed=0, device_init=True)
    try:
        m.alloc(B, L + 64, B * L)
        toks = torch.randint(0, cfg.vocab_size, (B * L,), generator=torch.Generator().manual_seed(0)).cuda()
        nxt = m.prefill(toks, [L] * B)
        assert torch.isfinite(m.last_hidden).all()
        g = DecodeGraph(m, max_timestep=L + 8)
        g.tokens.copy_(nxt)
        for _ in range(4):
            out = g.step()
        torch.cuda.synchronize()
        h, d = m.last_decode_state
        assert torch.isfinite(h).all() and torch.isfinite(d).all()
        assert int(out.min()) >= 0 and int(out.max()) < cfg.vocab_size
    finally:
        del m
        torch.cuda.empty_cache()
