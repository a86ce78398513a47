"""-m gpu: LServe masks of the decode attention (SURVEY section 8 row a8): static streaming heads (sink + local ring
pages) and dynamic page selection, against the oracle with the reference's index semantics
(.../fused_attention_fine_grained/sparse_attention/decoderMaskedMultiheadAttentionTemplate.hpp:1559-1598,1631-1655;
ring mapping common/kvCacheUtils.h:117-126)."""
import numpy as np
import pytest
import torch

from tests.gpu_util import qkv_views, ref_module, reference_outputs, t

pytestmark = pytest.mark.gpu
TOL = 2e-3
NORTH_STAR = 1e-3


def _vs_reference_kernel(tag, got, exact, r):
    """Row a8 pinning: the same case through the REFERENCE's rebuilt kernel (oracle/_ref, or its recorded outputs `r`).
    Our distance to exact arithmetic must not exceed the reference's own (or the 1e-3 north-star tolerance, whichever is
    larger), and the two kernels must agree to 3e-3 of the output scale."""
    sc = np.abs(exact).max()
    e_ours = np.abs(got - exact).max() / sc
    e_ref = r.stat("err_vs_exact", lambda ref: np.abs(ref["out"].astype(np.float32) - exact).max() / sc)
    a, b = r.pair("out", got)
    d = np.abs(a - b.astype(np.float32)).max() / sc
    print(f"\n{tag}: |ours-exact|={e_ours:.3e} |ref-exact|={e_ref:.3e} |ours-ref|={d:.3e}")
    assert e_ours <= max(e_ref, NORTH_STAR)
    assert d <= 3e-3


def _ring(blk, sink_blk, local_blk):
    return blk if blk < sink_blk else sink_blk + (blk - sink_blk) % local_blk


def _fill_stream(cache, table, L, sink_blk, local_blk, rng):
    """Write tokens 0..L-1 of every head in order through the ring mapping (older local pages get overwritten)."""
    from oracle import kv4
    k = rng.standard_normal((L, cache.H, cache.Dh)).astype(np.float16)
    v = rng.standard_normal((L, cache.H, cache.Dh)).astype(np.float16)
    qk, sk, zk = kv4.kv4_quant(k)
    qv, sv, zv = kv4.kv4_quant(v)
    for pos in range(L):
        page, slot = int(table[_ring(pos >> 6, sink_blk, local_blk)]), pos & 63
        cache.data("k", page)[:, slot, :] = kv4.pack_nibbles(qk[pos]); cache.scales("k", page)[:, slot] = sk[pos]; cache.zeros("k", page)[:, slot] = zk[pos]
        cache.data("v", page)[:, slot, :] = kv4.pack_nibbles(qv[pos]); cache.scales("v", page)[:, slot] = sv[pos]; cache.zeros("v", page)[:, slot] = zv[pos]


def _ptrs(cache, tables):
    kpool, vpool = t(cache.k_pool), t(cache.v_pool)
    B, P = tables.shape
    p = np.zeros((B, 2, P), np.int64)
    p[:, 0] = kpool.data_ptr() + tables * cache.k_page_bytes
    p[:, 1] = vpool.data_ptr() + tables * cache.v_page_bytes
    return kpool, vpool, t(p)


@pytest.mark.parametrize("lens", [(500, 130), (40, 1000), (385, 386)])
def test_streaming_heads_sink_plus_local_ring(lens):
    from omniserve_b200.backend import fused_attention_fine_grained_dense as op
    from oracle import kv4
    rng = np.random.default_rng(sum(lens))
    B, Hq, Hkv, Dh = len(lens), 8, 2, 128
    sink, local, sink_blk, local_blk = 128, 256, 2, 5
    P = sink_blk + local_blk
    cache = kv4.PagedKV4(B * P, Hkv, Dh)
    tables = rng.permutation(B * P).reshape(B, P)
    maxblk = (max(lens) >> 6) + 1
    virt = np.zeros((B, maxblk), np.int64)   # logical block -> physical page through the ring
    for b, L in enumerate(lens):
        _fill_stream(cache, tables[b], L - 1, sink_blk, local_blk, rng)
        for blk in range(maxblk):
            virt[b, blk] = tables[b, _ring(blk, sink_blk, local_blk)]
    q = rng.standard_normal((B, Hq, Dh)).astype(np.float16)
    k = rng.standard_normal((B, Hkv, Dh)).astype(np.float16)
    v = rng.standard_normal((B, Hkv, Dh)).astype(np.float16)
    kpool, vpool, ptrs = _ptrs(cache, tables)
    _, tq, tk, tv = qkv_views(q, k, v)
    flags = t(np.zeros(Hkv, np.int32))           # every kv head is a streaming head
    rank = t(np.arange(Hkv, dtype=np.int32))
    out = op.single_query_attention(tq, tk, tv, None, ptrs, flags, rank, t(np.asarray(lens, np.int32)), None, 2048, 64,
                                    0, Hkv * Dh // 2, sink, local, sink_blk, local_blk, 0, Hkv, max(lens) - 1, 128,
                                    500000.0, 1.0, True, True, True, 2048)
    torch.cuda.synchronize()

    def positions(b, hq, tl):
        n_valid = min(sink + local - 1, tl)
        gap = tl - n_valid
        return np.array([i if i < sink else i + gap for i in range(n_valid)], dtype=np.int64)
    pools0 = (cache.k_pool.copy(), cache.v_pool.copy())
    ref = kv4.decode_attention(q, k, v, cache, virt, lens, 128, 500000.0, mimic=False, positions_fn=positions).astype(np.float32)
    got = out.cpu().numpy().astype(np.float32)
    assert np.abs(got - ref).max() <= TOL * np.abs(ref).max()
    np.testing.assert_array_equal(kpool.cpu().numpy(), cache.k_pool)   # append went through the ring mapping
    np.testing.assert_array_equal(vpool.cpu().numpy(), cache.v_pool)
    rm = ref_module("fused_attention_fine_grained_dense")

    def run():
        cache.k_pool[:], cache.v_pool[:] = pools0
        kpool2, vpool2, ptrs2 = _ptrs(cache, tables)
        o2 = rm.single_query_attention(tq, tk, tv, None, ptrs2, flags, rank, t(np.asarray(lens, np.int32)), None, 2048, 64,
                                       0, Hkv * Dh // 2, sink, local, sink_blk, local_blk, 0, Hkv, max(lens) - 1, 128,
                                       500000.0, 1.0, True, True, True, 2048)
        torch.cuda.synchronize()
        return {"out": o2, "k_pool": kpool2, "v_pool": vpool2}
    r = reference_outputs(f"lserve_streaming_{'_'.join(map(str, lens))}", rm is not None, run,
                          bases={"k_pool": pools0[0], "v_pool": pools0[1]})
    _vs_reference_kernel(f"streaming heads lens={lens}", got, ref, r)
    a, b = r.pair("v_pool", vpool)
    assert (a != b).mean() == 0     # V bytes identical; K differs only through RoPE intrinsics
    a, b = r.pair("k_pool", kpool)
    assert (a != b).mean() < 1e-3


@pytest.mark.parametrize("lens,P", [((700, 300), 4), ((1281, 1025), 9), ((64, 65), 1), ((2100, 2300), 4), ((4500, 4400), 64)])
def test_dynamic_page_selection(lens, P):
    from omniserve_b200.backend import fused_attention_fine_grained_sparse as op
    from oracle import kv4
    from tests.gpu_util import assert_k_pool_equal, device_tables, make_kv_case
    B, Hq, Hkv = len(lens), 8, 2
    # the sparse op also folds the appended key into the K pages' kmax / kmin statistics (4 sub-chunks of 16 tokens)
    cache, bt, q, k, v = make_kv_case(B, Hq, Hkv, lens, seed=P * 100 + sum(lens), k_stats_subchunks=4)
    rng = np.random.default_rng(P)
    for pg in range(cache.P):   # non-trivial stored statistics so that the max / min with the new key is exercised
        kmax, kmin = cache.kstats(pg)
        kmax[:] = rng.standard_normal(kmax.shape).astype(np.float16)
        kmin[:] = rng.standard_normal(kmin.shape).astype(np.float16)
    dyn = np.zeros((B, Hq, P), np.int32)
    for b, L in enumerate(lens):
        newest = (L - 2) // 64 if L >= 2 else 0     # page of the last cached token
        for h in range(Hq):
            others = rng.permutation(max(newest, 1))[: P - 1] if newest > 0 else np.zeros(P - 1, np.int64)
            if len(others) < P - 1:
                others = np.resize(others, P - 1)
            dyn[b, h, : P - 1] = others
            dyn[b, h, P - 1] = newest
    kpool, vpool, ptrs = device_tables(cache, bt)
    _, tq, tk, tv = qkv_views(q, k, v)
    flags = t(np.ones(Hkv, np.int32))
    rank = t(np.arange(Hkv, dtype=np.int32))
    out = op.single_query_attention(tq, tk, tv, ptrs, None, flags, rank, t(dyn), t(np.asarray(lens, np.int32)), None, 8192,
                                    64, Hkv * 64, 0, 0, 0, 0, 0, Hkv, 0, max(lens) - 1, 128, 500000.0, 1.0, True, True, True,
                                    16, Hkv * 128, 2048)
    torch.cuda.synchronize()

    def positions(b, hq, tl):
        if tl <= 0:
            return np.zeros(0, np.int64)
        pos = []
        for j in range(P):
            n = 64 if j < P - 1 else (tl - 1) % 64 + 1
            pos.extend(range(int(dyn[b, hq, j]) * 64, int(dyn[b, hq, j]) * 64 + n))
        return np.asarray(pos, np.int64)
    pools0 = (cache.k_pool.copy(), cache.v_pool.copy())
    ref = kv4.decode_attention(q, k, v, cache, bt, lens, 128, 500000.0, mimic=False, positions_fn=positions,
                               update_stats_sub_chunk=16).astype(np.float32)
    got = out.cpu().numpy().astype(np.float32)
    assert np.abs(got - ref).max() <= TOL * np.abs(ref).max()
    assert_k_pool_equal(kpool, cache, max_pos=max(lens))   # nibbles, scales, zeros exact; kmax / kmin to the last fp16 bits
    np.testing.assert_array_equal(vpool.cpu().numpy(), cache.v_pool)
    rm = ref_module("fused_attention_fine_grained_sparse")
    # The reference dispatches its SMEM_PRELOAD variant below timestep 2048 (sparse_attention/fused_attention.cpp:
    # smem_preload_switch), whose K loop asserts tokens_per_block % 128 == 0 -- with 64-token pages it can only run its
    # dynamic-page path at timestep >= 2048 (LServe only selects pages beyond the 4096-token budget anyway).  Its multi-block
    # split also misbehaves for small page counts at long contexts (observed on B200: ctx 4500, P = 9 -> 18 % away from exact
    # arithmetic while ours is 4e-4 away), so the long cases use LServe's operating point P = 64 (budget 4096 tokens).
    if max(lens) - 1 >= 2048:
        def run():
            cache.k_pool[:], cache.v_pool[:] = pools0
            kpool2, vpool2, ptrs2 = device_tables(cache, bt)
            # memory_max_seqlen must cover the context (the reference sizes its logits buffer from it)
            o2 = rm.single_query_attention(tq, tk, tv, ptrs2, None, flags, rank, t(dyn), t(np.asarray(lens, np.int32)), None,
                                           8192, 64, Hkv * 64, 0, 0, 0, 0, 0, Hkv, 0, max(lens) - 1, 128, 500000.0, 1.0, True,
                                           True, True, 16, Hkv * 128, 2048)
            torch.cuda.synchronize()
            return {"out": o2, "k_pool": kpool2, "v_pool": vpool2}
        r = reference_outputs(f"lserve_dynamic_{'_'.join(map(str, lens))}_P{P}", rm is not None, run,
                              bases={"k_pool": pools0[0], "v_pool": pools0[1]})
        _vs_reference_kernel(f"dynamic pages lens={lens} P={P}", got, ref, r)
        a, b = r.pair("v_pool", vpool)
        assert (a != b).mean() == 0
        a, b = r.pair("k_pool", kpool)
        assert (a != b).mean() < 2e-3   # incl. the kmax / kmin fold of the appended (fast-math RoPE) key


def test_mixed_retrieval_and_streaming_heads_with_rank_table():
    from omniserve_b200.backend import fused_attention_fine_grained_dense as op
    from oracle import kv4
    from tests.gpu_util import device_tables, make_kv_case
    lens = (450, 300)
    B, Hq, Hkv, Dh = 2, 8, 4, 128
    sink, local, sink_blk, local_blk = 64, 128, 1, 3
    flags_np = np.array([1, 0, 0, 1], np.int32)      # kv heads 0,3 retrieval (ranks 0,1); 1,2 streaming (ranks 0,1)
    rank_np = np.array([0, 0, 1, 1], np.int32)
    rng = np.random.default_rng(77)
    # retrieval pool: 2 heads
    rc, rbt, q, _, _ = make_kv_case(B, Hq, 2, lens, seed=5)
    Ps = sink_blk + local_blk
    sc = kv4.PagedKV4(B * Ps, 2, Dh)
    stab = rng.permutation(B * Ps).reshape(B, Ps)
    maxblk = (max(lens) >> 6) + 1
    virt = np.zeros((B, maxblk), np.int64)
    for b, L in enumerate(lens):
        _fill_stream(sc, stab[b], L - 1, sink_blk, local_blk, rng)
        for blk in range(maxblk):
            virt[b, blk] = stab[b, _ring(blk, sink_blk, local_blk)]
    k = rng.standard_normal((B, Hkv, Dh)).astype(np.float16)
    v = rng.standard_normal((B, Hkv, Dh)).astype(np.float16)
    rk, rv, rptrs = device_tables(rc, rbt)
    sk, sv_, sptrs = _ptrs(sc, stab)
    _, tq, tk, tv = qkv_views(q, k, v)
    out = op.single_query_attention(tq, tk, tv, rptrs, sptrs, t(flags_np), t(rank_np), t(np.asarray(lens, np.int32)), None,
                                    2048, 64, 2 * 64, 2 * 64, sink, local, sink_blk, local_blk, 2, 2, max(lens) - 1, 128,
                                    500000.0, 1.0, True, True, True, 2048)
    torch.cuda.synchronize()
    got = out.cpu().numpy().astype(np.float32)

    def spos(b, hq, tl):
        n_valid = min(sink + local - 1, tl)
        gap = tl - n_valid
        return np.array([i if i < sink else i + gap for i in range(n_valid)], dtype=np.int64)
    # oracle per pool: feed the pool's own two kv heads (+ their 2 query heads each)
    g = Hq // Hkv
    for pool_heads, cache, table, pf in (([0, 3], rc, rbt, None), ([1, 2], sc, virt, spos)):
        qh = np.concatenate([q[:, h * g:(h + 1) * g] for h in pool_heads], axis=1)
        ref = kv4.decode_attention(qh, k[:, pool_heads], v[:, pool_heads], cache, table, lens, 128, 500000.0, mimic=False,
                                   positions_fn=pf).astype(np.float32)
        mine = np.concatenate([got[:, h * g:(h + 1) * g] for h in pool_heads], axis=1)
        assert np.abs(mine - ref).max() <= TOL * np.abs(ref).max()
    np.testing.assert_array_equal(rk.cpu().numpy(), rc.k_pool)
    np.testing.assert_array_equal(sk.cpu().numpy(), sc.k_pool)


def _random_pages(cache, rng):
    """Valid random KV4 pages without running the per-token quantiser: any nibble bytes, positive scales, mid-range
    zero points, N(0,1) statistics.  (The attention reads whatever the pages hold.)"""
    for pool in (cache.k_pool, cache.v_pool):
        pool[:, :cache.data_bytes] = rng.integers(0, 256, (cache.P, cache.data_bytes), dtype=np.uint8)
        n = cache.sz_bytes // 4
        sz = pool[:, cache.data_bytes:cache.data_bytes + cache.sz_bytes].view(np.float16)
        sz[:, :n] = rng.uniform(0.05, 0.15, (cache.P, n)).astype(np.float16)
        sz[:, n:] = rng.uniform(6.0, 9.0, (cache.P, n)).astype(np.float16)
    if cache.stats_bytes:
        st = cache.k_pool[:, cache.data_bytes + cache.sz_bytes:].view(np.float16)
        st[:] = rng.standard_normal(st.shape).astype(np.float16)


def test_c3_shape_256k_context_head_split_from_fixture():
    """BASELINE config 3 shape: Llama-3-8B-Instruct-Gradient-1048k, bs = 1, 262 144 cached tokens, dynamic budget 4096
    tokens -> P = 64 pages per retrieval q-head, streaming heads attend 128 sink + 256 local tokens through the ring,
    retrieval / streaming head split of one layer from the reference's attn_patterns TSV at static_sparsity 0.5
    (tests/golden/head_split_llama3_8b_1048k_s50.json, derived by tests/golden/make_head_split.py with the rule of
    omniserve/attn_config.py:113-150).  Checked against the exact oracle and the reference's sparse kernel."""
    import json
    import os
    from omniserve_b200.backend import fused_attention_fine_grained_sparse as op
    from oracle import kv4
    from tests.gpu_util import ROOT, device_tables
    fx = json.load(open(os.path.join(ROOT, "tests", "golden", "head_split_llama3_8b_1048k_s50.json")))
    layer = 9
    flags_np = np.asarray(fx["retrieval_head_flags"][layer], np.int32)
    rank_np = np.asarray(fx["head_rank_table"][layer], np.int32)
    Hq, Hkv, Dh, g = 32, 8, 128, 4
    Hr, Hs = int(flags_np.sum()), int(Hkv - flags_np.sum())
    assert 0 < Hr < Hkv
    ctx, P = 262144, 64
    lens = [ctx + 1]
    sink, local, sink_blk, local_blk = 128, 256, 2, 5
    rng = np.random.default_rng(2025)
    n_pages = ctx // 64 + 1
    rc = kv4.PagedKV4(n_pages, Hr, Dh, k_stats_subchunks=4)
    _random_pages(rc, rng)
    rbt = rng.permutation(n_pages).reshape(1, n_pages)
    sc = kv4.PagedKV4(sink_blk + local_blk, Hs, Dh)
    _random_pages(sc, rng)
    stab = rng.permutation(sink_blk + local_blk).reshape(1, -1)
    blks = np.arange(n_pages)
    virt = stab[:, np.where(blks < sink_blk, blks, sink_blk + (blks - sink_blk) % local_blk)]
    dyn = np.zeros((1, Hq, P), np.int32)
    newest = (ctx - 1) // 64
    for h in range(Hq):
        dyn[0, h, :P - 1] = rng.choice(newest, P - 1, replace=False)
        dyn[0, h, P - 1] = newest
    q = rng.standard_normal((1, Hq, Dh)).astype(np.float16)
    k = rng.standard_normal((1, Hkv, Dh)).astype(np.float16)
    v = rng.standard_normal((1, Hkv, Dh)).astype(np.float16)
    _, tq, tk, tv = qkv_views(q, k, v)
    args = lambda rp, sp: (tq, tk, tv, rp, sp, t(flags_np), t(rank_np), t(dyn), t(np.asarray(lens, np.int32)), None,  # noqa: E731
                           1 << 20, 64, Hr * 64, Hs * 64, sink, local, sink_blk, local_blk, Hr, Hs, ctx, 128, 500000.0, 1.0,
                           True, True, True, 16, Hr * 128, 2048)
    rk, rv, rptrs = device_tables(rc, rbt)
    sk, sv_, sptrs = _ptrs(sc, stab)
    out = op.single_query_attention(*args(rptrs, sptrs))
    torch.cuda.synchronize()
    got = out.cpu().numpy().astype(np.float32)
    rm = ref_module("fused_attention_fine_grained_sparse")

    def run():
        rk2, rv2, rptrs2 = device_tables(rc, rbt)
        sk2, sv2, sptrs2 = _ptrs(sc, stab)
        o2 = rm.single_query_attention(*args(rptrs2, sptrs2))
        torch.cuda.synchronize()
        return {"out": o2}
    r = reference_outputs("lserve_c3_shape_262144", rm is not None, run)

    def rpos(b, hq_local, tl):      # hq_local indexes the q heads of the retrieval pool in pool order
        hq = r_q_heads[hq_local]
        pos = []
        for j in range(P):
            n = 64 if j < P - 1 else (tl - 1) % 64 + 1
            pos.extend(range(int(dyn[b, hq, j]) * 64, int(dyn[b, hq, j]) * 64 + n))
        return np.asarray(pos, np.int64)

    def spos(b, hq_local, tl):
        n_valid = min(sink + local - 1, tl)
        gap = tl - n_valid
        return np.array([i if i < sink else i + gap for i in range(n_valid)], dtype=np.int64)
    r_heads = [h for h in range(Hkv) if flags_np[h] == 1]
    s_heads = [h for h in range(Hkv) if flags_np[h] == 0]
    r_heads.sort(key=lambda h: rank_np[h])
    s_heads.sort(key=lambda h: rank_np[h])
    r_q_heads = [h * g + i for h in r_heads for i in range(g)]
    exact = np.zeros_like(got)
    for heads, cache, table, pf, kw in ((r_heads, rc, rbt, rpos, dict(update_stats_sub_chunk=16)), (s_heads, sc, virt, spos, {})):
        qh = np.concatenate([q[:, h * g:(h + 1) * g] for h in heads], axis=1)
        e = kv4.decode_attention(qh, k[:, heads], v[:, heads], cache, table, lens, 128, 500000.0, mimic=False,
                                 positions_fn=pf, **kw).astype(np.float32)
        for i, h in enumerate(heads):
            exact[:, h * g:(h + 1) * g] = e[:, i * g:(i + 1) * g]
    # At position 262 144 the fp32 rotation angle pos / base^(2i/d) carries ~1e-2 rad of rounding for the fastest dimension
    # pairs (one fp32 ulp of powf, times the position) on EVERY implementation -- this oracle, our kernel (accurate sincosf)
    # and the reference (fast-math __sinf / __cosf, far worse at such arguments) -- so q.k of the rotated new token, and with
    # it the output, agree to ~3e-3 rather than 1e-3; the cached (already rotated) keys are unaffected.
    assert np.abs(got - exact).max() <= 5e-3 * np.abs(exact).max()
    # the appended token went to page 4096 of the retrieval pool / through the ring in the streaming pool: V bytes are
    # not rotated and must be identical; of the K pools everything but the appended row must be untouched
    np.testing.assert_array_equal(rv.cpu().numpy(), rc.v_pool)
    np.testing.assert_array_equal(sv_.cpu().numpy(), sc.v_pool)
    new_r, new_s = int(rbt[0, ctx // 64]), int(virt[0, ctx // 64])
    gk, gs = rk.cpu().numpy(), sk.cpu().numpy()
    keep_r = np.ones(rc.P, bool); keep_r[new_r] = False
    keep_s = np.ones(sc.P, bool); keep_s[new_s] = False
    np.testing.assert_array_equal(gk[keep_r], rc.k_pool[keep_r])
    np.testing.assert_array_equal(gs[keep_s], sc.k_pool[keep_s])
    assert (gk[new_r] != rc.k_pool[new_r]).mean() < 0.02 and (gs[new_s] != sc.k_pool[new_s]).mean() < 0.02   # one token row
    sc_ = np.abs(exact).max()
    e_ref = r.stat("err_vs_exact", lambda ref: np.abs(ref["out"].astype(np.float32) - exact).max() / sc_)
    a, b = r.pair("out", got)
    d = np.abs(a - b.astype(np.float32)).max() / sc_
    print(f"\nC3 shape (256K ctx, P=64, TSV head split): |ours-exact|={np.abs(got - exact).max() / sc_:.3e} "
          f"|ref-exact|={e_ref:.3e} |ours-ref|={d:.3e}")
    assert np.abs(got - exact).max() / sc_ <= max(e_ref, 5e-3)
    assert d <= 5e-2


def test_lserve_decoder_graph_replay_equals_eager_small():
    """omniserve_b200/lserve_model.py (the C3 bench's model): graph-replayed sparse decode step == eager step, selector and
    reuse variants, on a small stack with a mixed retrieval / streaming head split."""
    from omniserve_b200.lserve_model import LServeDecodeGraphs, LServeDecoder
    from omniserve_b200.model import LlamaConfig
    cfg = LlamaConfig(hidden_size=1024, intermediate_size=2048, num_hidden_layers=2, num_attention_heads=8, num_key_value_heads=4,
                      vocab_size=2048)
    flags = [[1, 0, 1, 1], [0, 1, 1, 0]]
    ctx = 6000                                  # > the 4096-token budget: the selector path is taken
    outs = []
    for use_graph in (False, True):
        dec = LServeDecoder(cfg, flags, "cuda", token_budget=1024)
        dec.alloc(ctx + 64)
        torch.manual_seed(0)
        dec.fill_random(ctx)
        tok = torch.tensor([5], device="cuda")
        if use_graph:
            gr = LServeDecodeGraphs(dec, ctx)
            gr.tokens.copy_(tok)
            a = gr.step(True).clone()
            gr.tokens.copy_(tok)
            b = gr.step(False).clone()
        else:
            saved = dec.context_lens.clone()
            a = dec.decode_step(tok, ctx, True).clone()
            dec.context_lens.copy_(saved)
            b = dec.decode_step(tok, ctx, False).clone()
        torch.cuda.synchronize()
        outs.append((a, b, [d.clone() for d in dec.dyn]))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])
    for x, y in zip(outs[0][2], outs[1][2]):
        assert torch.equal(x, y)
        assert int(x[..., -1].min()) == (ctx - 1) // 64 == int(x[..., -1].max())
