"""-m gpu: static per-tensor INT8 KV pages (SURVEY.md section 8 row f4) -- fused_attention_per_tensor_{dense,sparse} vs
oracle/kv8.py and vs the reference's own fused_attention_per_tensor_dense kernels (oracle/_ref, or their recorded outputs).

Tolerance: the stored codes are consumed exactly (int8 -> fp16 is exact, fp32 accumulation), so the distance to the
EXACT-arithmetic oracle is bounded by the fp16 probability rounding: 2e-3 of the output scale, as for KV4
(tests/test_gpu_attention.py).  Page bytes of the appended token and of the prefill writer: bit-exact."""
import numpy as np
import pytest
import torch

from tests.gpu_util import device_tables, qkv_views, ref_module, reference_outputs, t

pytestmark = pytest.mark.gpu
TOL_EXACT = 2e-3
BASE = 500000.0


def _scales(kmax=4.5, vmax=4.5):
    sqo = np.asarray([kmax / 127.0, vmax / 127.0], np.float32)
    return sqo, (1.0 / sqo).astype(np.float32)


def _case(B, Hq, Hkv, lens, seed, extra_pages=2, sub=0):
    from oracle import kv8
    rng = np.random.default_rng(seed)
    n_pages = sum((l + 63) // 64 for l in lens) + extra_pages
    cache = kv8.PagedKV8(n_pages, Hkv, 128, sub)
    perm = rng.permutation(n_pages)
    bt = np.zeros((B, max((l + 63) // 64 for l in lens)), np.int64)
    c = 0
    for b, l in enumerate(lens):
        for j in range((l + 63) // 64):
            bt[b, j] = perm[c]; c += 1
    cache.k_pool[:, : cache.data_bytes] = rng.integers(0, 256, (n_pages, cache.data_bytes), dtype=np.uint8)
    cache.v_pool[:, : cache.data_bytes] = rng.integers(0, 256, (n_pages, cache.data_bytes), dtype=np.uint8)
    if sub:
        cache.k_pool[:, cache.data_bytes + cache.sz_bytes:] = rng.standard_normal(
            (n_pages, cache.stats_bytes // 2)).astype(np.float16).view(np.uint8)
    q = rng.standard_normal((B, Hq, 128)).astype(np.float16)
    k = rng.standard_normal((B, Hkv, 128)).astype(np.float16)
    v = rng.standard_normal((B, Hkv, 128)).astype(np.float16)
    return cache, bt, q, k, v


def _copy(cache):
    from oracle import kv8
    c = kv8.PagedKV8(cache.P, cache.H, cache.Dh, cache.n_sub)
    c.k_pool[:], c.v_pool[:] = cache.k_pool, cache.v_pool
    return c


def _run(B, Hq, Hkv, lens, seed, force_split=0):
    from omniserve_b200.backend import _attn_common as AC
    from oracle import kv8
    cache, bt, q, k, v = _case(B, Hq, Hkv, lens, seed)
    sqo, soq = _scales()
    kpool, vpool, ptrs = device_tables(cache, bt)
    _, tq, tk, tv = qkv_views(q, k, v)
    out = AC.single_query(tq, tk, tv, ptrs, None, None, None, None, t(np.asarray(lens, np.int32)), 64, Hkv, 0, 0, 0, 0, 0,
                          max(lens) - 1, 128, BASE, 1.0, force_split=force_split, kv8_scales=(t(sqo), t(soq)))
    torch.cuda.synchronize()
    got = out.cpu().numpy().astype(np.float32)
    c1 = _copy(cache)
    ref = kv8.decode_attention(q, k, v, c1, bt, lens, 128, BASE, sqo, soq).astype(np.float32)
    sc = np.abs(ref).max()
    assert not np.isnan(got).any()
    assert np.abs(got - ref).max() <= TOL_EXACT * sc, (np.abs(got - ref).max() / sc)
    np.testing.assert_array_equal(vpool.cpu().numpy(), c1.v_pool)          # appended V codes: no rotation -> bit exact
    kdiff = kpool.cpu().numpy() != c1.k_pool                               # K: fp32 RoPE last-bit differences move a code by 1
    assert kdiff.mean() < 1e-5
    d = np.abs(kpool.cpu().numpy().view(np.int8).astype(np.int32) - c1.k_pool.view(np.int8).astype(np.int32))
    assert d.max() <= 1


@pytest.mark.parametrize("Hq,Hkv", [(8, 2), (32, 8), (4, 4), (8, 1), (16, 8)])
def test_kv8_dense_gqa_groups(Hq, Hkv):
    _run(3, Hq, Hkv, (70, 200, 129), seed=Hq * 10 + Hkv)


def test_kv8_edge_lengths():
    _run(4, 8, 2, (1, 2, 64, 65), seed=1)
    _run(2, 8, 2, (63, 128), seed=2)


@pytest.mark.parametrize("split", [2, 3, 5])
def test_kv8_split_kv_merge(split):
    _run(2, 8, 2, (700, 333), seed=split, force_split=split)


def test_kv8_ragged_batch_c2_like():
    _run(6, 32, 8, (1024, 1100, 1535, 1, 300, 1279), seed=11)


def test_kv8_reference_named_ops_prefill_then_decode():
    """The reference's call sequence (ctx_update_kv.py:49-92 then decoding_attention.py:185-236) through the mirrored ops:
    prefill writer page bytes == oracle, then a decode step over what it wrote."""
    from omniserve_b200.backend import fused_attention_per_tensor_dense as op
    from oracle import kv8
    rng = np.random.default_rng(7)
    Hq, Hkv, Dh = 8, 2, 128
    lens = [70, 5, 130]
    T = sum(lens)
    n_pages = sum((l + 64) // 64 for l in lens)
    cache = kv8.PagedKV8(n_pages, Hkv, Dh)
    bt = np.zeros((3, 4), np.int64)
    perm = rng.permutation(n_pages)
    c = 0
    for b, l in enumerate(lens):
        for j in range((l + 64) // 64):
            bt[b, j] = perm[c]; c += 1
    qkv = rng.standard_normal((T, (Hq + 2 * Hkv) * Dh)).astype(np.float16)
    sqo, soq = _scales()
    kpool, vpool, ptrs = device_tables(cache, bt)
    tqkv, sl = t(qkv), t(np.asarray(lens, np.int32))
    cu = t(np.concatenate([[0], np.cumsum(lens)]).astype(np.int32))
    pad = op.compute_padding_offsets(cu, max(lens), T)
    op.apply_bias_rope_update_kv_cache(tqkv, t(soq), sl, None, pad, ptrs, None, None, None, Hq, Hkv, max(lens), 64, Hkv * Dh, 0,
                                       0, 0, 0, 0, Hkv, 0, 128, BASE, 1.0, 0, True, False, False)
    torch.cuda.synchronize()
    ref_qkv = qkv.copy()
    kv8.prefill_write(cache, bt, ref_qkv, lens, Hq, 128, BASE, soq)
    np.testing.assert_array_equal(vpool.cpu().numpy(), cache.v_pool)
    d = np.abs(kpool.cpu().numpy().view(np.int8).astype(np.int32) - cache.k_pool.view(np.int8).astype(np.int32))
    assert d.max() <= 1 and (d != 0).mean() < 1e-4
    # decode one token per sequence on top of the device-written pages
    cache.k_pool[:], cache.v_pool[:] = kpool.cpu().numpy(), vpool.cpu().numpy()
    q = rng.standard_normal((3, Hq, Dh)).astype(np.float16)
    k = rng.standard_normal((3, Hkv, Dh)).astype(np.float16)
    v = rng.standard_normal((3, Hkv, Dh)).astype(np.float16)
    _, tq, tk, tv = qkv_views(q, k, v)
    lens1 = [l + 1 for l in lens]
    out = op.single_query_attention(tq, tk, tv, t(sqo), t(soq), ptrs, None, None, None, t(np.asarray(lens1, np.int32)), None, 4096,
                                    64, Hkv * Dh, 0, 0, 0, 0, 0, Hkv, 0, max(lens), 128, BASE, 1.0, True, False, False, 2048)
    ref = kv8.decode_attention(q, k, v, cache, bt, lens1, 128, BASE, sqo, soq).astype(np.float32)
    assert np.abs(out.cpu().numpy().astype(np.float32) - ref).max() <= TOL_EXACT * np.abs(ref).max()
    with pytest.raises(NotImplementedError):   # the per-tensor path has no KV4 / zero-point variant
        op.single_query_attention(tq, tk, tv, t(sqo), t(soq), ptrs, None, None, None, None, None, 4096, 64, Hkv * Dh, 0, 0, 0, 0, 0,
                                  Hkv, 0, max(lens), 128, BASE, 1.0, True, True, True, 2048)


def test_kv8_sparse_streaming_and_dynamic_pages():
    """fused_attention_per_tensor_sparse: retrieval heads attend the chosen pages, streaming heads sink + local ring pages
    (index semantics as tests/test_gpu_lserve.py); the appended key is folded into the page statistics that sit behind the
    (unused) scale area."""
    from omniserve_b200.backend import fused_attention_per_tensor_sparse as op
    from oracle import kv8
    from oracle.kv4 import rope_neox
    rng = np.random.default_rng(5)
    B, Hq, Hkv, sub = 2, 8, 4, 16
    lens = [1501, 1411]
    flags = np.asarray([1, 0, 0, 1], np.int32)       # kv heads 0, 3 retrieval (ranks 0, 1); 1, 2 streaming (ranks 0, 1)
    rank = np.asarray([0, 0, 1, 1], np.int32)
    sink, local, sink_blk, local_blk = 64, 128, 1, 3
    rc, rbt, q, _, _ = _case(B, Hq, 2, lens, 3, sub=4)
    Ps = sink_blk + local_blk
    sc, _, _, _, _ = _case(1, 1, 2, [B * Ps * 64], 4, extra_pages=0)
    stab = rng.permutation(B * Ps).reshape(B, Ps)
    maxblk = (max(lens) >> 6) + 1
    virt = np.zeros((B, maxblk), np.int64)
    for b in range(B):
        for blk in range(maxblk):
            virt[b, blk] = stab[b, blk if blk < sink_blk else sink_blk + (blk - sink_blk) % local_blk]
    k = rng.standard_normal((B, Hkv, 128)).astype(np.float16)
    v = rng.standard_normal((B, Hkv, 128)).astype(np.float16)
    sqo, soq = _scales()
    rk, rv, rptr = device_tables(rc, rbt)
    sk, sv_, sptr = device_tables(sc, stab)
    P = 6
    dyn = np.zeros((B, Hq, P), np.int32)
    for b in range(B):
        npg = (lens[b] - 1) // 64 + 1
        for h in range(Hq):
            dyn[b, h, : P - 1] = np.sort(rng.choice(npg - 1, P - 1, replace=False))
            dyn[b, h, P - 1] = npg - 1
    _, tq, tk, tv = qkv_views(q, k, v)
    stats0 = []
    for b in range(B):
        a, c = rc.kstats(int(rbt[b, (lens[b] - 1) // 64]))
        stats0.append((a.copy(), c.copy()))
    out = op.single_query_attention(tq, tk, tv, t(sqo), t(soq), rptr, sptr, t(flags), t(rank), t(dyn),
                                    t(np.asarray(lens, np.int32)), None, 8192, 64, 2 * 128, 2 * 128, sink, local, sink_blk, local_blk,
                                    2, 2, max(lens) - 1, 128, BASE, 1.0, True, False, False, sub, 2 * 128, 2048)
    torch.cuda.synchronize()
    got = out.cpu().numpy().astype(np.float32)
    g = Hq // Hkv

    def spos(b, hq, tl):
        n_valid = min(sink + local - 1, tl)
        gap = tl - n_valid
        return np.array([i if i < sink else i + gap for i in range(n_valid)], dtype=np.int64)
    for pool_heads, cache, table, retr in (([0, 3], rc, rbt, True), ([1, 2], sc, virt, False)):
        qh = np.concatenate([q[:, h * g:(h + 1) * g] for h in pool_heads], axis=1)
        qidx = [h * g + i for h in pool_heads for i in range(g)]

        def rpos(b, hq_local, tl):
            return np.concatenate([np.arange(p_ * 64, min((p_ + 1) * 64, tl)) for p_ in dyn[b, qidx[hq_local]]])
        ref = kv8.decode_attention(qh, k[:, pool_heads], v[:, pool_heads], _copy(cache), table, lens, 128, BASE, sqo, soq,
                                   positions_fn=rpos if retr else spos, append=False).astype(np.float32)
        mine = got[:, qidx]
        assert np.abs(mine - ref).max() <= TOL_EXACT * np.abs(ref).max(), np.abs(mine - ref).max() / np.abs(ref).max()
    # statistics of the appended key (retrieval heads): element-wise max / min against the stored values
    kp = rk.cpu().numpy()
    o, n = rc.data_bytes + rc.sz_bytes, 4 * 2 * 128 * 2
    for b in range(B):
        tl = lens[b] - 1
        page, slot = int(rbt[b, tl // 64]), tl % 64
        gmax = kp[page, o: o + n].view(np.float16).reshape(4, 256)
        gmin = kp[page, o + n: o + 2 * n].view(np.float16).reshape(4, 256)
        for hk in (0, 3):
            kr = rope_neox(k[b, hk], tl, 128, BASE)
            sl = slice(rank[hk] * 128, rank[hk] * 128 + 128)
            em, en = np.maximum(stats0[b][0][slot // sub, sl], kr), np.minimum(stats0[b][1][slot // sub, sl], kr)
            assert np.abs(gmax[slot // sub, sl].astype(np.float32) - em.astype(np.float32)).max() <= 4e-3
            assert np.abs(gmin[slot // sub, sl].astype(np.float32) - en.astype(np.float32)).max() <= 4e-3
            code = kv8.kv8_quant(kr, soq[0])          # ... and its INT8 row landed in the page
            gotc = kp[page, : rc.data_bytes].view(np.int8).reshape(2, 64, 128)[rank[hk], slot]
            assert np.abs(gotc.astype(np.int32) - code.astype(np.int32)).max() <= 1


def test_kv8_vs_reference_kernels():
    """The reference's own per-tensor kernels (oracle/_ref, rebuilt for sm_100) on the same pages: prefill writer bytes equal
    ours; decode output within 3e-3 of the output scale of ours (the reference rounds dequantised values and probabilities
    to fp16; ours is closer to exact)."""
    ref = ref_module("fused_attention_per_tensor_dense")
    from omniserve_b200.backend import fused_attention_per_tensor_dense as ours
    from oracle import kv8
    rng = np.random.default_rng(17)
    Hq, Hkv, Dh = 32, 8, 128
    lens = [300, 77, 1030]
    B, T = len(lens), sum(lens)
    n_pages = sum((l + 64) // 64 for l in lens)
    sqo, soq = _scales()
    flags, rank = t(np.ones(Hkv, np.int32)), t(np.arange(Hkv, dtype=np.int32))
    pools = []
    for _ in range(2):
        cache = kv8.PagedKV8(n_pages, Hkv, Dh)
        bt = np.arange(n_pages, dtype=np.int64)
        btab = np.zeros((B, max((l + 64) // 64 for l in lens)), np.int64)
        c = 0
        for b, l in enumerate(lens):
            for j in range((l + 64) // 64):
                btab[b, j] = bt[c]; c += 1
        pools.append((cache, btab) + device_tables(cache, btab))
    qkv = rng.standard_normal((T, (Hq + 2 * Hkv) * Dh)).astype(np.float16)
    sl = t(np.asarray(lens, np.int32))
    cu = t(np.concatenate([[0], np.cumsum(lens)]).astype(np.int32))
    pad = ours.compute_padding_offsets(cu, max(lens), T)
    db = pools[0][0].data_bytes

    def prefill(mod, kp, vp, ptr):
        x = t(qkv)
        mod.apply_bias_rope_update_kv_cache(x, t(soq), sl, None, pad, ptr, None, flags, rank, Hq, Hkv, max(lens), 64, Hkv * Dh, 0,
                                            0, 0, 0, 0, Hkv, 0, 128, BASE, 1.0, 8192, True, False, False)   # max_positions != 0
        torch.cuda.synchronize()
        return kp.cpu().numpy().copy(), vp.cpu().numpy().copy()
    q = rng.standard_normal((B, Hq, Dh)).astype(np.float16)
    k = rng.standard_normal((B, Hkv, Dh)).astype(np.float16)
    v = rng.standard_normal((B, Hkv, Dh)).astype(np.float16)
    lens1 = t(np.asarray([l + 1 for l in lens], np.int32))

    def decode(mod, kp, vp, ptr, pages):
        kp.copy_(torch.from_numpy(pages[0]).cuda()); vp.copy_(torch.from_numpy(pages[1]).cuda())   # same pages for both
        _, tq, tk, tv = qkv_views(q, k, v)
        o = mod.single_query_attention(tq, tk, tv, t(sqo), t(soq), ptr, None, flags, rank, lens1, None, 4096, 64, Hkv * Dh, 0, 0, 0,
                                       0, 0, Hkv, 0, max(lens), 128, BASE, 1.0, True, False, False, 2048)
        torch.cuda.synchronize()
        return o.cpu().numpy().astype(np.float32)
    mine = prefill(ours, *pools[1][2:])

    def run():
        kp_ref, vp_ref = prefill(ref, *pools[0][2:])
        return {"k_data": kp_ref[:, :db], "v_data": vp_ref[:, :db], "out": decode(ref, *pools[0][2:], mine)}
    r = reference_outputs("kv8_300_77_1030", ref is not None, run)
    a, b = r.pair("v_data", mine[1][:, :db])
    np.testing.assert_array_equal(a, b)
    a, b = r.pair("k_data", mine[0][:, :db])
    dk = np.abs(a.view(np.int8).astype(np.int32) - b.view(np.int8).astype(np.int32))
    assert dk.max() <= 1 and (dk != 0).mean() < 1e-3
    got = decode(ours, *pools[1][2:], mine)
    sc = np.abs(got).max()
    a, b = r.pair("out", got)
    assert np.abs(a - b).max() <= 3e-3 * sc, np.abs(a - b).max() / sc
