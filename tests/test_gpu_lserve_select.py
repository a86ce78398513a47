"""-m gpu: LServe page statistics (a11), page selector (a9) and the dynamic-sparse decode loop built from them,
through the C ABI, against the oracle and the reference's own kernels rebuilt for sm_100 (oracle/_ref, or their
recorded outputs in tests/golden/ref_kernels.npz) (sparse_utils/ContextPool, sparse_utils/KVPageSelector)."""
import numpy as np
import pytest
import torch

from tests.gpu_util import assert_k_pool_equal, qkv_views, ref_module, reference_outputs, t

pytestmark = pytest.mark.gpu


def _case(lens, H, seed, extra=1):
    from oracle import kv4
    rng = np.random.default_rng(seed)
    n_pages = sum((l + 63) // 64 for l in lens) + extra
    cache = kv4.PagedKV4(n_pages, H, 128, k_stats_subchunks=4)
    perm = rng.permutation(n_pages)
    bt = np.zeros((len(lens), max((l + 63) // 64 for l in lens)), np.int64)
    c = 0
    for b, l in enumerate(lens):
        for j in range((l + 63) // 64):
            bt[b, j] = perm[c]
            c += 1
    return cache, bt, rng


def _ptrs(cache, bt):
    kpool, vpool = t(cache.k_pool), t(cache.v_pool)
    B, P = bt.shape
    p = np.zeros((B, 2, P), np.int64)
    p[:, 0] = kpool.data_ptr() + bt * cache.k_page_bytes
    p[:, 1] = vpool.data_ptr() + bt * cache.v_page_bytes
    return kpool, vpool, t(p)


@pytest.mark.parametrize("lens", [(70, 33), (1, 16, 17), (1024, 999), (64,)])
def test_paged_min_max_pool_bit_exact(lens):
    from omniserve_b200.backend import fused_attention_ctx_pool as op
    from oracle import kv4
    H_in, idx = 5, np.array([3, 1], np.int32)
    cache, bt, rng = _case(lens, 2, seed=sum(lens))
    cache.k_pool[:] = rng.integers(0, 256, cache.k_pool.shape, dtype=np.uint8)   # everything but the pooled rows must survive
    keys = rng.standard_normal((sum(lens), H_in, 128)).astype(np.float16)
    cu = np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)
    kpool, _, ptrs = _ptrs(cache, bt)
    op.paged_min_max_pool(t(keys), ptrs, t(cu), t(idx), max(lens), 16, 64, 2 * 64, True)
    torch.cuda.synchronize()
    kv4.paged_min_max_pool(cache, bt, keys, lens, 16, pooling_heads_idx=idx)
    np.testing.assert_array_equal(kpool.cpu().numpy(), cache.k_pool)
    ref = ref_module("fused_attention_ctx_pool")

    def run():
        kpool2, _, ptrs2 = _ptrs(cache, bt)
        kpool2.view(torch.uint8)[:] = 7
        ref.paged_min_max_pool(t(keys), ptrs2, t(cu), t(idx), max(lens), 16, 64, 2 * 64, True)
        torch.cuda.synchronize()
        return {"k_pool": kpool2}
    r = reference_outputs(f"ctx_pool_{'_'.join(map(str, lens))}", ref is not None, run)
    # compare only the statistics the reference wrote (its pool was filled with 7s first)
    mine, a = r.pair("k_pool", kpool)
    wrote = a != 7
    np.testing.assert_array_equal(a[wrote], mine[wrote])
    assert r.stat("bytes_written", lambda ref_: (ref_["k_pool"] != 7).sum()) >= 2 * 2 * 256 * sum((l + 15) // 16 for l in lens) * 0.95


def _selector_args(tq, tk, tv, ptrs, flags, rank, lens_t, Hkv_r, timestep):
    return (tq, tk, tv, ptrs, None, flags, rank, None, lens_t, None, 1 << 20, 64, Hkv_r * 64, 0, 0, 0, 0, 0, Hkv_r, 0,
            timestep, 128, 500000.0, 1.0, True, True, True, 16, Hkv_r * 128, 1000000)


@pytest.mark.parametrize("lens,group", [((200, 200), 4), ((1030,), 4), ((130, 130, 130), 1), ((777,), 8), ((200, 137), 2)])
def test_page_selector_scores(lens, group):
    from omniserve_b200.backend import fused_attention_selector as op
    from oracle import kv4
    Hkv = 2
    Hq = Hkv * group
    flags_np = np.array([1, 0], np.int32) if group == 2 else np.array([1, 1], np.int32)
    rank_np = np.array([0, 0], np.int32) if group == 2 else np.array([1, 0], np.int32)   # kv head 0 lives in row 1
    Hr = int(flags_np.sum())
    cache, bt, rng = _case(lens, Hr, seed=sum(lens) + group)
    keys = rng.standard_normal((sum(l - 1 for l in lens), Hr, 128)).astype(np.float16)
    kv4.paged_min_max_pool(cache, bt, keys, [l - 1 for l in lens], 16)
    q = rng.standard_normal((len(lens), Hq, 128)).astype(np.float16)
    k = rng.standard_normal((len(lens), Hkv, 128)).astype(np.float16)
    v = rng.standard_normal((len(lens), Hkv, 128)).astype(np.float16)
    _, tq, tk, tv = qkv_views(q, k, v)
    kpool, _, ptrs = _ptrs(cache, bt)
    timestep = max(lens) - 1
    lens_t = t(np.asarray(lens, np.int32))
    args = _selector_args(tq, tk, tv, ptrs, t(flags_np), t(rank_np), lens_t, Hr, timestep)
    out = op.single_query_page_selector(*args)
    torch.cuda.synchronize()
    exp = kv4.page_selector(q, cache, bt, lens, timestep, 128, 500000.0, retrieval_flags=flags_np, head_rank=rank_np,
                            n_kv_heads=Hkv)
    got = out.cpu().numpy()
    assert got.shape == exp.shape
    g32, e32 = got.astype(np.float32), exp.astype(np.float32)
    # same fp16 operation order as the reference; the rotated q may differ in the last fp16 bit of a few elements
    # (fp32 sincosf vs numpy), so: >= 99 % of the scores bit-identical, all within 2e-3 of the score scale
    assert (got == exp).mean() >= 0.99
    assert np.abs(g32 - e32).max() <= 2e-3 * max(1.0, np.abs(e32).max())
    np.testing.assert_array_equal((g32 == 0), (e32 == 0))     # zero rows / padding in the same places



@pytest.mark.parametrize("lens,group", [((200, 200), 4), ((1030,), 4), ((777,), 8)])
def test_page_selector_scores_vs_reference_kernel(lens, group, tmp_path):
    """Row a9 second opinion: the reference's OWN selector kernel (oracle/_ref, unmodified) on the same inputs.  It is run
    in a subprocess with oracle/ref_launch_shim.c preloaded: the reference launches it with 0 bytes of dynamic shared
    memory although the kernel stages the rotated query in `extern __shared__` (KVPageSelectorTemplate.hpp:834,1001-1053
    vs :1345-1347), which faults on sm_100; the shim supplies the missing bytes, the kernel itself is untouched."""
    import os
    import subprocess
    import sys
    from omniserve_b200.backend import fused_attention_selector as op
    from oracle import kv4
    from tests.gpu_util import REF_DIR, ROOT
    shim = os.path.join(ROOT, "oracle", "_ref", "libref_launch_shim.so")
    live = os.path.exists(os.path.join(REF_DIR, "fused_attention_selector.so")) and os.path.exists(shim)
    Hkv = 2
    Hq = Hkv * group
    flags_np, rank_np = np.array([1, 1], np.int32), np.array([1, 0], np.int32)
    Hr = 2
    cache, bt, rng = _case(lens, Hr, seed=sum(lens) + group + 1)
    keys = rng.standard_normal((sum(l - 1 for l in lens), Hr, 128)).astype(np.float16)
    kv4.paged_min_max_pool(cache, bt, keys, [l - 1 for l in lens], 16)
    q = rng.standard_normal((len(lens), Hq, 128)).astype(np.float16)
    k = rng.standard_normal((len(lens), Hkv, 128)).astype(np.float16)
    v = rng.standard_normal((len(lens), Hkv, 128)).astype(np.float16)
    timestep = max(lens) - 1
    def run():
        inp, outp = str(tmp_path / "in.npz"), str(tmp_path / "out.npz")
        np.savez(inp, k_pool=cache.k_pool, bt=bt, k_page_bytes=cache.k_page_bytes, q=q, k=k, v=v, flags=flags_np, rank=rank_np,
                 lens=np.asarray(lens, np.int32), timestep=timestep, Hr=Hr)
        env = dict(os.environ, LD_PRELOAD=shim)
        r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "ref_selector_worker.py"), inp, outp], env=env,
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, f"reference selector failed even with the shared-memory shim:\n{r.stdout[-1500:]}\n{r.stderr[-1500:]}"
        return {"out": np.load(outp)["out"]}
    rec = reference_outputs(f"selector_{'_'.join(map(str, lens))}_g{group}", live, run)
    _, tq, tk, tv = qkv_views(q, k, v)
    kpool, _, ptrs = _ptrs(cache, bt)
    out = op.single_query_page_selector(*_selector_args(tq, tk, tv, ptrs, t(flags_np), t(rank_np), t(np.asarray(lens, np.int32)),
                                                        Hr, timestep))
    torch.cuda.synchronize()
    got, ref_out = rec.pair("out", out)
    g32, r32 = got.astype(np.float32), ref_out.astype(np.float32)
    # the reference rotates q with fast-math sin/cos (ours: accurate sincosf), so a few scores differ in the last bits
    print(f"\nselector vs reference kernel lens={lens} group={group}: identical={np.mean(got == ref_out):.4f} "
          f"max|d|={np.abs(g32 - r32).max():.3e} scale={np.abs(r32).max():.3e}")
    assert np.abs(g32 - r32).max() <= 4e-3 * max(1.0, np.abs(r32).max())
    assert (got == ref_out).mean() >= 0.90
    np.testing.assert_array_equal((g32 == 0), (r32 == 0))


def test_dynamic_sparse_decode_loop_end_to_end():
    """prefill statistics -> selector -> top-k -> sparse attention (+ statistics update on append), several steps,
    against the oracle driving the same loop with the reference's Python page choice."""
    from omniserve_b200 import lserve
    from oracle import kv4
    B, Hq, Hkv = 1, 8, 2
    L0, steps, budget = 700, 5, 256        # 700 cached tokens > budget -> the selector path is taken
    lens0 = [L0]
    cache, bt, rng = _case([L0 + steps + 1], Hkv, seed=9)
    ks, _ = kv4.fill_random(cache, bt, lens0, rng)
    kv4.paged_min_max_pool(cache, bt, ks[0], lens0, 16)       # the fp16 keys that were quantised = post-RoPE keys
    cfg = lserve.SparseDecodeConfig(dynamic_sparse_token_budget=budget, selector_update_interval=2)
    kpool, vpool, ptrs = _ptrs(cache, bt)
    flags, rank = t(np.ones(Hkv, np.int32)), t(np.arange(Hkv, dtype=np.int32))
    cached = None
    for s in range(steps):
        ctx = L0 + s                                           # cached tokens before this step
        q = rng.standard_normal((B, Hq, 128)).astype(np.float16)
        k = rng.standard_normal((B, Hkv, 128)).astype(np.float16)
        v = rng.standard_normal((B, Hkv, 128)).astype(np.float16)
        _, tq, tk, tv = qkv_views(q, k, v)
        lens = np.asarray([ctx + 1], np.int32)
        out, cached_new = lserve.sparse_decode_attention(tq, tk, tv, ptrs, None, flags, rank, t(lens), 0, 0, 0, 0, Hkv, 0,
                                                         ctx, cfg, cached)
        torch.cuda.synchronize()
        if ctx % cfg.selector_update_interval == 0 or cached is None:
            stats = kv4.page_selector(q, cache, bt, lens, ctx, 128, 500000.0)
            exp_idx = kv4.select_topk_pages(stats, ctx, budget)
            got_idx = cached_new.cpu().numpy()
            assert got_idx.shape == exp_idx.shape == (B, Hq, budget // 64)
            assert (got_idx[..., -1] == (ctx - 1) // 64).all()
            # same page sets up to near-ties of the fp16 scores
            same = np.mean([len(set(got_idx[0, h]) & set(exp_idx[0, h])) / got_idx.shape[-1] for h in range(Hq)])
            assert same >= 0.9
        cached = cached_new
        dyn = cached.cpu().numpy()

        def positions(b, hq, tl):
            pos = []
            P = dyn.shape[-1]
            for j in range(P):
                n = 64 if j < P - 1 else (tl - 1) % 64 + 1
                pos.extend(range(int(dyn[b, hq, j]) * 64, int(dyn[b, hq, j]) * 64 + n))
            return np.asarray(pos, np.int64)
        ref = kv4.decode_attention(q, k, v, cache, bt, lens, 128, 500000.0, mimic=False, positions_fn=positions,
                                   update_stats_sub_chunk=16).astype(np.float32)
        got = out.cpu().numpy().astype(np.float32)
        assert np.abs(got - ref).max() <= 2e-3 * np.abs(ref).max()
        assert_k_pool_equal(kpool, cache)
        np.testing.assert_array_equal(vpool.cpu().numpy(), cache.v_pool)
        # keep the oracle's statistics in lock-step with the device's (they may differ in the last fp16 bit), so that
        # a one-ulp difference cannot flip a later page choice
        cache.k_pool[:] = kpool.cpu().numpy()


def test_selector_full_size_properties():
    """BASELINE config 3 scale (256K context, bs=1, 4 retrieval kv heads of 8, 32 q heads): statistics of random pages,
    properties instead of the loop oracle: (i) rows of streaming heads are zero, (ii) every score bounds q.k of every
    key a sub-chunk could hold, checked on sampled sub-chunks, (iii) the pitch/padding is the host's."""
    from omniserve_b200.backend import fused_attention_selector as op
    from oracle import kv4
    ctx = 262144
    Hq, Hkv, Hr = 32, 8, 4
    n_pages = ctx // 64
    flags_np = np.array([1, 0, 1, 0, 1, 0, 1, 0], np.int32)
    rank_np = np.array([0, 0, 1, 1, 2, 2, 3, 3], np.int32)
    page_bytes = Hr * 64 * 64 + Hr * 64 * 4 + 2 * 4 * Hr * 128 * 2
    g = torch.Generator(device="cuda").manual_seed(0)
    pool = torch.zeros((n_pages, page_bytes), dtype=torch.uint8, device="cuda")
    stats = pool[:, Hr * 64 * 64 + Hr * 64 * 4:].view(torch.float16).view(n_pages, 2, 4, Hr * 128)
    centre = torch.randn((n_pages, 1, 4, Hr * 128), generator=g, device="cuda")
    spread = torch.rand((n_pages, 1, 4, Hr * 128), generator=g, device="cuda")
    stats[:, 0:1] = (centre + spread).half()
    stats[:, 1:2] = (centre - spread).half()
    perm = torch.randperm(n_pages, generator=g, device="cuda")
    ptrs = torch.zeros((1, 2, n_pages), dtype=torch.int64, device="cuda")
    ptrs[0, 0] = pool.data_ptr() + perm * page_bytes
    q = torch.randn((1, Hq, 128), generator=g, device="cuda").half()
    k = torch.randn((1, Hkv, 128), generator=g, device="cuda").half()
    v = torch.randn((1, Hkv, 128), generator=g, device="cuda").half()
    lens_t = torch.tensor([ctx + 1], dtype=torch.int32, device="cuda")
    out = op.single_query_page_selector(*_selector_args(q, k, v, ptrs, t(flags_np), t(rank_np), lens_t, Hr, ctx))
    torch.cuda.synchronize()
    assert out.shape == (1, Hq, ctx // 16)
    o = out[0].float().cpu().numpy()
    for hq in range(Hq):
        if flags_np[hq // 4] == 0:
            assert not o[hq].any()
    q_r = kv4.rope_neox(q[0].cpu().numpy(), ctx, 128, 500000.0).astype(np.float64)
    st = stats.cpu().numpy()
    pm = perm.cpu().numpy()
    rng = np.random.default_rng(0)
    for _ in range(64):
        hq = int(rng.integers(0, Hq))
        if flags_np[hq // 4] == 0:
            continue
        sc = int(rng.integers(0, ctx // 16))
        page, sub = pm[sc // 4], sc % 4
        r = rank_np[hq // 4]
        kmax = st[page, 0, sub, r * 128:(r + 1) * 128].astype(np.float64)
        kmin = st[page, 1, sub, r * 128:(r + 1) * 128].astype(np.float64)
        bound = np.maximum(q_r[hq] * kmax, q_r[hq] * kmin).sum()
        assert abs(o[hq, sc] - bound) <= 4e-3 * abs(bound) + 0.1
        key = kmin + (kmax - kmin) * rng.random(128)           # any key inside the box
        assert (key * q_r[hq]).sum() <= o[hq, sc] + 4e-3 * abs(bound) + 0.1
