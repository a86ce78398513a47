"""-m gpu: round-2 parity tightening (VERDICT r1 "What's weak" 1-3, ADVICE r1 PDL hazards).

* INT32 accumulators asserted as integers: with s1 = sa = 1, sz = 0 and |acc| <= 2048 the fp16 output IS the s32
  accumulator (every integer of that range is a fp16 number), for data-parallel tiles, stream-K (L2 bulk-reduce) and
  cluster split-K (DSMEM reduce-scatter), per-channel and per-group (incl. the 8-bit wrap of q*s2+z).
* attention error measured side by side: |reference kernel - exact| and |ours - exact| on the same inputs; ours must not
  be worse than the reference's own distance to exact arithmetic (north star: 1e-3 rel on the softmax tail).
* stream-ordered hazards: prefill KV write -> decode attention with NO host synchronisation in between.
"""
import numpy as np
import pytest
import torch

from tests.gpu_util import device_tables, make_kv_case, qkv_views, ref_module, reference_outputs, t

pytestmark = pytest.mark.gpu


# --------------------------------------------------------------------------------------------------------- GEMM
def _sparse_pm1(rng, M, K, nnz):
    a = np.zeros((M, K), np.int8)
    for m in range(M):
        idx = rng.choice(K, nnz, replace=False)
        a[m, idx] = rng.choice(np.array([-1, 1], np.int8), nnz)
    return a


def _launch(per_group, a, qw, z2, s2, s1, sa, szs, ssum, M, N, K, bn, mode, ctas):
    from omniserve_b200 import _lib as L
    out = torch.full((M, N), float("nan"), dtype=torch.float16, device="cuda")
    keep = [t(a), t(qw), t(s1), t(sa)]
    if per_group:
        keep += [t(z2), t(s2)]
        code = L.lib().ob_w4a8_gemm_ex(1, L.ptr(keep[0]), L.ptr(keep[1]), L.ptr(keep[4]), L.ptr(keep[5]), L.ptr(keep[2]),
                                       L.ptr(keep[3]), 0, 0, L.ptr(out), M, N, K, N, bn, mode, ctas, L.stream())
    else:
        keep += [t(szs), t(ssum)]
        code = L.lib().ob_w4a8_gemm_ex(0, L.ptr(keep[0]), L.ptr(keep[1]), 0, 0, L.ptr(keep[2]), L.ptr(keep[3]),
                                       L.ptr(keep[4]), L.ptr(keep[5]), L.ptr(out), M, N, K, N, bn, mode, ctas, L.stream())
    torch.cuda.synchronize()
    assert code == 0
    return out.cpu().numpy()


# (force_bn, force_mode, force_ctas): -1 auto, 0 data-parallel tiles, 1 stream-K (L2 bulk reduce), 2 cluster split-K (DSMEM),
# 3 decode kernel (w4a8_gemm_decode.cu: red.global.add.s32 split-K), M <= 64 only
SCHEDULES = [(0, -1, 0), (0, 0, 0), (0, 1, 0), (0, 1, 37), (0, 2, 2), (0, 2, 4), (0, 2, 8), (16, 1, 148), (128, 0, 5),
             (0, 3, 0), (0, 3, 37), (0, 3, 296), (64, 3, 100), (0, 3, 1)]


@pytest.mark.parametrize("M,N,K", [(64, 4096, 4096), (64, 512, 14336), (17, 256, 2048), (200, 1024, 1024)])
def test_int32_accumulators_exact_per_channel(M, N, K):
    from oracle import w4a8 as ow
    rng = np.random.default_rng(M + N + K)
    q = rng.integers(0, 16, (N, K), dtype=np.uint8)
    a = _sparse_pm1(rng, M, K, 128)                       # |acc| <= 128 * 15 = 1920 < 2048
    qw = ow.pack_w4(q)
    ones_n, ones_m = np.ones(N, np.float16), np.ones(M, np.float16)
    zero_n, junk_m = np.zeros(N, np.float16), rng.standard_normal(M).astype(np.float16)   # sz = 0 kills the sum term
    want = (a.astype(np.int64) @ q.astype(np.int64).T).astype(np.int32)
    assert np.abs(want).max() <= 2048
    for bn, mode, ctas in SCHEDULES:
        if (mode == 2 and (K // 128) < ctas) or (mode == 3 and M > 64):
            continue
        got = _launch(False, a, qw, None, None, ones_n, ones_m, zero_n, junk_m, M, N, K, bn, mode, ctas)
        np.testing.assert_array_equal(got.astype(np.int32), want, err_msg=f"schedule bn={bn} mode={mode} ctas={ctas}")
        assert (got == got.astype(np.int32)).all()


@pytest.mark.parametrize("M,N,K", [(64, 4096, 4096), (33, 256, 2048), (128, 512, 1024)])
def test_int32_accumulators_exact_per_group_with_byte_wrap(M, N, K):
    from oracle import w4a8 as ow
    rng = np.random.default_rng(M * 3 + N + K)
    q = rng.integers(0, 16, (N, K), dtype=np.uint8)
    ng = K // 128
    # level-2 scales / zeros chosen so that some byte products q*s2 exceed 255 (carry into the neighbour byte) and the
    # __vadd4 wraps: the oracle restates exactly that arithmetic (per_group/gemm_cuda.cu:289-329)
    s2 = rng.integers(1, 20, (N, ng)).astype(np.int64)
    z = rng.integers(0, 16, (N, ng)).astype(np.int64)
    s2p = ow.pack_s2(s2).astype(np.int8)
    z2p = (ow.pack_s2(-z) * ow.pack_s2(s2)).astype(np.int8)
    qw = ow.pack_w4(q)
    w8 = ow.dequant_per_group_w8(qw, z2p, s2p).astype(np.int64)
    a = _sparse_pm1(rng, M, K, 16)                        # |acc| <= 16 * 128 = 2048
    want = (a.astype(np.int64) @ w8.T).astype(np.int32)
    assert np.abs(want).max() <= 2048
    ones_n, ones_m = np.ones(N, np.float16), np.ones(M, np.float16)
    for bn, mode, ctas in SCHEDULES:
        if (mode == 2 and (K // 128) < ctas) or (mode == 3 and M > 64):
            continue
        got = _launch(True, a, qw, z2p, s2p, ones_n, ones_m, None, None, M, N, K, bn, mode, ctas)
        np.testing.assert_array_equal(got.astype(np.int32), want, err_msg=f"schedule bn={bn} mode={mode} ctas={ctas}")


# ---------------------------------------------------------------------------------------------------- attention
def _err(x, exact):
    return float(np.abs(x.astype(np.float32) - exact.astype(np.float32)).max() / np.abs(exact.astype(np.float32)).max())


NORTH_STAR = 1e-3


@pytest.mark.parametrize("lens", [(70, 200, 129), (1024, 1100, 1535), (1, 64, 65), (333,)])
def test_dense_attention_not_worse_than_reference_kernel(lens, record_property):
    """|ours - exact| <= max(|reference kernel - exact|, 1e-3): the reference's fp16 rounding points (fp16 dequant, fp16
    q.k partial sums, fp16 probabilities) put it ~1e-3 from exact arithmetic; both errors are measured here."""
    from oracle import kv4
    from omniserve_b200.backend import fused_attention_pure_dense as ours
    B, Hq, Hkv = len(lens), 32, 8
    cache, bt, q, k, v = make_kv_case(B, Hq, Hkv, lens, seed=sum(lens) + 5)

    def call(impl):
        kpool, vpool, ptrs = device_tables(cache, bt)
        _, tq, tk, tv = qkv_views(q, k, v)
        o = impl.single_query_attention(tq, tk, tv, ptrs, t(np.asarray(lens, np.int32)), None, 2048, 64, Hkv * 64, max(lens),
                                        128, 500000.0, True, True, True)
        torch.cuda.synchronize()
        return o.cpu().numpy()
    live = ref_module("fused_attention_pure_dense") is not None
    r = reference_outputs(f"parity_attention_{'_'.join(map(str, lens))}", live,
                          lambda: {"out": call(ref_module("fused_attention_pure_dense"))})
    got = call(ours)
    exact = kv4.decode_attention(q, k, v, cache, bt, lens, 128, 500000.0, mimic=False, append=False)
    e_ours = _err(got, exact)
    record_property("err_ours", e_ours)
    e_ref = r.stat("err_vs_exact", lambda ref: _err(ref["out"], exact))
    record_property("err_ref", e_ref)
    a, b = r.pair("out", got)
    print(f"\nattention lens={lens}: |ours-exact|={e_ours:.3e} |ref-exact|={e_ref:.3e} "
          f"|ours-ref|={np.abs(a.astype(np.float32) - b.astype(np.float32)).max() / np.abs(exact).max():.3e}")
    assert e_ours <= max(e_ref, NORTH_STAR)


def test_prefill_write_then_decode_without_host_sync():
    """ADVICE r1: the decode kernel streams pages before its grid dependency resolves; a decode launched right behind the
    prefill writer of the same pages (same stream, PDL, no synchronize) must still see every page complete."""
    from oracle import kv4
    from omniserve_b200.backend import fused_attention_fine_grained_dense as wr
    from omniserve_b200.backend import fused_attention_pure_dense as at
    rng = np.random.default_rng(5)
    Hq, Hkv, Dh = 32, 8, 128
    lens = [640, 257, 1000, 64]
    B, T = len(lens), sum(lens)
    n_pages = sum((l + 64) // 64 for l in lens)
    cache = kv4.PagedKV4(n_pages, Hkv, Dh)
    bt = np.zeros((B, max((l + 64) // 64 for l in lens)), np.int64)
    perm = rng.permutation(n_pages)
    c = 0
    for b, l in enumerate(lens):
        for j in range((l + 64) // 64):
            bt[b, j] = perm[c]; c += 1
    qkv = rng.standard_normal((T, (Hq + 2 * Hkv) * Dh)).astype(np.float16)
    q = rng.standard_normal((B, Hq, Dh)).astype(np.float16)
    k = rng.standard_normal((B, Hkv, Dh)).astype(np.float16)
    v = rng.standard_normal((B, Hkv, Dh)).astype(np.float16)
    flags, rank = t(np.ones(Hkv, np.int32)), t(np.arange(Hkv, dtype=np.int32))
    sl = t(np.asarray(lens, np.int32))
    cu = t(np.concatenate([[0], np.cumsum(lens)]).astype(np.int32))
    dl = t(np.asarray([l + 1 for l in lens], np.int32))
    _, tq, tk, tv = qkv_views(q, k, v)
    results = []
    for sync in (True, False):
        kpool, vpool, ptrs = device_tables(cache, bt)
        tqkv = t(qkv)
        pad = wr.compute_padding_offsets(cu, max(lens), T)
        torch.cuda.synchronize()
        for _ in range(3 if not sync else 1):   # a few rounds so that the race, if any, has chances to show
            kpool.zero_(); vpool.zero_()
            tq2 = tqkv.clone()
            torch.cuda.synchronize()
            wr.apply_bias_rope_update_kv_cache(tq2, sl, None, pad, ptrs, None, flags, rank, Hq, Hkv, max(lens), 64, Hkv * 64, 0,
                                               0, 0, 0, 0, Hkv, 0, 128, 500000.0, 1.0, 8192, True, True, True)
            if sync:
                torch.cuda.synchronize()
            o = at.single_query_attention(tq, tk, tv, ptrs, dl, None, 2048, 64, Hkv * 64, max(lens), 128, 500000.0, True, True,
                                          True)
            torch.cuda.synchronize()
            results.append((o.cpu().numpy(), kpool.cpu().numpy(), vpool.cpu().numpy()))
    base = results[0]
    for r in results[1:]:
        np.testing.assert_array_equal(r[0], base[0])
        np.testing.assert_array_equal(r[1], base[1])
        np.testing.assert_array_equal(r[2], base[2])
