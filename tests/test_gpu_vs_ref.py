"""-m gpu: our kernels vs THE REFERENCE'S OWN kernels rebuilt for sm_100 (oracle/_ref, built by
oracle/build_ref.py from the reference's kernels/csrc, unmodified).  This is what pins parity: same seeded
inputs through both implementations on the same B200.  Without oracle/_ref the reference side is the record of such a
run in tests/golden/ref_kernels.npz (a fixed sample of every output plus its scale, and the bytes the kernels
changed in the KV pages; see tests/gpu_util.py)."""
import numpy as np
import pytest
import torch

from tests.gpu_util import device_tables, make_gemm_inputs, make_kv_case, qkv_views, ref_module, reference_outputs, t

pytestmark = pytest.mark.gpu


def _f32(x):
    return x.astype(np.float32)


@pytest.mark.parametrize("M,N,K", [(64, 6144, 4096), (64, 4096, 14336), (17, 4096, 4096), (1024, 4096, 4096), (300, 1024, 2048)])
def test_gemm_per_channel_bit_exact_vs_reference_kernel(M, N, K):
    from omniserve_b200.backend import qgemm_w4a8_per_chn as ours
    d = make_gemm_inputs(M, N, K, seed=M + N)
    args = [t(d[k]) for k in ("a", "qw", "s1", "sa", "szs", "ssum")]

    def run():
        o_ref = torch.zeros((M, N), dtype=torch.float16, device="cuda")
        ref_module("qgemm_w4a8_per_chn").gemm_forward_cuda(*args, o_ref)
        torch.cuda.synchronize()
        return {"out": o_ref}
    r = reference_outputs(f"gemm_per_chn_{M}x{N}x{K}", ref_module("qgemm_w4a8_per_chn") is not None, run)
    o_our = torch.zeros((M, N), dtype=torch.float16, device="cuda")
    ours.gemm_forward_cuda(*args, o_our)
    torch.cuda.synchronize()
    a, b = r.pair("out", o_our)
    assert np.abs(_f32(a) - _f32(b)).max() <= 1e-3 * r.absmax("out")
    assert (a == b).mean() > 0.999, "INT32 accumulate is exact; fp16 tails should match bit-for-bit"


@pytest.mark.parametrize("M,N,K", [(64, 4096, 4096), (200, 1024, 2048), (128, 6144, 4096)])
def test_gemm_per_group_bit_exact_vs_reference_kernel(M, N, K):
    from omniserve_b200.backend import qgemm_w4a8_per_group as ours
    d = make_gemm_inputs(M, N, K, seed=M + K, per_group=True)
    args = [t(d[k]) for k in ("a", "qw", "z2", "s2", "s1", "sa")]

    def run():
        o_ref = torch.zeros((M, N), dtype=torch.float16, device="cuda")
        ref_module("qgemm_w4a8_per_group").gemm_forward_cuda(*args, o_ref)
        torch.cuda.synchronize()
        return {"out": o_ref}
    r = reference_outputs(f"gemm_per_group_{M}x{N}x{K}", ref_module("qgemm_w4a8_per_group") is not None, run)
    o_our = torch.zeros((M, N), dtype=torch.float16, device="cuda")
    ours.gemm_forward_cuda(*args, o_our)
    torch.cuda.synchronize()
    a, b = r.pair("out", o_our)
    assert np.abs(_f32(a) - _f32(b)).max() <= 1e-3 * r.absmax("out")
    assert (a == b).mean() > 0.999


@pytest.mark.parametrize("T,H", [(64, 4096), (5, 14336), (3, 8192)])
def test_quant_and_norm_vs_reference_kernels(T, H):
    from omniserve_b200.backend import fused_kernels, layernorm_ops
    g = torch.Generator(device="cuda").manual_seed(T + H)
    x = (torch.randn((T, H), generator=g, device="cuda") * 2 + 0.1).half()
    w = (torch.randn((H,), generator=g, device="cuda") * 0.2 + 1).half()

    def bufs():
        return (torch.zeros((T, H), dtype=torch.int8, device="cuda"), torch.zeros(T, dtype=torch.float16, device="cuda"),
                torch.zeros(T, dtype=torch.float16, device="cuda"))

    def run():
        rk, rl = ref_module("fused_kernels"), ref_module("layernorm_ops")
        q1, s1, m1 = bufs()
        rk.invoke_quant_fuse_sum(q1, x, m1, s1)
        res = {"quant_q": q1, "quant_s": s1, "quant_m": m1}
        if H <= 8192:
            q1, s1, m1 = bufs()
            rl.rms_norm_general_fuse_sum(q1, x, w, m1, s1, 1e-5, True)
            res.update(norm_q=q1, norm_s=s1, norm_m=m1)
        torch.cuda.synchronize()
        return res
    live = ref_module("fused_kernels") is not None and ref_module("layernorm_ops") is not None
    r = reference_outputs(f"quant_norm_{T}x{H}", live, run)
    q2, s2, m2 = bufs()
    fused_kernels.invoke_quant_fuse_sum(q2, x, m2, s2)
    torch.cuda.synchronize()
    for name, ours in (("quant_q", q2), ("quant_s", s2)):
        a, b = r.pair(name, ours)
        assert np.array_equal(a, b), name
    a, b = r.pair("quant_m", m2)
    assert np.abs(_f32(a) - _f32(b)).max() <= 2e-3 * r.absmax("quant_m") + 2e-2
    if H <= 8192:
        q2, s2, m2 = bufs()
        layernorm_ops.rms_norm_general_fuse_sum(q2, x, w, m2, s2, 1e-5, True)
        torch.cuda.synchronize()
        a, b = r.pair("norm_q", q2)
        d = np.abs(a.astype(np.int32) - b.astype(np.int32))
        assert d.max() <= 1 and (d > 0).mean() <= 1e-3   # fp32 reduction order of mean / variance differs
        a, b = r.pair("norm_s", s2)
        assert np.abs(_f32(a) - _f32(b)).max() <= 1e-3 * r.absmax("norm_s")
        a, b = r.pair("norm_m", m2)
        assert np.abs(_f32(a) - _f32(b)).max() <= 0.05


def test_silu_vs_reference_kernel():
    from omniserve_b200.backend import activation_ops
    g = torch.Generator(device="cuda").manual_seed(3)
    x = (torch.randn((9, 2 * 14336), generator=g, device="cuda") * 2).half()

    def run():
        o1 = torch.zeros((9, 14336), dtype=torch.float16, device="cuda")
        ref_module("activation_ops").silu_and_mul(o1, x)
        torch.cuda.synchronize()
        return {"out": o1}
    r = reference_outputs("silu_9x14336", ref_module("activation_ops") is not None, run)
    o2 = torch.zeros((9, 14336), dtype=torch.float16, device="cuda")
    activation_ops.silu_and_mul(o2, x)
    torch.cuda.synchronize()
    a, b = r.pair("out", o2)
    assert np.abs(_f32(a) - _f32(b)).max() <= 1e-3 * r.absmax("out")
    assert (a == b).mean() > 0.995


@pytest.mark.parametrize("lens", [(70, 200, 129), (1024, 1100, 1535), (1, 64, 65)])
def test_decode_attention_vs_reference_kernel(lens):
    from omniserve_b200.backend import fused_attention_pure_dense as ours
    B, Hq, Hkv = len(lens), 32, 8
    cache, bt, q, k, v = make_kv_case(B, Hq, Hkv, lens, seed=sum(lens))

    def call(impl):
        kpool, vpool, ptrs = device_tables(cache, bt)
        _, tq, tk, tv = qkv_views(q, k, v)
        ln = t(np.asarray(lens, np.int32))
        o = impl.single_query_attention(tq, tk, tv, ptrs, ln, None, 2048, 64, Hkv * 128 // 2, max(lens), 128, 500000.0,
                                        True, True, True)
        torch.cuda.synchronize()
        return {"out": o, "k_pool": kpool, "v_pool": vpool}
    live = ref_module("fused_attention_pure_dense") is not None
    r = reference_outputs(f"decode_attention_{'_'.join(map(str, lens))}", live,
                          lambda: call(ref_module("fused_attention_pure_dense")),
                          bases={"k_pool": cache.k_pool, "v_pool": cache.v_pool})
    mine = call(ours)
    a, b = r.pair("out", mine["out"])
    assert np.abs(_f32(a) - _f32(b)).max() <= 3e-3 * r.absmax("out")   # the reference itself is ~1e-3 from exact arithmetic
    # appended K/V page bytes: identical formula; RoPE intrinsics differ (reference: __sinf/__cosf/__powf)
    a, b = r.pair("k_pool", mine["k_pool"])
    kd = (a != b).mean()
    a, b = r.pair("v_pool", mine["v_pool"])
    vd = (a != b).mean()
    assert vd == 0, "V is not rotated: appended bytes / scales / zeros must be identical to the reference's"
    assert kd < 1e-4


def test_prefill_writer_vs_reference_kernel():
    from omniserve_b200.backend import fused_attention_fine_grained_dense as ours
    from oracle import kv4
    rng = np.random.default_rng(17)
    Hq, Hkv, Dh = 32, 8, 128
    lens = [200, 64, 333]
    T = sum(lens)
    n_pages = sum((l + 63) // 64 for l in lens)
    cache = kv4.PagedKV4(n_pages, Hkv, Dh)
    bt = np.zeros((3, 6), np.int64)
    perm = rng.permutation(n_pages)
    c = 0
    for b, l in enumerate(lens):
        for j in range((l + 63) // 64):
            bt[b, j] = perm[c]; c += 1
    qkv = rng.standard_normal((T, (Hq + 2 * Hkv) * Dh)).astype(np.float16)
    flags = t(np.ones(Hkv, np.int32))
    rank = t(np.arange(Hkv, dtype=np.int32))

    def call(impl):
        kpool, vpool, ptrs = device_tables(cache, bt)
        tqkv = t(qkv)
        sl = t(np.asarray(lens, np.int32))
        cu = t(np.concatenate([[0], np.cumsum(lens)]).astype(np.int32))
        pad = impl.compute_padding_offsets(cu, max(lens), T)
        impl.apply_bias_rope_update_kv_cache(tqkv, sl, None, pad, ptrs, None, flags, rank, Hq, Hkv, max(lens), 64,
                                             Hkv * Dh // 2, 0, 0, 0, 0, 0, Hkv, 0, 128, 500000.0, 1.0, 8192, True, True,
                                             True)
        torch.cuda.synchronize()
        return {"qkv": tqkv, "k_pool": kpool, "v_pool": vpool, "padding_offset": pad}
    live = ref_module("fused_attention_fine_grained_dense") is not None
    r = reference_outputs("prefill_writer_200_64_333", live, lambda: call(ref_module("fused_attention_fine_grained_dense")))
    mine = call(ours)
    a, b = r.pair("padding_offset", mine["padding_offset"])
    assert np.array_equal(a, b)
    a, b = r.pair("v_pool", mine["v_pool"])
    assert np.array_equal(a, b)                                         # V pages byte-identical
    a, b = r.pair("qkv", mine["qkv"])
    assert np.abs(_f32(a) - _f32(b)).max() <= 8e-3                      # fast-math sincos of the reference at pos ~300
    # K nibbles follow the rotated values: one fp16 ulp on a token's min/max changes that token's scale/zero and
    # with it most of its 64 bytes, so a ~1% byte difference corresponds to ~1% of (token, head) rows
    a, b = r.pair("k_pool", mine["k_pool"])
    assert (a != b).mean() < 3e-2
