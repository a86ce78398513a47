"""CPU tests of the Mixtral mixture-of-experts stack: the routing / permutation / block definitions of oracle/moe.py, the
host-only schedule of the device-offset grouped GEMM (ob_debug_moe_device_plan) and the argument checks of the Python ops."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import act, moe, w4a8


def _torch_routing(logits, k):
    """Independent restatement: torch softmax -> topk -> renormalise (torch.topk's order is not specified on ties, so the
    random logits below have none)."""
    p = torch.softmax(torch.from_numpy(logits).float(), dim=-1)
    v, i = torch.topk(p, k, dim=-1)
    return (v / v.sum(-1, keepdim=True)).numpy(), i.int().reshape(-1).numpy()


@pytest.mark.parametrize("T,E,k", [(50, 8, 2), (20, 64, 8), (33, 4, 1), (7, 5, 5)])
def test_oracle_routing_matches_torch(T, E, k):
    lg = np.random.default_rng(T * E + k).standard_normal((T, E)).astype(np.float32) * 3
    w, ei = moe.topk_gating_softmax(lg, k)
    rw, rei = _torch_routing(lg, k)
    np.testing.assert_array_equal(ei, rei)
    np.testing.assert_allclose(w, rw, rtol=1e-6, atol=1e-7)
    assert w.dtype == np.float32 and ei.dtype == np.int32


def test_oracle_ties_lower_index_first_and_slot_order():
    lg = np.array([[0, 1, 1, 1], [2, 0, 2, 0], [0, 0, 0, 0], [1, 3, 2, 3]], np.float32)
    w, ei = moe.topk_gating_softmax(lg, 2)
    assert ei.reshape(4, 2).tolist() == [[1, 2], [0, 2], [0, 1], [1, 3]]
    np.testing.assert_array_equal(w[:3], np.full((3, 2), 0.5, np.float32))
    w3, ei3 = moe.topk_gating_softmax(lg, 3)
    assert ei3.reshape(4, 3).tolist() == [[1, 2, 3], [0, 2, 1], [0, 1, 2], [1, 3, 2]]   # descending p, then index
    assert np.all(np.diff(moe.softmax_f32(lg)[np.arange(4)[:, None], ei3.reshape(4, 3)], axis=1) <= 0)


@pytest.mark.parametrize("T,E,k", [(64, 8, 2), (1, 8, 2), (300, 16, 4), (10, 64, 8)])
def test_permutation_invariants(T, E, k):
    lg = np.random.default_rng(T + E).standard_normal((T, E)).astype(np.float32)
    _, ei = moe.topk_gating_softmax(lg, k)
    perm, off = moe.permutation(ei, E)
    n = T * k
    assert sorted(perm.tolist()) == list(range(n))                       # a bijection
    assert np.all(np.diff(ei[perm]) >= 0)                                # sorted by expert
    for e in range(E):
        seg = perm[off[e]:off[e + 1]]
        assert np.all(np.diff(seg) > 0)                                  # stable: (token, slot) ascending inside an expert
        assert np.all(ei[seg] == e)
    np.testing.assert_array_equal(np.diff(off), np.bincount(ei, minlength=E))
    assert off[0] == 0 and off[-1] == n


def _experts(rng, E, N, K):
    q = rng.integers(0, 16, (E, N, K), dtype=np.uint8)
    qw = np.stack([w4a8.pack_w4(q[e]) for e in range(E)])
    s1 = rng.uniform(0.002, 0.006, (E, N)).astype(np.float16)
    szs = (s1.astype(np.float32) * 8).astype(np.float16)
    return qw, s1, szs


def test_oracle_moe_block_equals_per_token_per_expert_loop():
    rng = np.random.default_rng(0)
    T, H, I, E, k = 9, 128, 128, 4, 2
    x = rng.standard_normal((T, H)).astype(np.float16)
    gate = (rng.standard_normal((E, H)) / np.sqrt(H)).astype(np.float16)
    w13, w2 = _experts(rng, E, 2 * I, H), _experts(rng, E, H, I)
    out, st = moe.moe_block(x, gate, w13, w2, k)
    # loop: each token, each of its experts, with the dense per-channel GEMM and the activation ops of the reference
    q, sc, ss = act.quant_fuse_sum(x)
    w, ei = st["weights"], st["expert_indices"].reshape(T, k)
    ref = np.zeros((T, H), np.float32)
    for tk in range(T):
        acc = np.zeros(H, np.float32)
        for j in range(k):
            e = ei[tk, j]
            _, gu = w4a8.gemm_per_chn(q[tk:tk + 1], w13[0][e], w13[1][e], sc[tk:tk + 1], w13[2][e], ss[tk:tk + 1])
            qm, sc2, ss2 = act.quant_fuse_sum(act.silu_and_mul(gu))
            _, y = w4a8.gemm_per_chn(qm, w2[0][e], w2[1][e], sc2, w2[2][e], ss2)
            acc = (acc + (w[tk, j] * y[0].astype(np.float32)).astype(np.float32)).astype(np.float32)
        ref[tk] = acc
    np.testing.assert_array_equal(out, ref.astype(np.float16))
    assert np.abs(out.astype(np.float32)).max() > 0


def _plan(E, N, K, offsets, total, sms=148, entries=True):
    from omniserve_b200 import _lib as L
    g, tpc = C.c_int(), C.c_int()
    off = (C.c_int * len(offsets))(*offsets)
    n = E * N // 128
    buf = (C.c_int * (6 * n))() if entries else None
    rc = L.lib().ob_debug_moe_device_plan(E, N, K, sms, off, total, C.byref(g), C.byref(tpc), buf, n if entries else 0)
    assert rc == 0
    ent = np.frombuffer(buf, dtype=np.int32).reshape(n, 6).copy() if entries else None
    return g.value, tpc.value, ent


@pytest.mark.parametrize("E,N,K", [(8, 28672, 4096), (8, 4096, 14336), (4, 1024, 256), (64, 256, 128)])
def test_device_plan_covers_every_expert_tile_once_and_rows_match(E, N, K):
    rng = np.random.default_rng(E + N)
    T, k = 32, 2
    sizes = np.bincount(rng.integers(0, E, T * k), minlength=E)
    offsets = [0] + np.cumsum(sizes).tolist()
    grid, tpc, ent = _plan(E, N, K, offsets, T * k)
    n_te = N // 128
    assert grid * tpc >= E * n_te > (grid - 1) * tpc and grid <= 2 * 148
    pairs = {(int(r[2]), int(r[3])) for r in ent}
    assert pairs == {(e, nt) for e in range(E) for nt in range(n_te)} and len(ent) == E * n_te
    for r in ent:
        cta, slot, e, nt, row0, rows = r.tolist()
        assert slot == e and 0 <= cta < grid
        assert row0 == offsets[e] and rows == sizes[e]
    ctas = ent[:, 0]
    assert np.all(np.diff(ctas) >= 0) and np.bincount(ctas).max() <= tpc   # contiguous whole tiles per CTA


def test_device_plan_grid_does_not_depend_on_offsets():
    E, N, K = 8, 28672, 4096
    first = None
    for offsets in ([0] * 9, [0, 64, 128, 128, 128, 128, 128, 128, 128], [0, 8, 16, 24, 32, 40, 48, 56, 64], [0, 1] + [1] * 7):
        total = offsets[-1]
        grid, tpc, ent = _plan(E, N, K, offsets, total)
        shape = (grid, tpc, ent[:, :4].tobytes())
        first = first or shape
        assert shape == first


def test_device_plan_clamps_malformed_offsets():
    E, N, K, total = 8, 256, 128, 20
    for offsets in ([0, 5, 3, 30, -4, 10, 100, 7, 20], [-9, -9, 50, 50, 1 << 30, -(1 << 30), 5, 25, 19],
                    [0, 200, 200, 200, 200, 200, 200, 200, 200]):
        _, _, ent = _plan(E, N, K, offsets, total)
        for r in ent:
            _, slot, _, _, row0, rows = r.tolist()
            assert 0 <= row0 <= total and 0 <= rows <= 64 and row0 + rows <= total
            lo = min(max(offsets[slot], 0), total)
            hi = min(max(offsets[slot + 1], lo), total)
            assert row0 == lo and rows == min(hi - lo, 64)


def test_device_plan_rejects_bad_shapes():
    from omniserve_b200 import _lib as L
    g, tpc = C.c_int(), C.c_int()
    for E, N, K in ((0, 256, 128), (65, 256, 128), (8, 200, 128), (8, 256, 100)):
        assert L.lib().ob_debug_moe_device_plan(E, N, K, 148, None, 0, C.byref(g), C.byref(tpc), None, 0) != 0


def test_argument_validation():
    from omniserve_b200.backend import moe_helpers as mh
    from omniserve_b200.backend import qgemm_w4a8_moe as op
    lg = torch.zeros((4, 8), dtype=torch.float32)
    with pytest.raises(ValueError):
        mh.moe_topk_gating_softmax(lg, 9)                                   # k > E
    with pytest.raises(ValueError):
        mh.moe_topk_gating_softmax(torch.zeros((4, 65)), 2)                 # E > 64
    with pytest.raises(ValueError):
        mh.moe_topk_gating_softmax(torch.zeros((4, 16)), 9)                 # k > 8
    with pytest.raises(ValueError):
        mh.moe_topk_gating_softmax(lg, 0)
    with pytest.raises(ValueError):
        mh.moe_topk_gating_softmax(torch.zeros(8), 2)                       # not [T, E]
    with pytest.raises(ValueError):
        mh.moe_topk_gating_softmax(lg.half(), 2)                            # not fp32
    with pytest.raises(ValueError):
        mh.moe_router_logits(torch.zeros((4, 64)), torch.zeros((8, 64), dtype=torch.float16))
    with pytest.raises(ValueError):
        mh.moe_router_logits(torch.zeros((4, 64), dtype=torch.float16), torch.zeros((8, 32), dtype=torch.float16))
    with pytest.raises(RuntimeError):                                       # valid, but no CUDA tensors
        mh.moe_topk_gating_softmax(lg, 2)
    with pytest.raises(RuntimeError):
        mh.moe_router_logits(torch.zeros((4, 64), dtype=torch.float16), torch.zeros((8, 64), dtype=torch.float16))
    with pytest.raises(RuntimeError):
        mh.moe_expand_inputs_and_scales(torch.zeros((4, 64), dtype=torch.int8), None, torch.zeros(4, dtype=torch.float16),
                                        torch.zeros(8, dtype=torch.int32))
    with pytest.raises(RuntimeError):
        mh.moe_finalize_routing(torch.zeros((8, 64), dtype=torch.float16), torch.zeros((4, 2)), torch.zeros(8, dtype=torch.int32), 4)
    x = torch.zeros((130, 128), dtype=torch.int8)
    qw = torch.zeros((8, 256, 64), dtype=torch.int8)
    s = torch.zeros((8, 256), dtype=torch.float16)
    a = torch.zeros(130, dtype=torch.float16)
    with pytest.raises(ValueError):                                         # > 64 tokens
        op.moe_gemm_forward_cuda_api_dev(x, qw, s, a, s, a, torch.zeros(9, dtype=torch.int32), 65)
    with pytest.raises(RuntimeError):
        op.moe_gemm_forward_cuda_api_dev(x[:64], qw, s, a[:64], s, a[:64], torch.zeros(9, dtype=torch.int32), 32)


def test_model_rejects_decode_batches_over_64_and_allocates_no_dense_mlp():
    from omniserve_b200.moe_model import MixtralConfig, MixtralW4A8
    m = MixtralW4A8(MixtralConfig.tiny(), device="cpu")
    for ly in m.layers:
        assert "gate_up_proj" not in ly and "down_proj" not in ly
        assert tuple(ly["w1_w3"].qweight.shape) == (4, 1024, 128) and tuple(ly["w2"].qweight.shape) == (4, 256, 256)
    m.alloc(65, 128, 65)
    assert m.buf.quantized_mlp_act_buffer.numel() == 0 and m.buf.gate_up_proj_act_buffer.numel() == 0
    with pytest.raises(ValueError):
        m.decode_step(torch.zeros(65, dtype=torch.int64), 1)
    with pytest.raises(ValueError):
        MixtralW4A8(MixtralConfig.tiny(num_local_experts=4, num_experts_per_tok=5), device="cpu")
    c = MixtralConfig.mixtral_8x7b()
    assert (c.hidden_size, c.intermediate_size, c.num_hidden_layers, c.num_attention_heads, c.num_key_value_heads,
            c.head_dim, c.vocab_size, c.rope_theta, c.rms_norm_eps, c.num_local_experts, c.num_experts_per_tok,
            c.group_size) == (4096, 14336, 32, 32, 8, 128, 32000, 1e6, 1e-5, 8, 2, -1)
