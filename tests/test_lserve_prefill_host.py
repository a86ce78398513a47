"""CPU tests of the LServe context stage: the token-streaming mask of the oracle, the host-side launch plan of the prefill
kernel (ob_debug_streaming_prefill_plan), and the argument checks of token_streaming_attn_func."""
import itertools
import math

import numpy as np
import pytest
import torch

from oracle import streaming_attn as sa


@pytest.mark.parametrize("L", [1, 2, 7, 64, 65, 130])
def test_oracle_mask_equals_brute_force(L):
    for sink, local in itertools.product([0, 1, 3, 64, L, L + 5], [1, 2, 5, 63, L - 1 if L > 1 else 1, L, L + 9]):
        want = np.zeros((L, L), bool)
        for i in range(L):
            for j in range(L):
                want[i, j] = j <= i and (j < sink or i - j < local)
        np.testing.assert_array_equal(sa.mask(L, sink, local), want)
        if sink + local >= L:
            np.testing.assert_array_equal(sa.mask(L, sink, local), np.tril(np.ones((L, L), bool)))


@pytest.mark.parametrize("sink,local,tl", [(128, 256, 499), (128, 256, 39), (128, 256, 384), (64, 128, 449), (0, 1, 10)])
def test_last_row_attends_what_the_decode_streaming_window_keeps(sink, local, tl):
    """Prefill query at position tl (the token a decode step would append after tl cached ones) attends exactly the cached
    positions the streaming-head decode test expects (tests/test_gpu_lserve.py positions()) plus itself."""
    n_valid = min(sink + local - 1, tl)
    gap = tl - n_valid
    decode = np.array([i if i < sink else i + gap for i in range(n_valid)], dtype=np.int64)
    np.testing.assert_array_equal(sa.attended_positions(tl, sink, local), np.append(decode, tl))


def _plan(cu, hq, hkv, heads, sinks, locals_):
    from omniserve_b200.prefill_attention import streaming_prefill_plan
    return streaming_prefill_plan(cu, hq, hkv, heads, sinks, locals_)


CASES = [
    ([0, 1000], 32, 8, [1, 3], [128, 0], [300, 1]),
    ([0, 1, 64, 129, 1129], 8, 8, [0, 5], [0, 4], [1, 64]),
    ([0, 63, 63, 5063], 16, 2, [0, 1], [200, 5000], [8192, 10]),
    ([0, 4097], 64, 8, [7], [128], [8192]),
    ([0] + list(np.cumsum([65] * 70)), 8, 2, [1], [3], [70]),     # > 64 sequences: two launches
]


@pytest.mark.parametrize("cu,hq,hkv,heads,sinks,locals_", CASES)
def test_plan_grid_covers_every_tile_once_and_visits_exactly_the_mask(cu, hq, hkv, heads, sinks, locals_):
    cu = [int(x) for x in cu]
    g = hq // hkv
    QT = 128 // g
    ctas = _plan(cu, hq, hkv, heads, sinks, locals_)
    seen = set()
    for c in ctas:
        key = (c["seq"], c["q_lo"], c["kv_head"])
        assert key not in seen
        seen.add(key)
        L = cu[c["seq"] + 1] - cu[c["seq"]]
        assert c["q_lo"] % QT == 0 and c["q_hi"] == min(c["q_lo"] + QT, L) - 1
        slot = heads.index(c["kv_head"])
        sink, local = sinks[slot], locals_[slot]
        # the key tiles that meet the mask of the tile's query rows
        m = sa.attends(np.arange(c["q_lo"], c["q_hi"] + 1)[:, None], np.arange(L)[None, :], sink, local)
        need = sorted({j // 64 for j in np.nonzero(m.any(axis=0))[0]})
        assert c["key_tiles"] == need, (c, need)
        bound = math.ceil(sink / 64) + math.ceil((local + QT - 1) / 64) + 1
        assert len(c["key_tiles"]) <= bound
    want = {(b, t * QT, h) for b in range(len(cu) - 1) for t in range((cu[b + 1] - cu[b] + QT - 1) // QT) for h in heads}
    assert seen == want


def test_plan_work_is_bounded_independent_of_length():
    n = [max(len(c["key_tiles"]) for c in _plan([0, L], 32, 8, [0], [128], [8192])) for L in (20000, 262144)]
    assert n[0] == n[1] <= math.ceil(128 / 64) + math.ceil((8192 + 32 - 1) / 64) + 1


def _qkv(T=10, hq=8, hkv=2, dh=128):
    x = torch.zeros((T, (hq + 2 * hkv) * dh), dtype=torch.float16)
    return (x[:, :hq * dh].view(T, hq, dh), x[:, hq * dh:(hq + hkv) * dh].view(T, hkv, dh),
            x[:, (hq + hkv) * dh:].view(T, hkv, dh))


GOOD_MT = [-1] * 4 + [0] * 4
GOOD_SI = [4, 16] * 8


@pytest.mark.parametrize("what", ["mask_value", "mask_mixed_group", "info_mixed_group", "info_length", "mask_length",
                                  "negative_sink", "zero_local", "cu_mismatch", "head_dim", "cu_bad_end"])
def test_token_streaming_attn_func_rejects_malformed_input(what):
    from omniserve_b200.prefill_attention import token_streaming_attn_func
    q, k, v = _qkv()
    mt, si = list(GOOD_MT), list(GOOD_SI)
    cq = ck = torch.tensor([0, 4, 10], dtype=torch.int32)
    if what == "mask_value":
        mt = [1] * 4 + [0] * 4
    elif what == "mask_mixed_group":
        mt[0] = 0
    elif what == "info_mixed_group":
        si[2] = 5
    elif what == "info_length":
        si = si[:-2]
    elif what == "mask_length":
        mt = mt[:-1]
    elif what == "negative_sink":
        si = [-1, 16] * 8
    elif what == "zero_local":
        si = [4, 0] * 8
    elif what == "cu_mismatch":
        ck = torch.tensor([0, 5, 10], dtype=torch.int32)
    elif what == "head_dim":
        q, k, v = (x[..., :64] for x in (q, k, v))
    elif what == "cu_bad_end":
        cq = ck = torch.tensor([0, 4, 9], dtype=torch.int32)
    with pytest.raises(ValueError):
        token_streaming_attn_func(q, k, v, cq, ck, torch.tensor(mt, dtype=torch.int32), torch.tensor(si, dtype=torch.int32),
                                  10, 10)


def test_token_streaming_attn_func_needs_cuda_tensors():
    from omniserve_b200.prefill_attention import streaming_prefill_attention, token_streaming_attn_func
    q, k, v = _qkv()
    cu = torch.tensor([0, 10], dtype=torch.int32)
    with pytest.raises(RuntimeError):
        token_streaming_attn_func(q, k, v, cu, cu, torch.tensor(GOOD_MT), torch.tensor(GOOD_SI), 10, 10)
    with pytest.raises(RuntimeError):
        streaming_prefill_attention(q, k, v, cu, [0], [4], [16])

