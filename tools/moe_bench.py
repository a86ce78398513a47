"""Mixtral-8x7B W4A8KV4 on one GPU (omniserve_b200/moe_model.py): prefill of a 32 x 1024 prompt, CUDA-graph decode steps at
bs = 1 / 32 / 64 after a real prefill, per-op times of the MoE block over the 32 layers' own weights, and achieved bytes/s of
the two grouped GEMMs against algorithmic bytes.

    python tools/moe_bench.py --out profiles/r4_mixtral_b200.json

Synthetic weights (seeded device generator), context 1024 per sequence.  Times are CUDA events after warm-up; every decode
figure covers >= 1 s of graph replays; per-op times replay a CUDA graph of the op launched once per layer (32 launches, PDL
between consecutive launches of the same op), so they show device time, not Python launch overhead.  The HBM floor uses the 6 487 GB/s device-to-device copy rate measured on the same
card type in round 1 (profiles/r1_bench_ours.json, SURVEY.md Rooflines); it is computed from shapes, not measured here.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

COPY_GBPS = 6487.0


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = [x.strip() for x in r.stdout.strip().splitlines()[0].split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def events_ms(fn, n):
    import torch
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b)


def decode_rate(m, B, L, min_s=1.0):
    """Graph-replayed decode steps of batch B after a prefill of B x L: ms / step over >= min_s of replays."""
    import torch
    from omniserve_b200.model import DecodeGraph
    room = m.max_ctx - L - 8
    g = DecodeGraph(m, max_timestep=m.max_ctx - 1)
    saved = m.context_lens.clone()

    def run(n):
        m.context_lens.copy_(saved)
        return events_ms(g.step, n)

    run(5)
    probe = run(20) / 20
    n = min(room, max(50, int(math.ceil(1.2 * min_s * 1e3 / probe))))
    total, steps = 0.0, 0
    while total < min_s * 1e3:
        total += run(n)
        steps += n
    m.context_lens.copy_(saved)
    ms = total / steps
    out = g.out.clone()
    assert int(out.min()) >= 0 and int(out.max()) < m.cfg.vocab_size
    return {"batch": B, "context": L, "ms_per_step": ms, "tok_per_s": B * 1e3 / ms, "timed_steps": steps, "timed_ms": total}


def prefill(m, B, L, toks, seq_offset=0):
    import torch
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    m.prefill(toks, [L] * B, seq_offset=seq_offset)
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b)


def moe_ops(m, B, reps):
    """Per-op time of the MoE block at B tokens over the 32 layers' weights (each op launched once per layer, `reps` passes)."""
    import torch
    cfg = m.cfg
    E, k, H, I = cfg.num_local_experts, cfg.num_experts_per_tok, cfg.hidden_size, cfg.intermediate_size
    n = B * k
    mb, b = m.moe_buf, m.buf
    mh, gemm = m.moe_helpers, m.moe_gemm
    x = torch.randn((B, H), generator=torch.Generator(device="cuda").manual_seed(0), device="cuda").half()
    m.moe_block(0, x, True)
    qh, sc, sm = b.quantized_hidden_states_buffer[:B], b.quantized_scale_buffer[:B], b.quantized_sum_buffer[:B]
    st = {}
    lg = mh.moe_router_logits(x, m.layers[0]["gate"], out=mb.logits[:B])
    st["w"], _, st["perm"] = mh.moe_topk_gating_softmax(lg, k, out_offsets=mb.offsets)
    layers = m.layers
    ops = {
        "router": lambda ly: mh.moe_router_logits(x, ly["gate"], out=mb.logits[:B]),
        "topk_sort": lambda ly: mh.moe_topk_gating_softmax(mb.logits[:B], k, out_offsets=mb.offsets),
        "quant": lambda ly: m.ops.fused_kernels.invoke_quant_fuse_sum(qh, x, sm, sc),
        "expand": lambda ly: mh.moe_expand_inputs_and_scales(qh, sm, sc, st["perm"], out=(mb.q_in[:n], mb.sum_in[:n],
                                                                                           mb.scale_in[:n], mb.inv[:n])),
        "w1_w3_gemm": lambda ly: gemm.moe_gemm_forward_cuda_api_dev(mb.q_in[:n], ly["w1_w3"].qweight, ly["w1_w3"].s1_scales,
                                                                    mb.scale_in[:n], ly["w1_w3"].s1_szeros, mb.sum_in[:n],
                                                                    mb.offsets, B, out=mb.gate_up[:n]),
        "silu_mul_quant": lambda ly: m.activation_ops.silu_and_mul_quant(mb.q_act[:n], mb.gate_up[:n], mb.sum_act[:n],
                                                                         mb.scale_act[:n]),
        "w2_gemm": lambda ly: gemm.moe_gemm_forward_cuda_api_dev(mb.q_act[:n], ly["w2"].qweight, ly["w2"].s1_scales,
                                                                 mb.scale_act[:n], ly["w2"].s1_szeros, mb.sum_act[:n],
                                                                 mb.offsets, B, out=mb.y[:n]),
        "finalize": lambda ly: mh.moe_finalize_routing(mb.y[:n], st["w"], mb.inv[:n], B, out=mb.out[:B]),
    }
    res = {}
    for name, op in ops.items():
        # one launch per layer, captured in a CUDA graph so that host launch overhead does not show (as in the decode step)
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            for ly in layers:
                op(ly)
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            for ly in layers:
                op(ly)
        graph.replay()
        torch.cuda.synchronize()
        ms = events_ms(graph.replay, reps)
        res[name] = {"us_per_layer": ms * 1e3 / (reps * len(layers)), "ms_per_step_32_layers": ms / reps}
        del graph
    wb = lambda N, K: E * N * K // 2 + 2 * E * N * 2          # packed weights + s1_scales / s1_szeros
    algo = {"w1_w3_gemm": wb(2 * I, H) + n * H + n * 4 + n * 2 * I * 2,
            "w2_gemm": wb(H, I) + n * I + n * 4 + n * H * 2}
    for name, by in algo.items():
        res[name]["algorithmic_bytes"] = by
        res[name]["achieved_GBps"] = by / (res[name]["us_per_layer"] * 1e-6) / 1e9
    res["sum_ms_per_step"] = sum(v["ms_per_step_32_layers"] for k_, v in res.items() if isinstance(v, dict))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r4_mixtral_b200.json"))
    ap.add_argument("--ctx", type=int, default=1024)
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    import torch
    from omniserve_b200.moe_model import MixtralConfig, MixtralW4A8

    info = gpu_info()
    cfg = MixtralConfig.mixtral_8x7b()
    L = args.ctx
    t0 = time.time()
    m = MixtralW4A8(cfg, "cuda", seed=0, device_init=True)
    torch.cuda.synchronize()
    res = {"gpu": info, "config": "Mixtral-8x7B W4A8KV4, per-channel, 8 experts top-2, synthetic weights",
           "weight_bytes": m.weight_bytes(), "init_s": time.time() - t0}
    E, H, I = cfg.num_local_experts, cfg.hidden_size, cfg.intermediate_size
    expert_bytes = E * 3 * H * I // 2
    res["expert_weight_bytes_per_layer"] = expert_bytes
    res["hbm_floor_ms_per_step_expert_weights"] = 32 * expert_bytes / (COPY_GBPS * 1e9) * 1e3
    res["hbm_floor_basis"] = f"{COPY_GBPS} GB/s device copy rate, profiles/r1_bench_ours.json (not measured in this run)"
    gen = torch.Generator().manual_seed(0)

    # bs = 32: a real 32 x 1024 prefill (timed twice, the second is reported), then graph decode
    B = 32
    m.alloc(B, L + 1024, B * L)
    toks = torch.randint(0, cfg.vocab_size, (B * L,), generator=gen).cuda()
    first = prefill(m, B, L, toks)
    ms = prefill(m, B, L, toks)
    res["prefill_32x1024"] = {"tokens": B * L, "ms": ms, "tok_per_s": B * L * 1e3 / ms, "first_run_ms": first}
    print(json.dumps(res["prefill_32x1024"]), flush=True)
    res["decode_bs32"] = decode_rate(m, B, L)
    print(json.dumps(res["decode_bs32"]), flush=True)
    res["moe_ops_bs32"] = moe_ops(m, B, args.reps)
    print(json.dumps(res["moe_ops_bs32"]), flush=True)

    # bs = 64 (two prefills of 32 sequences) and bs = 1
    m.alloc(64, L + 1024, 32 * L)
    toks64 = torch.randint(0, cfg.vocab_size, (64 * L,), generator=gen).cuda()
    prefill(m, 32, L, toks64[:32 * L], 0)
    prefill(m, 32, L, toks64[32 * L:], 32)
    res["decode_bs64"] = decode_rate(m, 64, L)
    print(json.dumps(res["decode_bs64"]), flush=True)
    res["moe_ops_bs64"] = moe_ops(m, 64, args.reps)
    m.alloc(1, L + 1024, L)
    prefill(m, 1, L, toks[:L])
    res["decode_bs1"] = decode_rate(m, 1, L)
    print(json.dumps(res["decode_bs1"]), flush=True)
    res["moe_ops_bs1"] = moe_ops(m, 1, args.reps)
    res["decode_32k_context"] = "not measured"
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: v for k, v in res.items() if not k.startswith("moe_ops")}, indent=1))


if __name__ == "__main__":
    main()
