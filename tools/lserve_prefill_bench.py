"""LServe context stage on one GPU: LServeDecoder.prefill with the streaming heads' sparse prefill mask vs every head dense
(the reference's sparse_prefill_mode on / off, scripts/lserve_benchmark/benchmark.sh:8,61), followed by one selector and one
reuse decode step; and the token-streaming kernel alone vs fused causal SDPA on the same streaming heads.

    python tools/lserve_prefill_bench.py --out result.json [--lengths 32768 131072 262144] [--layers 32]

Llama-3-8B shape, retrieval / streaming split of the reference's attn_patterns TSV at static sparsity 0.5
(tests/golden/head_split_llama3_8b_1048k_s50.json), ctx sink 128 / local 8192, decode sink 128 / local 256, budget 4096.
Times are CUDA events after one warm-up run of every timed shape.  FLOPs are counted from the mask: 4 * head_dim per
attended (query, key) pair.  The FP16 peak is the data-sheet figure (dense, 1000 W card), not a measurement.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

DATASHEET_FP16_DENSE_TFLOPS = 2250.0   # HGX B200 data sheet, per GPU, dense FP16 / BF16


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = [x.strip() for x in r.stdout.strip().splitlines()[0].split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def attended_pairs(L: int, sink: int, local: int) -> int:
    """Sum over query positions i < L of |{j <= i : j < sink or i - j < local}|."""
    i = np.arange(L, dtype=np.int64)
    return int((np.minimum(i + 1, local) + np.minimum(sink, np.maximum(0, i + 1 - local))).sum())


def timed(fn, reps=1):
    import torch
    fn()                                  # warm-up of this shape
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ts = []
    for _ in range(reps):
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return min(ts), ts


def kernel_vs_sdpa(L, flags, sink, local, reps):
    import torch
    from omniserve_b200.prefill_attention import _fused_sdpa, make, streaming_prefill_attention
    hq, hkv, dh = 32, 8, 128
    g = hq // hkv
    s_kv = [h for h in range(hkv) if flags[h] == 0]
    gen = torch.Generator(device="cuda").manual_seed(L)
    qkv = torch.randn((L, (hq + 2 * hkv) * dh), generator=gen, device="cuda").half()
    q = qkv[:, :hq * dh].view(L, hq, dh)
    k = qkv[:, hq * dh:(hq + hkv) * dh].view(L, hkv, dh)
    v = qkv[:, (hq + hkv) * dh:].view(L, hkv, dh)
    out = torch.empty((L, hq, dh), dtype=torch.float16, device="cuda")
    cu = [0, L]
    t_k, ts_k = timed(lambda: streaming_prefill_attention(q, k, v, cu, s_kv, [sink] * len(s_kv), [local] * len(s_kv), out), reps)
    qh = [h * g + i for h in s_kv for i in range(g)]
    qs, ks, vs = q[:, qh].contiguous(), k[:, s_kv].contiguous(), v[:, s_kv].contiguous()
    cu_t = torch.tensor(cu, dtype=torch.int32, device="cuda")
    att = make(cu_t, L, len(qh), len(s_kv), dh)

    def sdpa():
        with _fused_sdpa():
            att(qs, ks, vs)
    t_s, ts_s = timed(sdpa, reps)
    n_q = len(qh)
    f_k = 4 * dh * n_q * attended_pairs(L, sink, local)
    f_s = 4 * dh * n_q * (L * (L + 1) // 2)
    return {
        "streaming_kv_heads": s_kv, "q_heads": n_q,
        "kernel_ms": t_k, "kernel_ms_all": ts_k, "kernel_flop": f_k, "kernel_tflops": f_k / t_k / 1e9,
        "kernel_share_of_datasheet_fp16_dense": f_k / t_k / 1e9 / DATASHEET_FP16_DENSE_TFLOPS,
        "sdpa_dense_causal_ms": t_s, "sdpa_ms_all": ts_s, "sdpa_flop": f_s, "sdpa_tflops": f_s / t_s / 1e9,
        "sdpa_share_of_datasheet_fp16_dense": f_s / t_s / 1e9 / DATASHEET_FP16_DENSE_TFLOPS,
        "kernel_speedup_vs_sdpa": t_s / t_k,
    }


def model_run(L, flags, layers, reps):
    import torch
    from omniserve_b200.lserve_model import LServeDecoder
    from omniserve_b200.model import LlamaConfig
    cfg = LlamaConfig.llama3_8b(num_hidden_layers=layers)
    dec = LServeDecoder(cfg, flags[:layers], "cuda")
    dec.alloc(L + 64)
    toks = torch.randint(0, cfg.vocab_size, (L,), generator=torch.Generator().manual_seed(0)).cuda()
    res = {}
    for mode, sparse in (("sparse", True), ("dense", False)):
        nxt = {}

        def run():
            nxt["t"] = dec.prefill(toks, sparse_prefill=sparse)
        t, ts = timed(run, reps)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        t1 = dec.decode_step(nxt["t"], L, run_selector=True)
        b.record()
        torch.cuda.synchronize()
        t_sel = a.elapsed_time(b)
        a.record()
        t2 = dec.decode_step(t1, L + 1, run_selector=False)
        b.record()
        torch.cuda.synchronize()
        res[mode] = {"prefill_ms": t, "prefill_ms_all": ts, "selector_step_ms_eager": t_sel, "reuse_step_ms_eager": a.elapsed_time(b),
                     "next_token": int(nxt["t"]), "decoded": [int(t1), int(t2)]}
    res["sparse_speedup"] = res["dense"]["prefill_ms"] / res["sparse"]["prefill_ms"]
    del dec
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--lengths", type=int, nargs="+", default=[32768, 131072, 262144])
    ap.add_argument("--layers", type=int, default=32)
    ap.add_argument("--reps", type=int, default=1)
    ap.add_argument("--kernel-reps", type=int, default=3)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    fx = json.load(open(os.path.join(ROOT, "tests", "golden", "head_split_llama3_8b_1048k_s50.json")))
    flags = fx["retrieval_head_flags"]
    layer = 9
    out = {"gpu": gpu_info(), "model": "Llama-3-8B shape (random W4A8 weights)", "layers": args.layers,
           "head_split": "tests/golden/head_split_llama3_8b_1048k_s50.json",
           "streaming_kv_heads_total": int(sum(len(f) - sum(f) for f in flags[:args.layers])),
           "kv_heads_total": int(sum(len(f) for f in flags[:args.layers])),
           "ctx_sink": 128, "ctx_local": 8192, "decode_sink": 128, "decode_local": 256, "token_budget": 4096,
           "datasheet_fp16_dense_tflops": DATASHEET_FP16_DENSE_TFLOPS, "results": {}}
    for L in args.lengths:
        r = {"kernel_vs_sdpa_layer9": kernel_vs_sdpa(L, flags[layer], 128, 8192, args.kernel_reps)}
        torch.cuda.empty_cache()
        r["context_stage"] = model_run(L, flags, args.layers, args.reps)
        out["results"][str(L)] = r
        print(json.dumps({str(L): r}), flush=True)
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        json.dump(out, open(args.out, "w"), indent=1)
    out["gpu_after"] = gpu_info()
    json.dump(out, open(args.out, "w"), indent=1)


if __name__ == "__main__":
    main()
