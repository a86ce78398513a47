#!/usr/bin/env python
"""Benchmark of the W4A8KV4 hot path on B200: Llama-3-8B decode at bs=64 (BASELINE.json configs[1]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" = one decode iteration of the whole batch (64 sequences -> 64 new tokens) through the 32-layer
W4A8KV4 stack: per layer rmsnorm+quant, qkv GEMM, KV4 attention (+append), quant, o_proj GEMM, add,
rmsnorm+quant, gate_up GEMM, silu*mul+quant, down GEMM, add; then final norm, lm_head, argmax.
The KV pages are filled beforehand by a real prefill of 64 x 1024 synthetic prompt tokens (reported separately
as prefill tok/s and GEMM TOPS).  Context grows from 1024 during the run and wraps back to 1024 when the
24-page budget (1536 tokens = in 1024 + out 512, README.md:281) is exhausted.

Prints ONE JSON line (see the contract in the task description); `--impl reference` runs the same step through
the reference's own kernels rebuilt for sm_100 (oracle/_ref), eagerly (the reference has no CUDA graphs and no TP).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

PROMPT_LEN, GEN_LEN, BATCH = 1024, 512, 64
PREFILL_SUB_BATCH = 8  # sequences per prefill chunk (8192 tokens), like the reference's chunked prefill


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops", 1590.0), "measured"
    return 6650.0, 1590.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, dev_index: int):
        self.idx, self.proc, self.lines = dev_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.idx)], stdout=subprocess.PIPE, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx = float(f[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def ref_loader():
    import importlib.machinery
    import importlib.util
    d = os.path.join(ROOT, "oracle", "_ref", "omniserve_backend")

    def load(name):
        path = os.path.join(d, f"{name}.so")
        if not os.path.exists(path):
            raise FileNotFoundError(path)
        loader = importlib.machinery.ExtensionFileLoader(name, path)
        spec = importlib.util.spec_from_loader(name, loader)
        m = importlib.util.module_from_spec(spec)
        loader.exec_module(m)
        return m
    return load


def usable_cores() -> int:
    """Host cores this process may really use: the scheduler affinity mask clipped by the cgroup CPU quota (the GPU lease
    runs in a container; os.cpu_count() reports the whole host and oversubscribes a small quota 10-50x)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    quota = None
    try:   # cgroup v2
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            quota = float(q) / float(per)
    except Exception:
        try:   # cgroup v1
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / per
        except Exception:
            pass
    if quota is not None:
        n = max(1, min(n, int(quota + 0.5)))
    return max(1, n)


CPU_BASELINE_REPS = 5


def cpu_baseline(cfg, reps: int = CPU_BASELINE_REPS):
    """torch-fp16 CPU path (oracle/cpu_path.py) for the same decode step on the host cores: ONE layer timed a FIXED number
    of times (min and median reported), x32 extrapolated (bounded sample, stated in `sample`)."""
    from oracle import cpu_path
    cores = usable_cores()
    torch.set_num_threads(cores)
    c = dict(hidden=cfg.hidden_size, inter=cfg.intermediate_size, hq=cfg.num_attention_heads,
             hkv=cfg.num_key_value_heads, dh=cfg.head_dim, eps=cfg.rms_norm_eps, base=cfg.rope_theta)
    g = torch.Generator().manual_seed(0)
    p = cpu_path.random_layer(c, g)
    ctx = PROMPT_LEN + GEN_LEN // 2
    kc = torch.randn(BATCH, c["hkv"], ctx + 8, c["dh"], generator=g).half()
    vc = torch.randn(BATCH, c["hkv"], ctx + 8, c["dh"], generator=g).half()
    x = torch.randn(BATCH, c["hidden"], generator=g).half()
    lens = torch.full((BATCH,), ctx, dtype=torch.int64)
    cpu_path.decode_layer(x, p, kc, vc, lens, c)  # warm-up
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        cpu_path.decode_layer(x, p, kc, vc, lens, c)
        ts.append(time.perf_counter() - t0)
    ts.sort()
    best, med = ts[0], ts[len(ts) // 2]
    L = cfg.num_hidden_layers
    return {"value": BATCH / (best * L), "value_median": BATCH / (med * L), "unit": "tok/s", "cores": cores, "kind": "port",
            "host_cpu_count": os.cpu_count(), "layer_ms_min": best * 1e3, "layer_ms_median": med * 1e3,
            "sample": f"1 decoder layer (bs={BATCH}, ctx={ctx}) x {reps} runs after 1 warm-up (value = fastest, value_median = "
                      f"median), x{L} layers extrapolated; lm_head/embedding excluded; torch CPU fp16 storage / fp32 math; "
                      f"threads = affinity mask clipped by the cgroup cpu quota"}


def time_kernels(model, graph_ctx: int):
    """Per-kernel device time, measured live with CUDA events on the launching stream: each kernel class is
    launched once per layer over the 32 layers' own weights / KV pools (>> L2, so every launch is HBM-cold)."""
    cfg, b, B = model.cfg, model.buf, model.batch
    ops = model.ops
    res = {}

    def timed(fn, reps=3):
        """fn launches the kernel once per layer; it is captured into a CUDA graph so that the CUDA events
        bracket device time only (no Python / ctypes launch overhead between the launches)."""
        fn()  # warm-up (lazy workspaces, tensor maps)
        torch.cuda.synchronize()
        if not model.fuse_add_norm:  # reference kernels launch on the legacy default stream: not capturable
            best = 1e9
            for _ in range(reps):
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                fn()
                e1.record()
                torch.cuda.synchronize()
                best = min(best, e0.elapsed_time(e1))
            return best / cfg.num_hidden_layers
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            fn()
        best = 1e9
        for _ in range(reps):
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            g.replay()
            e1.record()
            torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        return best / cfg.num_hidden_layers  # ms per launch

    qh, sc, sm = b.quantized_hidden_states_buffer[:B], b.quantized_scale_buffer[:B], b.quantized_sum_buffer[:B]
    qh.random_(-127, 127); sc.fill_(0.02); sm.fill_(0.1)
    b.quantized_attn_buffer[:B].random_(-127, 127); b.quantized_mlp_act_buffer[:B].random_(-127, 127)
    gemm_bytes = {}
    for name, x, out in (("qkv_proj", qh, b.qkv_proj_act_buffer[:B]), ("o_proj", b.quantized_attn_buffer[:B], b.out_down_proj_act_buffer[:B]),
                         ("gate_up_proj", qh, b.gate_up_proj_act_buffer[:B]), ("down_proj", b.quantized_mlp_act_buffer[:B], b.out_down_proj_act_buffer[:B])):
        def run(name=name, x=x, out=out):
            for ly in model.layers:
                ly[name](x, sc, sm, out)
        res[name] = timed(run)
        lin = model.layers[0][name]
        gemm_bytes[name] = lin.qweight.numel() + B * lin.in_features + 2 * B * lin.out_features + 4 * lin.out_features + 4 * B
    # attention at the bench's mid-run context
    qkv = b.qkv_proj_act_buffer[:B]
    qkv.normal_()
    q3 = qkv[:, :model.q_size].view(B, model.hq, cfg.head_dim)
    k3 = qkv[:, model.q_size:model.q_size + model.kv_size].view(B, model.hkv, cfg.head_dim)
    v3 = qkv[:, model.q_size + model.kv_size:].view(B, model.hkv, cfg.head_dim)
    lens = torch.full((B,), graph_ctx + 1, dtype=torch.int32, device=model.device)

    def attn():
        for li in range(cfg.num_hidden_layers):
            ops.fused_attention_pure_dense.single_query_attention(q3, k3, v3, model.kv.tables[li], lens, None, model.max_ctx,
                                                                  64, model.kv_size // 2, graph_ctx, cfg.head_dim,
                                                                  cfg.rope_theta, True, True, True)
    res["attention"] = timed(attn)
    attn_bytes = B * graph_ctx * model.hkv * (128 + 8) + B * (2 * model.hq + 2 * model.hkv) * 128 * 2
    return res, gemm_bytes, attn_bytes


def prefill_gemm_tops(model, M=8192):
    """Prefill-shaped W4A8 GEMMs (M = 8192-token chunk) timed with CUDA events -> achieved INT8 TOPS."""
    dev = model.device
    x = torch.randint(-127, 128, (M, max(model.cfg.hidden_size, model.inter)), dtype=torch.int8, device=dev)
    sc = torch.full((M,), 0.02, dtype=torch.float16, device=dev)
    sm = torch.full((M,), 0.1, dtype=torch.float16, device=dev)
    out = {}
    tot_ops = tot_ms = 0.0
    for name in ("qkv_proj", "o_proj", "gate_up_proj", "down_proj"):
        lin = model.layers[0][name]
        xin = x[:, :lin.in_features].contiguous()
        o = torch.empty((M, lin.out_features), dtype=torch.float16, device=dev)
        for _ in range(2):
            lin(xin, sc, sm, o)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n = 0
        e0.record()
        for ly in model.layers[:8]:
            ly[name](xin, sc, sm, o)
            n += 1
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / n
        ops_ = 2.0 * M * lin.out_features * lin.in_features
        out[name] = {"ms": ms, "tops": ops_ / ms / 1e9}
        tot_ops += ops_; tot_ms += ms
        del o
    out["all"] = {"ms": tot_ms, "tops": tot_ops / tot_ms / 1e9}
    return out


# DRAM traffic per roofline unit from one `ncu --set full` capture per kernel (tools/ncu_targets.py, round 1):
# the four decode GEMM launches of a layer: qkv 14.52 + o 9.79 + gate_up 59.48 + down 31.42 MB; attention 90.02 + 2.84 MB.
NCU_DRAM_BYTES = {"w4a8_gemm(decode,4 launches/layer)": 115.2e6, "kv4_decode_attention": 92.9e6}   # round-1 captures (fallback)


def ncu_traffic():
    """DRAM bytes per roofline unit from the newest committed `ncu --set full` capture (tools/ncu_targets.py ->
    tools/ncu_summary.py -> profiles/r<N>_ncu/traffic.json)."""
    for rnd in ("r2", "r1"):
        f = os.path.join(ROOT, "profiles", f"{rnd}_ncu", "traffic.json")
        if os.path.exists(f):
            try:
                d = json.load(open(f))
                if d.get("per_layer_dram_bytes"):
                    return d["per_layer_dram_bytes"], f"profiles/{rnd}_ncu/traffic.json ({d.get('source', '')})"
            except Exception:
                pass
    return NCU_DRAM_BYTES, "constants recorded from the round-1 captures (profiles/r1_ncu/*.raw.csv)"
INT8_PEAK_RECORDED = 4350.0  # TOPS, tools/umma_rate.cu on this pool's B200 (profiles/r1_umma_rate.log): 8188 MAC/clk/SM


def int8_peak():
    """Dense INT8 tensor-pipe peak measured on this GPU with the stand-alone tcgen05.mma probe (128x128x32 kind::i8
    MMAs issued back to back on all SMs, no loads); falls back to the value recorded in profiles/ when the probe
    binary was not built."""
    exe = os.path.join(ROOT, "tools", "_build", "umma_rate")
    try:
        out = subprocess.run([exe], capture_output=True, text=True, timeout=60).stdout
        for ln in out.splitlines():
            if ln.startswith("i8  128x128x32  A=tmem") and "ctas=148" in ln:
                return float(ln.split("->")[1].split()[0]) * 1000.0, "measured live (tools/umma_rate.cu)"
    except Exception:
        pass
    return INT8_PEAK_RECORDED, "recorded (profiles/r1_umma_rate.log)"


def measure_secondary(cfg, dev, rank, world, steps, warmup, tp, batch=BATCH, tag=None):
    """A second decode measurement next to the headline: tp == world -> tensor parallel (column/row sharded W4A8 layers, one
    exchange after o_proj and after down_proj; same global batch, strong scaling), tp == 1 -> one replica per GPU
    (weak scaling, no data-path collective).  Same protocol as the headline (real prefill, graph replay, max over ranks)."""
    import torch.distributed as dist
    from omniserve_b200.model import DecodeGraph, LlamaW4A8
    model = LlamaW4A8(cfg, dev, rank if tp > 1 else 0, tp, seed=0 if tp > 1 else rank)
    BATCH_ = batch
    max_ctx = PROMPT_LEN + GEN_LEN
    sub = min(PREFILL_SUB_BATCH, BATCH_)
    model.alloc(BATCH_, max_ctx, sub * PROMPT_LEN)
    g = torch.Generator().manual_seed(42)
    prompts = torch.randint(0, cfg.vocab_size, (BATCH_, PROMPT_LEN), generator=g)
    first, chunk_ms = [], []
    for s0 in range(0, BATCH_, sub):
        toks = prompts[s0:s0 + sub].reshape(-1).to(dev)
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record()
        first.append(model.prefill(toks, [PROMPT_LEN] * sub, seq_offset=s0))
        c1.record()
        chunk_ms.append((c0, c1))
    torch.cuda.synchronize()
    per_chunk = sorted(x.elapsed_time(y) for x, y in chunk_ms)
    prefill_ms = (sum(per_chunk[:-1]) * len(per_chunk) / max(1, len(per_chunk) - 1)) if len(per_chunk) > 1 else per_chunk[0]
    collective = "none (independent replicas)" if tp == 1 else \
        "NCCL all-reduce (fp16 sum, [batch, hidden]) after o_proj and after down_proj, inside the CUDA graph"
    if tp > 1 and os.environ.get("OB_PEER_ALLREDUCE", "1") != "0":
        try:   # all-reduce fused into the following add+norm+quant kernel over NVLink peer memory
            model.enable_peer_allreduce()
            collective = ("all-reduce fused into the add+norm+quant kernel that consumes it: partial sums read from NVLink "
                          "peer (symmetric) memory, per-block epoch flags, no NCCL call in the decode layers")
        except Exception as e:  # symmetric memory unavailable: keep NCCL
            print("peer all-reduce unavailable, using NCCL:", repr(e)[:200], file=sys.stderr)
    graph = DecodeGraph(model, max_ctx)
    graph.tokens.copy_(torch.cat(first))
    for _ in range(max(3, warmup)):
        graph.graph.replay()
    dist.barrier(); torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(steps):
        graph.graph.replay()
    t1.record()
    dist.barrier(); torch.cuda.synchronize()
    tms = torch.tensor([t0.elapsed_time(t1)], device=dev)
    dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    ms = float(tms.item())
    del graph, model
    torch.cuda.empty_cache()
    reps = world if tp == 1 else 1
    return {"value": BATCH_ * reps * steps / (ms / 1e3), "unit": "tok/s", "ms_per_step": ms / steps, "steps": steps,
            "parallelism": f"tp{world}" if tp > 1 else f"dp{world}", "scaling": "strong" if tp > 1 else "weak",
            "global_batch": BATCH_ * reps, "model": tag or "Llama-3-8B",
            "prefill_tok_per_s": BATCH_ * reps * PROMPT_LEN / (prefill_ms / 1e3),
            "collective": collective}


def dump_outputs(d, arrays):
    """What the last timed step computed, as d/<name>.npy: integers (token ids) as float64, everything else as float32."""
    os.makedirs(d, exist_ok=True)
    for name, x in arrays.items():
        x = x.detach().cpu()
        x = x.double() if not x.is_floating_point() else x.float()
        np.save(os.path.join(d, f"{name}.npy"), x.numpy())


def bench_c3(a, real_stdout):
    """BASELINE config 3: LServe sparse decode, Llama-3-8B-Instruct-Gradient-1048k shape, 256K context, bs = 1 (1 GPU).
    Harness semantics of scripts/lserve_benchmark (lserve_benchmark.py:79-144): per-token decode latency at a fixed context;
    the context (prompt) stage is NOT run -- its attention is third-party flash / block-sparse attention outside this
    repository's scope -- pages are filled with valid random KV4 data and statistics instead (stated in `data`)."""
    from omniserve_b200.lserve_model import LServeDecodeGraphs, LServeDecoder
    from omniserve_b200.model import LlamaConfig
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    cfg = LlamaConfig.llama3_8b()
    fx = json.load(open(os.path.join(ROOT, "tests", "golden", "head_split_llama3_8b_1048k_s50.json")))
    ctx = int(os.environ.get("OB_C3_CTX", 262144))
    dec = LServeDecoder(cfg, fx["retrieval_head_flags"], dev)
    dec.alloc(ctx + 64)
    dec.fill_random(ctx)
    graphs = LServeDecodeGraphs(dec, ctx)
    interval = dec.sp.selector_update_interval
    pin_in = torch.zeros((1,), dtype=torch.int64).pin_memory()
    pin_out = torch.zeros((1,), dtype=torch.int64).pin_memory()

    def run(n, e2e=False):
        for i in range(n):
            if e2e:
                graphs.tokens.copy_(pin_in, non_blocking=True)
            graphs.step(i % interval == 0)
            if e2e:
                pin_out.copy_(graphs.out, non_blocking=True)
                torch.cuda.current_stream().synchronize()
                pin_in.copy_(pin_out)

    def timed(n, e2e=False):
        torch.cuda.synchronize()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record(); run(n, e2e); t1.record(); torch.cuda.synchronize()
        return t0.elapsed_time(t1)
    steps = a.steps
    run(max(3, a.warmup))
    sampler = ClockSampler(0); sampler.start()
    ms = timed(steps)
    clocks = sampler.stop()
    ms_e2e = timed(steps, e2e=True)
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, {"next_tokens": graphs.out})

    def one(sel, n=8):
        torch.cuda.synchronize()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(n):
            graphs.step(sel)
        t1.record(); torch.cuda.synchronize()
        return t0.elapsed_time(t1) / n
    ms_sel, ms_reuse = one(True), one(False)
    hbm_peak, _, peak_src = peaks()
    P = dec.dyn[0].shape[-1]
    g = cfg.num_attention_heads // cfg.num_key_value_heads
    attn_bytes = sum(hr * g * P * 64 * 136 + hs * (dec.sink + dec.local) * 136 for hr, hs in zip(dec.hr, dec.hs))
    stats_bytes = sum(hr * (ctx // 64) * 2 * 4 * 128 * 2 for hr in dec.hr)             # selector, every `interval` steps
    weight_bytes = dec.m.weight_bytes() + dec.m.lm_head.numel() * 2
    floor_ms = (weight_bytes + attn_bytes + stats_bytes / interval) / hbm_peak / 1e6
    line = {
        "metric": "LServe sparse decode tok/s, Llama-3-8B-Instruct-Gradient-1048k W4A8KV4, 256K ctx, bs=1", "value": steps / (ms / 1e3),
        "unit": "tok/s", "n_gpus": 1, "steps": steps, "warmup": max(3, a.warmup), "ms_per_step": ms / steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "int8 (W4A8, s32 accumulate) + fp16 KV4 attention",
        "data": "synthetic (random-init weights; KV pages and kmax/kmin statistics filled with valid random data -- the context stage is not run)",
        "config": {"workload": "BASELINE config 3: LServe sparse decode (static sparsity 0.5 head split from attn_patterns, dynamic budget "
                               "4096 tokens = 64 pages per retrieval q-head, selector every 4 steps, sink 128 + local 256 streaming heads)",
                   "ctx": ctx, "global_batch": 1, "parallelism": "tp1", "cuda_graph": True, "layers": cfg.num_hidden_layers,
                   "retrieval_kv_heads_per_layer": dec.hr, "kv_pool_gb": dec.kv_bytes() / 1e9,
                   "l2": "per-step working set (3.5 GB W4 weights + 1 GB lm_head) >> 126 MB L2; no flush needed"},
        "e2e": {"value": steps / (ms_e2e / 1e3), "unit": "tok/s", "h2d_bytes_per_step": 8, "d2h_bytes_per_step": 8, "ms_per_step": ms_e2e / steps},
        "gpu_launches": int((10 * cfg.num_hidden_layers + 1) * steps + 2 * sum(1 for h in dec.hr if h) * steps / interval),
        "clocks": clocks,
        "per_token_latency_ms": {"mean": ms / steps, "selector_step": ms_sel, "reuse_step": ms_reuse},
        "roofline": {"bound": "hbm", "kernel": "whole decode step (weights at M=1 + sparse KV4 attention + selector statistics / 4)",
                     "achieved": (weight_bytes + attn_bytes + stats_bytes / interval) / (ms / steps) / 1e6, "peak": hbm_peak, "unit": "GB/s",
                     "frac": floor_ms / (ms / steps), "traffic": None, "peak_source": peak_src,
                     "algorithmic_bytes": {"weights_and_lm_head": weight_bytes, "sparse_attention": attn_bytes,
                                           "selector_statistics_per_selector_step": stats_bytes}},
        "step_floor_ms_at_measured_hbm": floor_ms,
    }
    if not a.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline(LlamaConfig.llama3_8b())
        line["cpu_baseline"]["sample"] += " (dense bs=64 layer of configs[1]; the C3 workload has no separate CPU port)"
    real_stdout.write(json.dumps(line) + "\n")
    real_stdout.flush()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=256)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--layers", type=int, default=0, help="debug only: fewer layers (result is then marked invalid)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--workload", default="c2", choices=["c2", "c3"],
                    help="c2 = BASELINE configs[1] (Llama-3-8B bs=64 in=1024 out=512, the headline); c3 = configs[2] (LServe sparse "
                         "decode, 256K context, bs=1, one GPU)")
    ap.add_argument("--parallelism", default="auto", choices=["auto", "dp", "tp"],
                    help="N > 1: tp = tensor parallel over all GPUs (BASELINE north star: head / column sharding, one "
                         "exchange after o_proj and after down_proj; same global batch of 64 -> strong scaling), dp = one "
                         "bs=64 replica per GPU (weak scaling, no data-path collective).  auto = tp as the headline, with the "
                         "dp measurement added under \"dp\".")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (sampled next tokens; c2 also the final "
                         "hidden state of every sequence) as DIR/<name>.npy; the inputs are seeded, so runs with the same "
                         "arguments can be compared output for output")
    a = ap.parse_args()
    # Keep stdout clean for the ONE JSON line: libraries (NCCL banner, warnings) print to fd 1 in worker processes.
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    sys.stdout = sys.stderr

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if a.workload == "c3":
        return bench_c3(a, real_stdout) if rank == 0 and a.impl == "ours" else 0
    if a.impl == "reference" and rank != 0:
        return 0  # the reference is single-GPU, single-process (SURVEY.md F1): rank 0 alone runs it
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    use_dist = world > 1 and a.impl == "ours"
    if use_dist:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    mode = "tp" if a.parallelism in ("auto", "tp") else "dp"
    tp = world if (use_dist and mode == "tp") else 1
    replicas = world if (use_dist and mode == "dp") else 1

    from omniserve_b200.model import DecodeGraph, LlamaConfig, LlamaW4A8, Ops, kernel_launches_per_decode_step
    cfg = LlamaConfig.llama3_8b()
    if a.layers:
        cfg.num_hidden_layers = a.layers
    hbm_peak, bf16_peak, peak_src = peaks()

    if a.impl == "reference":
        try:
            ops = Ops(ref_loader())
        except Exception as e:  # oracle/_ref not shipped
            real_stdout.write(json.dumps({"impl": "reference", "unavailable": f"oracle/_ref not built: {e}"}) + "\n")
            real_stdout.flush()
            return 0
        model = LlamaW4A8(cfg, dev, 0, 1, fuse_silu_quant=False, ops=ops)
    else:
        model = LlamaW4A8(cfg, dev, rank if tp > 1 else 0, tp, seed=rank if replicas > 1 else 0)
    max_ctx = PROMPT_LEN + GEN_LEN
    model.alloc(BATCH, max_ctx, PREFILL_SUB_BATCH * PROMPT_LEN)

    # ---------------------------------------------------------------- prefill (fills the KV4 pages)
    g = torch.Generator().manual_seed(42)
    prompts = torch.randint(0, cfg.vocab_size, (BATCH, PROMPT_LEN), generator=g)
    skip_prefill = os.environ.get("OB_BENCH_SKIP_PREFILL") == "1"  # profiling aid only: result marked invalid
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    first = []
    if skip_prefill:
        for pool in model.kv.k_pools + model.kv.v_pools:
            u8 = pool.view(torch.uint8)
            u8.random_(0, 256)
            sz = u8[:, model.hkv * 4096:].view(torch.float16)
            sz[:, :model.hkv * 64] = 0.25
            sz[:, model.hkv * 64:] = 7.5
        model.context_lens.fill_(PROMPT_LEN)
        first = [torch.randint(0, cfg.vocab_size, (BATCH,), generator=g).to(dev)]
    else:
        chunk_ms = []
        for s in range(0, BATCH, PREFILL_SUB_BATCH):
            toks = prompts[s:s + PREFILL_SUB_BATCH].reshape(-1).to(dev)
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            c0.record()
            first.append(model.prefill(toks, [PROMPT_LEN] * PREFILL_SUB_BATCH, seq_offset=s))
            c1.record()
            chunk_ms.append((c0, c1))
    e1.record()
    torch.cuda.synchronize()
    prefill_ms = e0.elapsed_time(e1)
    if not skip_prefill:
        per_chunk = [a_.elapsed_time(b_) for a_, b_ in chunk_ms]
        print("prefill chunk ms:", [round(x, 1) for x in per_chunk], file=sys.stderr)
        # the first chunk pays one-time library initialisation (cuDNN SDPA plan, tensor-map encodes): report steady state
        prefill_ms_steady = sum(sorted(per_chunk)[:-1]) * len(per_chunk) / max(1, len(per_chunk) - 1)
    else:
        prefill_ms_steady = prefill_ms
    first = torch.cat(first)

    # ---------------------------------------------------------------- decode
    budget = GEN_LEN - 1  # steps until the page budget is exhausted
    pinned_in = torch.zeros((BATCH,), dtype=torch.int64).pin_memory()
    pinned_out = torch.zeros((BATCH,), dtype=torch.int64).pin_memory()
    pinned_in.copy_(first.cpu())

    collective = None
    if a.impl == "ours":
        if tp > 1:
            collective = "NCCL all-reduce (fp16 sum, [64, 4096]) after o_proj and after down_proj, inside the CUDA graph"
            if os.environ.get("OB_PEER_ALLREDUCE", "1") != "0":
                try:   # all-reduce fused into the following add+norm+quant kernel over NVLink peer memory
                    model.enable_peer_allreduce()
                    collective = ("all-reduce fused into the add+norm+quant kernel that consumes it: every rank's row-parallel "
                                  "partial sums are read straight from NVLink peer (symmetric) memory, per-block epoch flags, "
                                  "no NCCL call in the decode layers")
                except Exception as e:  # symmetric memory unavailable: keep NCCL
                    print("peer all-reduce unavailable, using NCCL:", repr(e)[:200], file=sys.stderr)
        graph = DecodeGraph(model, max_ctx)
        graph.tokens.copy_(first)

        def step():
            graph.graph.replay()

        tokens_buf, out_buf = graph.tokens, graph.out
    else:
        model.prepare_decode()
        tokens_buf = first.clone()
        out_buf = torch.zeros_like(tokens_buf)

        def step():
            nxt = model.decode_step(tokens_buf, max_ctx)
            out_buf.copy_(nxt)
            tokens_buf.copy_(nxt)

    state = {"done": 0}

    def run_steps(n, e2e=False):
        for _ in range(n):
            if state["done"] >= budget:  # wrap the context back to the prompt length (pages are overwritten)
                model.context_lens.fill_(PROMPT_LEN)
                state["done"] = 0
            if e2e:
                tokens_buf.copy_(pinned_in, non_blocking=True)
            step()
            if e2e:
                pinned_out.copy_(out_buf, non_blocking=True)
                torch.cuda.current_stream().synchronize()
                pinned_in.copy_(pinned_out)
            state["done"] += 1

    def barrier():
        if use_dist:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(n, e2e=False):
        barrier()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        run_steps(n, e2e)
        t1.record()
        barrier()
        ms = t0.elapsed_time(t1)
        if use_dist:
            tms = torch.tensor([ms], device=dev)
            dist.all_reduce(tms, op=dist.ReduceOp.MAX)
            ms = float(tms.item())
        return ms

    run_steps(max(3, a.warmup))
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ctx_start = PROMPT_LEN + state["done"]
    ms = timed(a.steps)
    clocks = sampler.stop() if rank == 0 else None
    run_steps(3, e2e=True)
    ms_e2e = timed(a.steps, e2e=True)
    if a.dump_outputs and rank == 0:
        h, delta = model.last_decode_state
        outs = {"next_tokens": out_buf}
        if torch.is_tensor(delta):   # hidden state after the last layer, before the final norm
            outs["final_hidden"] = h.float() + delta.float()
        dump_outputs(a.dump_outputs, outs)

    value = BATCH * replicas * a.steps / (ms / 1e3)
    e2e_value = BATCH * replicas * a.steps / (ms_e2e / 1e3)

    # ---------------------------------------------------------------- per-kernel roofline (rank 0 shapes)
    mid_ctx = PROMPT_LEN + GEN_LEN // 2
    kt, gemm_bytes, attn_bytes = time_kernels(model, mid_ctx)
    gemm_ms = sum(kt[k] for k in gemm_bytes)
    gemm_b = sum(gemm_bytes.values())
    kernels = {
        "w4a8_gemm(decode,4 launches/layer)": {"ms_per_layer": gemm_ms, "algorithmic_bytes": gemm_b,
                                                "gbs": gemm_b / gemm_ms / 1e6, "frac_hbm": gemm_b / gemm_ms / 1e6 / hbm_peak,
                                                "per_shape_ms": {k: kt[k] for k in gemm_bytes}},
        "kv4_decode_attention": {"ms_per_layer": kt["attention"], "algorithmic_bytes": attn_bytes, "ctx": mid_ctx,
                                 "gbs": attn_bytes / kt["attention"] / 1e6,
                                 "frac_hbm": attn_bytes / kt["attention"] / 1e6 / hbm_peak},
    }
    dom = "w4a8_gemm(decode,4 launches/layer)" if gemm_ms >= kt["attention"] else "kv4_decode_attention"
    roof = {"bound": "hbm", "kernel": dom, "achieved": kernels[dom]["gbs"], "peak": hbm_peak, "unit": "GB/s",
            "frac": kernels[dom]["frac_hbm"], "traffic": (ncu_traffic()[0].get(dom) if tp == 1 else None), "peak_source": peak_src,
            "traffic_source": "ncu --set full dram__bytes_read.sum + dram__bytes_write.sum, cold launches: " + ncu_traffic()[1],
            "share_of_step": cfg.num_hidden_layers * kernels[dom]["ms_per_layer"] / (ms / a.steps)}
    prefill = None
    if a.impl == "ours" and tp == 1 and not skip_prefill:
        pg = prefill_gemm_tops(model)
        i8_peak, i8_src = int8_peak() if rank == 0 else (INT8_PEAK_RECORDED, "")
        prefill = {"tok_per_s": BATCH * replicas * PROMPT_LEN / (prefill_ms_steady / 1e3), "ms": prefill_ms_steady,
                   "ms_incl_first_chunk_init": prefill_ms, "gemm_M8192": pg,
                   "int8_peak_tops": i8_peak, "int8_peak_source": i8_src,
                   "gemm_frac_of_int8_peak": pg["all"]["tops"] / i8_peak}

    step_floor_ms = (model.weight_bytes() + model.lm_head.numel() * 2
                     + BATCH * mid_ctx * model.hkv * 136 * cfg.num_hidden_layers) / hbm_peak / 1e6
    want_dp = use_dist and mode == "tp" and a.parallelism == "auto" and os.environ.get("OB_BENCH_DP", "1") != "0"
    want_c4 = use_dist and mode == "tp" and world == 8 and os.environ.get("OB_BENCH_C4", "1") != "0"
    if rank != 0 and not (want_dp or want_c4):
        return 0
    line = {
        "metric": "decode tok/s Llama-3-8B W4A8KV4 bs=64",
        "value": value, "unit": "tok/s", "n_gpus": world if use_dist else 1, "steps": a.steps, "warmup": max(3, a.warmup),
        "ms_per_step": ms / a.steps, "higher_is_better": True,
        "scaling": ("weak" if mode == "dp" else "strong") if use_dist else "weak",
        "vs_baseline": None,
        "dtype": "int8 (W4A8, s32 accumulate) + fp16 KV4 attention", "data": "synthetic (random-init weights, random prompts)",
        "config": {"workload": "Llama-3-8B W4A8KV4 per-channel, qserve_benchmark.py semantics bs=64 in=1024 out=512: "
                               "decode steps after a real 64x1024 prefill", "global_batch": BATCH * replicas, "prompt_len": PROMPT_LEN,
                   "ctx_at_first_timed_step": ctx_start,
                   "parallelism": (f"dp{replicas} (one bs={BATCH} replica per GPU, no data-path collective)" if replicas > 1
                                   else f"tp{tp}"), "collective": collective, "cuda_graph": a.impl == "ours",
                   "l2": "per-step working set (3.5 GB W4 weights + 2.8 GB KV4 + 1 GB lm_head) >> 126 MB L2; no flush needed",
                   "layers": cfg.num_hidden_layers},
        "e2e": {"value": e2e_value, "unit": "tok/s", "h2d_bytes_per_step": BATCH * replicas * 8,
                "d2h_bytes_per_step": BATCH * replicas * 8,
                "ms_per_step": ms_e2e / a.steps},
        "gpu_launches": (kernel_launches_per_decode_step(cfg, True) * a.steps * replicas) if a.impl == "ours" else 0,
        "clocks": clocks, "roofline": roof, "kernels": kernels, "prefill": prefill,
        "step_floor_ms_at_measured_hbm": step_floor_ms,
    }
    if a.layers:
        line["invalid"] = "debug run with fewer layers"
    if skip_prefill:
        line["invalid"] = "OB_BENCH_SKIP_PREFILL=1: KV pages filled with random bytes (profiling aid)"
    if a.impl == "reference":
        line["impl"] = "reference"
        line["config"]["note"] = ("reference = mit-han-lab/omniserve's own CUDA kernels (Ampere-era mma.sync / CUDA-core MMHA) "
                                  "rebuilt for sm_100 by oracle/build_ref.py, same decoder-step sequencing, eager launches")
    if not a.no_cpu_baseline and rank == 0 and world == 1:   # contract: rank 0 at N = 1 only
        line["cpu_baseline"] = cpu_baseline(LlamaConfig.llama3_8b())

    def emit():
        real_stdout.write(json.dumps(line) + "\n")
        real_stdout.flush()

    if want_dp or want_c4:
        # Secondary measurements.  They must never take the headline down: exceptions are recorded, and a watchdog prints
        # the line and ends the process if one hangs.
        done = threading.Event()

        def watchdog():
            if not done.wait(timeout=float(os.environ.get("OB_BENCH_SECONDARY_TIMEOUT", "420"))):
                if rank == 0:
                    line.setdefault("dp", {"error": "secondary measurement timed out"})
                    emit()
                os._exit(0)
        threading.Thread(target=watchdog, daemon=True).start()
        del graph, model
        torch.cuda.empty_cache()
        if want_dp:   # one bs=64 replica per GPU, no data-path collective (how an 8B model is usually served)
            try:
                line["dp"] = measure_secondary(cfg, dev, rank, world, min(a.steps, 64), a.warmup, tp=1)
            except Exception as e:
                line["dp"] = {"error": repr(e)[:300]}
        if want_c4:   # BASELINE config 4: Llama-3-70B W4A8KV4, tensor-parallel 8, bs = 16
            try:
                c70 = LlamaConfig.llama3_70b()
                line["c4"] = measure_secondary(c70, dev, rank, world, min(a.steps, 32), a.warmup, tp=world, batch=16,
                                               tag="Llama-3-70B (BASELINE config 4: TP=8, bs=16, in=1024)")
            except Exception as e:
                line["c4"] = {"error": repr(e)[:300]}
        done.set()
    if rank != 0:
        return 0
    emit()
    return 0


if __name__ == "__main__":
    sys.exit(main())
