"""Sampling pick timings on the GPU (CUDA events), printed as JSON lines with the GPU name and power limit.

    python tools/sample_bench.py [--iters N] [--steps N] [--skip-model]

1. zl_sample vs zl_argmax vs a torch implementation of the same contract (torch.sort + cumsum + searchsorted) on the same
   fp32 logits, V = 128256, T in {1, 8, 32, 64}; every row samples (top_p 0.9, top_k 50, rep 1.1 over 64 seen tokens).
2. Device-loop decode steps of the llama-3.1-8b preset (W4 GPTQ, synthetic weights) at batch 1 and 32: every task
   sampling (top_p 0.9, top_k 50, rep 1.1) against greedy, alternating the two, same decoder.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, pl = [s.strip() for s in out.split(",")]
        return name, pl
    except Exception:
        import torch
        return torch.cuda.get_device_name(0), "unknown"


def time_ms(fn, iters):
    import torch
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / iters


def torch_sample(logits, seen_mask, temperature, top_p, top_k, rep, u):
    """The same contract in torch ops: penalties, softmax, stable descending sort, cumsum, top-k cap, searchsorted."""
    import torch
    l = torch.where(seen_mask, torch.where(logits < 0, logits * rep, logits / rep), logits)
    p = torch.softmax(l / temperature, dim=-1)
    ps, order = torch.sort(p, dim=-1, descending=True, stable=True)
    cum = torch.cumsum(ps, dim=-1)
    P = torch.minimum(torch.full_like(cum[:, :1], top_p), cum[:, top_k - 1:top_k])
    v = (u[:, None] * P * cum[:, -1:]).contiguous()
    j = torch.searchsorted(cum, v).clamp_(max=cum.shape[1] - 1)
    return order.gather(1, j).squeeze(1)


def bench_ops(iters):
    import torch
    from zhilight_b200 import ops
    dev = torch.device("cuda:0")
    V = 128256
    rows = []
    for T in (1, 8, 32, 64):
        g = torch.Generator(device=dev).manual_seed(T)
        logits = torch.randn(T, V, device=dev, generator=g) * 3
        words = (V + 31) // 32
        seen_np = np.zeros((T, words), np.uint32)
        mask_np = np.zeros((T, V), bool)
        rng = np.random.default_rng(T)
        for t in range(T):
            toks = rng.integers(0, V, 64)
            mask_np[t, toks] = True
            for tok in toks:
                seen_np[t, tok >> 5] |= np.uint32(1 << (tok & 31))
        seen = torch.from_numpy(seen_np.view(np.int32)).to(dev)
        mask = torch.from_numpy(mask_np).to(dev)
        params = ops.sample_params([dict(top_p=0.9, top_k=50, repetition_penalty=1.1, seed=t) for t in range(T)], dev, V)
        cnt = torch.zeros(T, dtype=torch.int32, device=dev)
        u = torch.rand(T, device=dev)
        t_s = time_ms(lambda: ops.sample(logits, params, seen, cnt), iters)
        t_a = time_ms(lambda: ops.argmax(logits), iters)
        t_t = time_ms(lambda: torch_sample(logits, mask, 1.0, 0.9, 50, 1.1, u), max(5, iters // 4))
        rows.append(dict(bench="sample_op", V=V, T=T, zl_sample_us=round(t_s * 1e3, 2), zl_argmax_us=round(t_a * 1e3, 2),
                         torch_sort_us=round(t_t * 1e3, 2)))
    return rows


def bench_model(steps, rounds):
    import torch
    from zhilight_b200.llama import LlamaDecoder, MODEL_PRESETS
    cfg = dict(MODEL_PRESETS["llama-3.1-8b"])
    rows = []
    for B in (1, 32):
        dec = LlamaDecoder(quant_type=5, group_size=128, sym=True, max_batch=B, max_seq=2048, **cfg)
        dec.init_synthetic(0)
        tok = np.arange(B, dtype=np.int32) * 17 % cfg["vocab_size"]
        res = {"greedy": [], "sample": []}
        for r in range(rounds):
            for mode in ("greedy", "sample"):
                for t in range(B):
                    if mode == "sample":
                        dec.set_sampling(t, top_p=0.9, top_k=50, repetition_penalty=1.1, seed=1000 * r + t)
                    else:
                        dec.clear_sampling(t)
                dec.set_state(tok, np.full(B, 512, np.int32))
                for _ in range(3):
                    dec.step_device(B)
                dec.sync()
                t0 = time.perf_counter()
                for _ in range(steps):
                    dec.step_device(B)
                dec.sync()
                res[mode].append((time.perf_counter() - t0) / steps)
        dec.close()
        g, s = np.median(res["greedy"]), np.median(res["sample"])
        rows.append(dict(bench="decode_step", preset="llama-3.1-8b", batch=B, greedy_ms=round(g * 1e3, 4),
                         sample_ms=round(s * 1e3, 4), sample_cost_us=round((s - g) * 1e6, 2),
                         sample_cost_pct=round(100 * (s - g) / g, 2), greedy_tok_s=round(B / g, 1),
                         sample_tok_s=round(B / s, 1), greedy_ms_all=[round(x * 1e3, 4) for x in res["greedy"]],
                         sample_ms_all=[round(x * 1e3, 4) for x in res["sample"]]))
        del dec
        torch.cuda.empty_cache()
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--skip-model", action="store_true")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("sample_bench needs a CUDA device")
    from zhilight_b200 import build
    build.build()
    name, pl = gpu_info()
    rows = bench_ops(a.iters)
    if not a.skip_model:
        rows += bench_model(a.steps, a.rounds)
    for r in rows:
        r.update(gpu=name, power_limit=pl)
        print(json.dumps(r), flush=True)


if __name__ == "__main__":
    main()
