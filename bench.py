#!/usr/bin/env python
"""bench.py -- decode tokens/s of Llama-3.1-8B GPTQ-int4 (g128) on B200, the BASELINE.json metric.

    python bench.py --gpus N --steps K --warmup W [--batch B] [--prompt P] [--impl reference] [--model NAME]

A "step" is one decode step of the whole batch through the hot path (32 layers of W4A16 Linear +
decode attention + RMSNorm/RoPE fusions, lm_head, greedy pick).  Random-init weights of the named
architecture in HF-GPTQ layout, synthetic prompt token ids ("data": "synthetic").

  value   tokens/s with inputs resident in HBM: the step replays on the device, feeding the picked token
          back on the device (K steps between CUDA events on the driver's stream, max over ranks).
  e2e     the same step through the public host-buffer API (zl_llama_decode): pinned-host token ids and
          positions are copied H2D and the picked tokens are read back D2H inside every timed step.
  roofline  the dominant kernel (W4A16 GEMM): all 128 GEMM launches of a step replayed on their own real
          weights between CUDA events; achieved = algorithmic bytes / time against MEASURED_PEAKS.json.
  cpu_baseline  the oracle's dequant-to-bf16 torch CPU path on a bounded sample (1 of 32 layers + lm_head),
          a reported baseline, not a target.

--impl reference times that CPU path as the whole arm (the reference has no CPU implementation of its own;
SURVEY.md section 8d names this torch dequant path as the side-by-side baseline).

N > 1: tensor parallel over the N GPUs of one node (the reference's row/column split), one process per GPU; the
partial sums of the row-parallel Linears are exchanged with the one-shot NVLink peer-memory all-reduce
(zhilight_b200/csrc/comm.cu), NCCL only bootstraps.  value = tokens/s of the whole TP group ("scaling": "strong").
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def read_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu = gpu_index
        self.samples = []
        self.stamps = []          # host time of every sample
        self.t_region = None      # mark_region_start(): only samples taken after it describe the timed region
        self.stop_flag = False
        self.proc = None

    def mark_region_start(self):
        self.t_region = time.time()

    def _run_nvml(self):
        """5 ms NVML polling (nvidia_ml_py): enough samples inside a ~100 ms timed region.  Any failure falls back to
        the nvidia-smi loop below."""
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(self.gpu)
        mx = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
        get_reasons = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
            pynvml.nvmlDeviceGetCurrentClocksThrottleReasons
        bits = {"sw_power_cap": 0x4, "hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}
        while not self.stop_flag:
            sm = pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
            r = int(get_reasons(h))
            flags = ["Active" if r & bits[k] else "Not Active"
                     for k in ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")]
            self.samples.append([str(self.gpu), str(sm), str(mx), "", ""] + flags)
            self.stamps.append(time.time())
            time.sleep(0.005)

    def run(self):
        try:
            self._run_nvml()
            return
        except Exception:
            pass
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                if self.stop_flag:
                    break
                self.samples.append([x.strip() for x in line.split(",")])
                self.stamps.append(time.time())
        except Exception:
            pass

    def finish(self):
        self.stop_flag = True
        if self.proc:
            self.proc.terminate()
        sm, mx, reasons = [], [], set()
        picked = [s for s, ts in zip(self.samples, self.stamps) if self.t_region is None or ts >= self.t_region]
        for s in (picked or self.samples):   # too short a region for the sampling period: fall back to all samples
            try:
                sm.append(float(s[1]))
                mx.append(float(s[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def model_cfg(name):
    from zhilight_b200.llama import MODEL_PRESETS
    return dict(MODEL_PRESETS[name])


def gptq_shift(kk):
    return (kk >> 1) * 4 + (kk & 1) * 16


class CpuReference:
    """The CPU baseline (SURVEY.md 8d "reference side-by-side (ii)"): dequantise W4 -> bf16 on every call (what a
    dequant-to-bf16 path pays), then x @ W^T in torch on the host cores.  One layer's seven linears are materialised; a
    full decode step runs them num_layers times (the packed weights of a layer, 109 MB, do not stay in the CPU caches)
    and the lm_head once.  Inputs are generated outside the timed region."""

    def __init__(self, cfg, quant, batch, threads=None):
        import numpy as np
        import torch
        self.torch = torch
        # torch's bf16 matmul stops scaling (and oversubscribes badly) beyond a few dozen threads
        self.threads = threads or min(os.cpu_count() or 1, 32)
        torch.set_num_threads(self.threads)
        self.cfg, self.quant, self.batch = cfg, quant, batch
        d_model, d, ff, v = cfg["dim_model"], cfg["dim_head"], cfg["dim_ff"], cfg["vocab_size"]
        shapes = [(d_model, cfg["num_heads"] * d), (d_model, cfg["num_kv_heads"] * d), (d_model, cfg["num_kv_heads"] * d),
                  (cfg["num_heads"] * d, d_model), (d_model, ff), (d_model, ff), (ff, d_model)]
        rng = np.random.default_rng(0)
        self.lin = []
        for k, n in shapes:
            x = torch.from_numpy(rng.standard_normal((batch, k)).astype(np.float32)).bfloat16()
            if quant:
                qw = torch.from_numpy(rng.integers(0, 2 ** 31, size=(n, k // 8), dtype=np.int64).astype(np.int32))
                qz = torch.from_numpy(rng.integers(0, 16, size=(n, k // 128), dtype=np.int64).astype(np.uint8))
                sc = torch.from_numpy((0.002 + 0.004 * rng.random((n, k // 128))).astype(np.float32)).bfloat16()
                self.lin.append((x, qw, qz, sc, k, n))
            else:
                self.lin.append((x, torch.from_numpy(rng.standard_normal((n, k)).astype(np.float32)).bfloat16(), k, n))
        self.lm = torch.from_numpy(rng.standard_normal((v, d_model)).astype(np.float32) * 0.02).bfloat16()
        self.x_lm = torch.from_numpy(rng.standard_normal((batch, d_model)).astype(np.float32)).bfloat16()
        self.shifts = torch.tensor([gptq_shift(i) for i in range(8)], dtype=torch.int32)

    def layer(self):
        for item in self.lin:
            if self.quant:
                x, qw, qz, sc, k, n = item
                # k-major unpack (q_gemm_k_major.cu:74-98 nibble order), (q - z) * s, to bf16 once per call
                q = ((qw.unsqueeze(-1) >> self.shifts) & 0xF).reshape(n, k).to(self.torch.bfloat16)
                w = (q - qz.to(self.torch.bfloat16).repeat_interleave(128, dim=1)) * sc.repeat_interleave(128, dim=1)
                _ = x @ w.T
            else:
                x, w, k, n = item
                _ = x @ w.T

    def step(self):
        """one whole decode step: every layer + lm_head"""
        for _ in range(self.cfg["num_layers"]):
            self.layer()
        _ = self.x_lm @ self.lm.T

    def run(self, max_steps, budget_s):
        """Times WHOLE steps (no extrapolation): as many of `max_steps` as fit `budget_s`, at least one.
        Returns (tokens/s, seconds per step, steps executed, description)."""
        self.layer()                                   # thread pool / allocator warm-up, not a step
        times = []
        t_all = time.perf_counter()
        while len(times) < max_steps:
            t0 = time.perf_counter()
            self.step()
            times.append(time.perf_counter() - t0)
            if (time.perf_counter() - t_all) + times[-1] > budget_s:
                break
        t_step = sum(times) / len(times)
        sample = ("%d whole decode steps timed (%d layers x 7 linears%s, M=%d, + lm_head; one layer's weight set reused for "
                  "every layer), %d torch threads" % (len(times), self.cfg["num_layers"],
                                                      " W4->bf16 dequant + matmul" if self.quant else " bf16 matmul",
                                                      self.batch, self.threads))
        return self.batch / t_step, t_step, len(times), sample


def run_reference_arm(args, cfg, workload):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    quant = args.model != "llama-3.2-1b"
    ref = CpuReference(cfg, quant, args.batch)
    v, t_step, n_steps, sample = ref.run(max(1, args.steps), budget_s=args.ref_budget)
    out = {
        "impl": "reference", "metric": "decode tokens/s", "value": v, "unit": "tokens/s", "n_gpus": args.gpus,
        "steps": n_steps, "steps_requested": args.steps, "warmup": 0, "ms_per_step": t_step * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": workload},
        "cpu_baseline": {"value": v, "unit": "tokens/s", "cores": ref.threads, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "whole steps are timed; the step count is bounded by --ref-budget seconds instead of --steps",
    }
    print(json.dumps(out))


TINY = dict(num_layers=2, dim_model=256, num_heads=4, num_kv_heads=2, dim_head=64, dim_ff=512, vocab_size=512,
            eps=1e-5, rope_theta=10000.0, rope_llama3=None)
LAYERS8B = dict(num_layers=3, dim_model=4096, num_heads=32, num_kv_heads=8, dim_head=128, dim_ff=14336, vocab_size=2048,
                eps=1e-5, rope_theta=500000.0, rope_llama3=dict(factor=8.0, low=1.0, high=4.0, orig=8192.0))


def run_tp_parity(rank, world, local_rank):
    """Correctness gate of every N > 1 line (the oracle is the CHECKER here, before any timed region): the fp16 one-shot
    all-reduce must equal the exact rank-ordered sum bit for bit, and TP decode of a tiny model and of three
    Llama-3.1-8B-shaped GPTQ layers must match oracle/model.py on every rank's vocabulary shard (rel L2 <= 3e-3).
    Rank 0 runs the oracle and broadcasts the reference logits.  Raises SystemExit(3) on failure."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from oracle import model as omodel, ops as oops
    from zhilight_b200 import dist as zdist
    from zhilight_b200.llama import LlamaDecoder
    dev = torch.device("cuda", local_rank)
    res = {}
    comm = zdist.TPComm(4 * 8192, rank, world)
    rng = np.random.default_rng(0)
    parts = [rng.standard_normal((4, 8192)).astype(np.float16) for _ in range(world)]
    resid = rng.standard_normal((4, 8192)).astype(np.float16)
    mine = torch.from_numpy(parts[rank]).to(dev)
    exact = True
    for it in range(4):      # both parities of the double-buffered inboxes
        out = comm.allreduce(mine, torch.from_numpy(resid).to(dev) if it % 2 else None)
        torch.cuda.synchronize()
        exp = oops.allreduce_exact(parts)
        if it % 2:
            exp = oops.residual_add(exp, resid)
        exact = exact and bool(np.array_equal(out.float().cpu().numpy(), exp))
    res["allreduce_bit_exact"] = exact
    comm.close()
    worst = 0.0
    for name, cfg, sym, scales in (("tiny", TINY, False, None), ("llama8b_layers", LAYERS8B, True, (0.0003, 0.0008))):
        if cfg["num_heads"] % world or cfg["num_kv_heads"] % world:
            continue
        sd = omodel.make_state_dict(cfg, 5, 128, sym, seed=2, scale_range=scales)
        dec = LlamaDecoder(quant_type=5, group_size=128, sym=sym, max_batch=2, max_seq=32, tp_rank=rank, tp_size=world, **cfg)
        c2 = zdist.TPComm(2 * cfg["dim_model"], rank, world)
        dec.set_comm(c2)
        dec.load_state_dict(zdist.shard_state_dict(sd, rank, world))
        orc = omodel.OracleLlama(cfg, sd, 5, 128, sym, "f16", fuse_norm=True) if rank == 0 else None
        tok = np.array([5, 99], dtype=np.int32)
        vs = cfg["vocab_size"] // world
        w_model = 0.0
        for step in range(4):
            pos = np.full(2, step, dtype=np.int32)
            nxt, logits = dec.decode(tok, pos, want_logits=True)       # this rank's vocabulary shard
            ref = torch.empty((2, cfg["vocab_size"]), dtype=torch.float32, device=dev)
            if rank == 0:
                ref.copy_(torch.from_numpy(orc.decode(tok, pos).astype(np.float32)))
            dist.broadcast(ref, 0)
            r = ref.cpu().numpy()[:, rank * vs:(rank + 1) * vs]
            w_model = max(w_model, float(np.linalg.norm(logits - r) / max(np.linalg.norm(r), 1e-30)))
            tok = nxt
        res["max_rel_" + name] = w_model
        res["kernels_per_step_" + name] = int(dec.stats(2)[1])
        worst = max(worst, w_model)
        dec.close()
        c2.close()
    t = torch.tensor([worst, 0.0 if exact else 1.0], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    res["max_rel"] = float(t[0])
    res["allreduce_bit_exact"] = bool(t[1] == 0.0)
    res["tolerance"] = 3e-3
    res["ok"] = bool(res["max_rel"] <= 3e-3 and res["allreduce_bit_exact"])
    if not res["ok"]:
        if rank == 0:
            print(json.dumps({"tp_parity": res, "error": "tensor-parallel parity check failed"}))
        raise SystemExit(3)
    return res


def measure_decode(dec, B, steps, warm, stream, barrier, sampler_gpu=None):
    """K device-resident steps between CUDA events on the driver's stream; returns (ms, clocks or None)."""
    import torch
    for _ in range(warm):
        dec.step_device(B)
    barrier()
    sampler = None
    if sampler_gpu is not None:
        sampler = ClockSampler(sampler_gpu)
        sampler.start()
        time.sleep(0.3)           # lets the nvidia-smi fallback start up; the NVML sampler is already polling
        sampler.mark_region_start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        dec.step_device(B)
    e1.record(stream)
    e1.synchronize()
    barrier()
    return e0.elapsed_time(e1), (sampler.finish() if sampler else None)


def ingest_prompt(dec, B, prompt_len, vocab, rng):
    import numpy as np
    prompt = rng.integers(0, vocab, size=(prompt_len, B)).astype(np.int32)
    pos = np.zeros(B, dtype=np.int32)
    for t in range(prompt_len):
        dec.set_state(prompt[t], pos)
        dec.step_device(B)
        pos += 1
    dec.sync()


def step_bytes_of(cfg, weight_bytes, B, ctx):
    return weight_bytes + B * ctx * cfg["num_layers"] * 2 * cfg["num_kv_heads"] * cfg["dim_head"] * 2


DUMP_LOGITS_BYTES = 60 << 20


def dump_outputs(out_dir, tokens, logits):
    """What the caller of the timed step receives: the greedy picks, and the logits they were picked from.  Inputs are
    seeded, so two builds can be compared array by array; logits larger than DUMP_LOGITS_BYTES keep a fixed sample of rows."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "next_tokens.npy"), tokens.astype(np.float64))
    if logits.nbytes > DUMP_LOGITS_BYTES:
        rows = np.sort(np.random.RandomState(0).choice(logits.shape[0], DUMP_LOGITS_BYTES // logits[0].nbytes, replace=False))
        logits = logits[rows]
    np.save(os.path.join(out_dir, "logits.npy"), logits.astype(np.float32))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=128)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--batch", type=int, default=1)
    ap.add_argument("--prompt", type=int, default=128)
    ap.add_argument("--model", default="llama-3.1-8b", choices=sorted(["llama-3.1-8b", "llama-3.2-1b", "tiny", "llama-3.1-70b",
                                                                       "qwen2-72b"]))
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-pdl", action="store_true")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the batch sweep / Llama-3.2-1B / reference-kernel extras of the N=1 line")
    ap.add_argument("--no-tp-parity", action="store_true", help="N > 1: skip the oracle parity gate (experiments only)")
    ap.add_argument("--tp-int8", action="store_true", help="int8 group-32 payload for the TP all-reduce")
    ap.add_argument("--requests", type=int, default=32, help="requests for the TTFT/TPOT p50 (0 = skip)")
    ap.add_argument("--ref-budget", type=float, default=120.0, help="--impl reference: seconds of whole CPU steps to time")
    ap.add_argument("--quant", choices=["default", "int8", "fp8"], default="default",
                    help="default: the model's BASELINE quantisation (GPTQ int4 for 8B, bf16 for 1B); int8 / fp8: W8A8 Linear rows")
    ap.add_argument("--prefill-chunk", type=int, default=128, help="tokens per chunked-prefill pass of the TTFT measurement")
    ap.add_argument("--fuse", type=int, default=2, help="0: one kernel per reference op; 1: +RMSNorm fused; 2: +qkv RoPE/KV epilogue")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs as DIR/next_tokens.npy (B) and DIR/logits.npy (B, vocab/N of "
                         "rank 0; a fixed sample of rows above %d MB), float64 / float32" % (DUMP_LOGITS_BYTES >> 20))
    args = ap.parse_args()

    cfg = model_cfg(args.model)
    quant_name = "bf16" if args.model == "llama-3.2-1b" else "gptq-int4-g128-sym"
    if args.quant != "default":
        quant_name = {"int8": "w8a8-int8 (AutoInt8)", "fp8": "w8a8-fp8-e4m3"}[args.quant]
    workload = "%s %s greedy decode, batch=%d, prompt=%d, new=%d" % (args.model, quant_name, args.batch, args.prompt,
                                                                     args.steps)
    if args.impl == "reference":
        run_reference_arm(args, cfg, workload)
        return

    import numpy as np
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the hot path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    from zhilight_b200 import build
    from zhilight_b200.llama import LlamaDecoder
    build.build()
    from zhilight_b200 import dist as zdist

    tp_parity = None
    if world > 1 and not args.no_tp_parity:
        tp_parity = run_tp_parity(rank, world, local_rank)

    dense = args.model == "llama-3.2-1b" or args.quant != "default"   # every non-W4 Linear path reports k_dense/k_w8a8
    qtype = {"default": 0 if args.model == "llama-3.2-1b" else 5, "int8": 2, "fp8": 7}[args.quant]
    W = max(args.warmup, 3)
    extras = world == 1 and not args.no_extras and not dense and args.model == "llama-3.1-8b"
    sweep = [b for b in (8, 32) if b != args.batch] if extras else []
    max_batch = max([args.batch] + sweep)
    max_seq = args.prompt + 2 * W + 2 * args.steps + 16 + (len(sweep) + 1) * (W + 40)
    dec = LlamaDecoder(quant_type=qtype, group_size=128, sym=True, dtype="bf16" if args.model == "llama-3.2-1b" else "f16",
                       max_batch=max_batch, max_seq=max_seq, use_pdl=not args.no_pdl, use_graph=not args.no_graph, fuse=args.fuse,
                       tp_rank=rank, tp_size=world, tp_int8=args.tp_int8,
                       prefill_chunk=args.prefill_chunk if (world == 1 and args.requests > 0) else 0, **cfg)
    comm = None
    if world > 1:
        comm = zdist.TPComm(max_batch * cfg["dim_model"], rank, world)
        dec.set_comm(comm)
    dec.init_synthetic(seed=1)
    B = args.batch
    rng = np.random.default_rng(0)
    stream = torch.cuda.ExternalStream(dec.stream())

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # synthetic prompts ingested through the same decode path (fills every task's KV buffers to `prompt` tokens)
    ingest_prompt(dec, max_batch, args.prompt, cfg["vocab_size"], rng)
    tok_all, pos_all = dec.get_state(max_batch)
    dec.set_state(tok_all[:B], pos_all[:B])

    # ---- value: device-resident loop ----
    launches0 = dec.lib.zl_launch_count(0)
    ms_dev, clocks = measure_decode(dec, B, args.steps, W, stream, barrier, sampler_gpu=local_rank)
    weight_bytes, kernels_per_step = dec.stats(B)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dec.get_state(B)[0], dec.logits(B))

    # sanity of the synthetic model: the logits of the last timed step must be finite (a NaN step costs the same time)
    tok, pos = dec.get_state(B)
    _, chk_logits = dec.decode(tok, pos, want_logits=True)
    logits_finite = bool(np.isfinite(chk_logits).all())

    # ---- e2e: host buffers in/out every step ----
    tok, pos = dec.get_state(B)
    for _ in range(W):
        tok = dec.decode(tok, pos)
        pos = pos + 1
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        tok = dec.decode(tok, pos)
        pos = pos + 1
    barrier()
    ms_e2e = (time.perf_counter() - t0) * 1e3

    if world > 1:
        tt = torch.tensor([ms_dev, ms_e2e], device="cuda", dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms_dev, ms_e2e = tt.tolist()

    peak, peak_kind = read_peaks()
    tokens = B * args.steps          # one TP group decodes B sequences, whatever its size
    value = tokens / (ms_dev * 1e-3)
    e2e_value = tokens / (ms_e2e * 1e-3)
    ctx_mid = args.prompt + W + args.steps // 2
    step_bytes = step_bytes_of(cfg, weight_bytes, B, ctx_mid)
    step_roof = step_bytes / (ms_dev / args.steps * 1e-3) / 1e9

    out = {
        "metric": "decode tokens/s", "value": value, "unit": "tokens/s", "n_gpus": world, "steps": args.steps,
        "warmup": W, "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": {"int8": "int8 x int8 -> int32 (W8A8), f16 activations", "fp8": "e4m3 x e4m3 -> f32 (W8A8), f16 activations"}.get(
            args.quant, "bf16" if dense else "f16 (W4A16: int4 weights, fp16 activations, fp32 accumulate)"),
        "data": "synthetic (random-init HF-GPTQ tensors: uniform nibbles recentred on the symmetric zero point, scales 0.002-0.006)",
        "config": {"workload": workload, "parallelism": "single GPU" if world == 1 else "tp%d (NVLink peer-memory exchange fused into the GEMMs, %s payload)" % (world, "int8-g32 (stand-alone kernel)" if args.tp_int8 else "fp16"),
                   "l2": "weights per step (%.2f GB) exceed L2 (126 MB); no explicit flush" % (weight_bytes / 1e9),
                   "pdl": not args.no_pdl, "cuda_graph": not args.no_graph, "fuse": args.fuse},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "tokens/s", "h2d_bytes_per_step": 8 * B, "d2h_bytes_per_step": 4 * B,
                "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": int(kernels_per_step) * args.steps if kernels_per_step else int(dec.lib.zl_launch_count(0) - launches0),
        "kernels_per_step": kernels_per_step,
        "logits_finite": logits_finite,
        "step_roofline": {"algorithmic_bytes_per_step": step_bytes, "achieved": step_roof, "peak": peak, "unit": "GB/s",
                          "frac": step_roof / peak},
    }
    if tp_parity is not None:
        out["tp_parity"] = tp_parity

    # ---- latency view of the same path (SURVEY 8d): TTFT = chunked prefill of a fresh prompt + first token,
    # TPOT = (t_total - TTFT) / (n_out - 1), both wall clock through the host API, p50 over --requests requests ----
    if world == 1 and args.requests > 0:
        n_out = 16
        plen = min(args.prompt, max_seq - n_out - 1)
        ttft, tpot = [], []
        for r in range(args.requests):
            ptoks = rng.integers(0, cfg["vocab_size"], size=plen).astype(np.int32)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            t_next = dec.prefill(0, ptoks)
            t1 = time.perf_counter()
            tk = np.array([t_next], dtype=np.int32)
            ps = np.array([plen], dtype=np.int32)
            for _ in range(n_out - 1):
                tk = dec.decode(tk, ps)
                ps = ps + 1
            t2 = time.perf_counter()
            ttft.append((t1 - t0) * 1e3)
            tpot.append((t2 - t1) * 1e3 / (n_out - 1))
        out["latency"] = {"ttft_ms_p50": float(np.median(ttft)), "tpot_ms_p50": float(np.median(tpot)),
                          "requests": args.requests, "prompt_tokens": plen, "new_tokens": n_out, "batch": 1,
                          "prefill": "chunked, %d tokens per pass (tcgen05 GEMMs)" % args.prefill_chunk}

    # ---- extras of the N = 1 line: BASELINE config 3 batch sizes and config 2, through the same harness ----
    if sweep:
        out["batch_sweep"] = {}
        for b in sweep:
            dec.set_state(tok_all[:b], pos_all[:b])
            ms_b, _ = measure_decode(dec, b, 32, W, stream, barrier)
            wb, kps = dec.stats(b)
            sb = step_bytes_of(cfg, wb, b, args.prompt + W + 16)
            out["batch_sweep"][str(b)] = {"value": b * 32 / (ms_b * 1e-3), "unit": "tokens/s", "ms_per_step": ms_b / 32, "steps": 32,
                                          "kernels_per_step": kps, "step_roofline_frac": sb / (ms_b / 32 * 1e-3) / 1e9 / peak}

    # ---- roofline of the dominant kernel (W4A16 GEMM), live: the step's own kernel variants (fused RMSNorm prologue,
    # qkv-RoPE / SwiGLU / residual epilogues, PDL policy) on every layer's own weights.  Runs last: it rewrites the
    # residual stream and the KV rows of the current positions. ----
    dec.set_state(tok_all[:B], pos_all[:B])
    iters = 5
    g_ms, g_launches, g_bytes = dec.bench_gemms(B, iters)
    achieved = g_bytes * iters / (g_ms * 1e-3) / 1e9
    out["roofline"] = {
        "bound": "hbm",
        "kernel": ("k_w8a8_skinny (+ activation quant)" if args.quant != "default" else "k_dense_skinny") if dense
        else ("k_w4a16_v3 (integer IMMA, fused norm / RoPE / SwiGLU / residual variants as in the step)" if B <= 7
              else "k_w4a16_ts (tcgen05, A operand in TMEM, tensor-TMA)"),
        "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "peak_kind": peak_kind,
        "bytes_per_launch": g_bytes / g_launches, "us_per_launch": g_ms * 1e3 / iters / g_launches,
        "traffic": None,
        "traffic_note": "dram bytes are not observable from inside the run; ncu --set full captures: profiles/r01_w4a16_traffic.json (integer kernel: dram reads = algorithmic bytes within 0.1 %), profiles/r02_w4a16_ts_ncu_full.txt (tcgen05 kernel: 61.4 MB read for 61.0 MB algorithmic)",
    }

    if extras:
        dec.close()
        dec = None
        c1 = model_cfg("llama-3.2-1b")
        d1 = LlamaDecoder(quant_type=0, dtype="bf16", max_batch=1, max_seq=args.prompt + 2 * W + 80, **c1)
        d1.init_synthetic(seed=1)
        s1 = torch.cuda.ExternalStream(d1.stream())
        ingest_prompt(d1, 1, args.prompt, c1["vocab_size"], rng)
        ms1, _ = measure_decode(d1, 1, 64, W, s1, barrier)
        wb1, kps1 = d1.stats(1)
        out["llama_3_2_1b_bf16"] = {"value": 64 / (ms1 * 1e-3), "unit": "tokens/s", "ms_per_step": ms1 / 64, "steps": 64,
                                    "kernels_per_step": kps1,
                                    "step_roofline_frac": step_bytes_of(c1, wb1, 1, args.prompt + 40) / (ms1 / 64 * 1e-3) / 1e9 / peak}
        d1.close()
        # the reference's own decode kernels (recompiled for sm_100, oracle/_ref) chained for one 8B layer + lm_head on
        # this GPU, in a separate process: a reported side-by-side, not an arm
        ref_tool = os.path.join(ROOT, "tools", "ref_layer_bench.py")
        if os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libzl_ref.so")):
            try:
                r = subprocess.run([sys.executable, ref_tool, "--chain-only"], capture_output=True, text=True, timeout=240)
                lines = [json.loads(l) for l in r.stdout.splitlines() if l.startswith("{")]
                if lines:
                    out["reference_gpu_kernels"] = lines[0]
                    out["reference_gpu_kernels"]["ours_step_us"] = ms_dev / args.steps * 1e3
            except Exception as e:      # the side-by-side is optional
                out["reference_gpu_kernels"] = {"unavailable": str(e)[:200]}

    if rank == 0 and not args.no_cpu_baseline:
        ref = CpuReference(cfg, not dense, B)
        v, t_step, n_steps, sample = ref.run(2, budget_s=40.0)
        out["cpu_baseline"] = {"value": v, "unit": "tokens/s", "cores": ref.threads, "kind": "port", "sample": sample}
    if rank == 0:
        print(json.dumps(out))
    if dec is not None:
        dec.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
