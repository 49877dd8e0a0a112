"""Decode driver front end (zl_llama_* C-ABI).  Host buffers in, host buffers out.

Mirrors the slice of zhilight.LLaMA / DynamicBatchGenerator a decode step touches
(reference zhilight/llama.py:114-244, zhilight/dynamic_batch.py:382-639): config -> load_state_dict ->
step(tokens, positions) -> next tokens.  Scheduling (who is in the batch, at which position) stays with the
caller, exactly as the reference keeps it in src/generator.
"""
import ctypes

import numpy as np

from . import _lib

MODEL_PRESETS = {
    # SURVEY.md section 8: shapes of the BASELINE.json configs
    "llama-3.1-8b": dict(num_layers=32, dim_model=4096, num_heads=32, num_kv_heads=8, dim_head=128, dim_ff=14336,
                         vocab_size=128256, eps=1e-5, rope_theta=500000.0,
                         rope_llama3=dict(factor=8.0, low=1.0, high=4.0, orig=8192.0)),
    "llama-3.2-1b": dict(num_layers=16, dim_model=2048, num_heads=32, num_kv_heads=8, dim_head=64, dim_ff=8192,
                         vocab_size=128256, eps=1e-5, rope_theta=500000.0,
                         rope_llama3=dict(factor=32.0, low=1.0, high=4.0, orig=8192.0)),
    # north_star TP=8 target and BASELINE config 4 (Qwen2-72B GPTQ: FF padded to 29696 in the GPTQ build,
    # zhilight/config/qwen2_adapter.py:27-28; q/k/v bias, attention.cpp:105-109)
    "llama-3.1-70b": dict(num_layers=80, dim_model=8192, num_heads=64, num_kv_heads=8, dim_head=128, dim_ff=28672,
                          vocab_size=128256, eps=1e-5, rope_theta=500000.0,
                          rope_llama3=dict(factor=8.0, low=1.0, high=4.0, orig=8192.0)),
    "qwen2-72b": dict(num_layers=80, dim_model=8192, num_heads=64, num_kv_heads=8, dim_head=128, dim_ff=29696,
                      vocab_size=152064, eps=1e-6, rope_theta=1000000.0, rope_llama3=None, qkv_bias=True),
    "tiny": dict(num_layers=2, dim_model=256, num_heads=4, num_kv_heads=2, dim_head=64, dim_ff=512,
                 vocab_size=512, eps=1e-5, rope_theta=10000.0, rope_llama3=None),
}

QUANT_NONE, QUANT_AUTO_INT8, QUANT_GPTQ, QUANT_AWQ, QUANT_FP8 = 0, 2, 5, 6, 7     # model_config.hpp:132-144


class LlamaDecoder:
    def __init__(self, num_layers, dim_model, num_heads, num_kv_heads, dim_head, dim_ff, vocab_size, eps=1e-5,
                 rope_theta=10000.0, rope_llama3=None, quant_type=QUANT_NONE, group_size=128, sym=False,
                 dtype="f16", max_batch=1, max_seq=512, use_pdl=True, use_graph=True, tp_rank=0, tp_size=1, fuse=2, tp_int8=False,
                 prefill_chunk=0, qkv_bias=False):
        self.lib = _lib.load()
        l3 = rope_llama3 or {}
        self.cfg = _lib.LlamaConfig(
            num_layers, dim_model, num_heads, num_kv_heads, dim_head, dim_ff, vocab_size, eps, rope_theta,
            float(l3.get("factor", 0.0)), float(l3.get("low", 1.0)), float(l3.get("high", 4.0)),
            float(l3.get("orig", 8192.0)), quant_type, group_size, int(sym), {"f16": 0, "bf16": 1}[dtype],
            max_batch, max_seq, tp_rank, tp_size, int(use_pdl), int(use_graph), int(tp_int8), int(fuse), int(prefill_chunk), int(qkv_bias))
        self.vocab_size = vocab_size
        self.vocab_shard = vocab_size // tp_size      # lm_head is vocab-parallel: logits come back per rank shard
        self.max_batch = max_batch
        h = ctypes.c_void_p()
        _lib.check(self.lib.zl_llama_create(ctypes.byref(self.cfg), ctypes.byref(h)))
        self.h = h

    def set_comm(self, comm):
        """comm: zhilight_b200.dist.TPComm (kept alive by this object)."""
        self._comm = comm
        _lib.check(self.lib.zl_llama_set_comm(self.h, comm.handle))

    def close(self):
        if getattr(self, "h", None):
            self.lib.zl_llama_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def load_state_dict(self, state_dict):
        """state_dict: name -> numpy array (2-D or 1-D), HF/ZhiLight checkpoint layout."""
        for name, arr in state_dict.items():
            a = np.ascontiguousarray(arr)
            rows, cols = (1, a.shape[0]) if a.ndim == 1 else a.shape
            _lib.check(self.lib.zl_llama_load_tensor(self.h, name.encode(), a.ctypes.data_as(ctypes.c_void_p),
                                                     rows, cols, a.itemsize))
        _lib.check(self.lib.zl_llama_finalize(self.h))

    def init_synthetic(self, seed=0):
        _lib.check(self.lib.zl_llama_init_synthetic(self.h, seed))

    def decode(self, tokens, positions, want_logits=False):
        """One step: tokens/positions int32 host arrays (B).  Returns next tokens (B) [, logits (B, V/tp) fp32: this
        rank's vocabulary shard]."""
        t = np.ascontiguousarray(tokens, dtype=np.int32)
        p = np.ascontiguousarray(positions, dtype=np.int32)
        b = t.size
        nxt = np.empty(b, dtype=np.int32)
        logits = np.empty((b, self.vocab_shard), dtype=np.float32) if want_logits else None
        _lib.check(self.lib.zl_llama_decode(
            self.h, t.ctypes.data_as(ctypes.c_void_p), p.ctypes.data_as(ctypes.c_void_p), b,
            nxt.ctypes.data_as(ctypes.c_void_p),
            logits.ctypes.data_as(ctypes.c_void_p) if want_logits else None))
        return (nxt, logits) if want_logits else nxt

    def prefill(self, task, tokens, pos0=0, want_logits=False):
        """Chunked prefill of one task's prompt; returns the greedy next token [, logits of the last position]."""
        t = np.ascontiguousarray(tokens, dtype=np.int32)
        nxt = np.empty(1, dtype=np.int32)
        logits = np.empty((1, self.vocab_shard), dtype=np.float32) if want_logits else None
        _lib.check(self.lib.zl_llama_prefill(
            self.h, int(task), t.ctypes.data_as(ctypes.c_void_p), t.size, int(pos0),
            nxt.ctypes.data_as(ctypes.c_void_p), logits.ctypes.data_as(ctypes.c_void_p) if want_logits else None))
        return (int(nxt[0]), logits) if want_logits else int(nxt[0])

    def set_state(self, tokens, positions):
        t = np.ascontiguousarray(tokens, dtype=np.int32)
        p = np.ascontiguousarray(positions, dtype=np.int32)
        _lib.check(self.lib.zl_llama_set_state(self.h, t.ctypes.data_as(ctypes.c_void_p),
                                               p.ctypes.data_as(ctypes.c_void_p), t.size))

    def get_state(self, b):
        t = np.empty(b, dtype=np.int32)
        p = np.empty(b, dtype=np.int32)
        _lib.check(self.lib.zl_llama_get_state(self.h, t.ctypes.data_as(ctypes.c_void_p),
                                               p.ctypes.data_as(ctypes.c_void_p), b))
        return t, p

    def logits(self, b):
        """fp32 logits (B, V/tp) of the most recent step: this rank's vocabulary shard."""
        out = np.empty((b, self.vocab_shard), dtype=np.float32)
        _lib.check(self.lib.zl_llama_get_logits(self.h, out.ctypes.data_as(ctypes.c_void_p), b))
        return out

    def set_sampling(self, task, temperature=1.0, top_p=1.0, top_k=0, repetition_penalty=1.0, presence_penalty=0.0,
                     seed=0):
        """Seeded top-k / top-p sampling with repetition / presence penalties for `task` (SearchTask fields of the
        reference): clears the task's seen set and draw counter.  Picks of steps whose batch holds the task come from
        zl_sample; raises ZLError(-2) with tp_size > 1."""
        p = _lib.SampleParams(float(temperature), float(top_p), float(repetition_penalty), float(presence_penalty),
                              int(top_k), int(seed) & 0xFFFFFFFFFFFFFFFF)
        _lib.check(self.lib.zl_llama_set_sampling(self.h, int(task), ctypes.byref(p)))

    def clear_sampling(self, task):
        """Back to plain greedy picks for `task`."""
        _lib.check(self.lib.zl_llama_clear_sampling(self.h, int(task)))

    def step_device(self, b):
        _lib.check(self.lib.zl_llama_step_device(self.h, b))

    def sync(self):
        _lib.check(self.lib.zl_llama_sync(self.h))

    def stream(self):
        return self.lib.zl_llama_stream(self.h)

    def bench_gemms(self, b=1, iters=5):
        """-> (ms for `iters` passes, GEMM launches per pass, algorithmic bytes per pass)."""
        ms = ctypes.c_float()
        n = ctypes.c_int()
        by = ctypes.c_double()
        _lib.check(self.lib.zl_llama_bench_gemms(self.h, b, iters, ctypes.byref(ms), ctypes.byref(n), ctypes.byref(by)))
        return ms.value, n.value, by.value

    def stats(self, b=1):
        wb = ctypes.c_double()
        kn = ctypes.c_int()
        _lib.check(self.lib.zl_llama_stats(self.h, b, ctypes.byref(wb), ctypes.byref(kn)))
        return wb.value, kn.value
