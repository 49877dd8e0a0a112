"""GPU parity: the whole decode step (driver + every kernel) against the CPU oracle model on small
synthetic checkpoints -- the round trip a user of zhilight.LLaMA / DynamicBatchGenerator sees:
state_dict in (HF-GPTQ layout), (token, position) per task in, logits / greedy tokens out."""
import os

import numpy as np
import pytest

from oracle import model as omodel
from tests.helpers import rel_l2

pytestmark = pytest.mark.gpu

TINY = dict(num_layers=2, dim_model=256, num_heads=4, num_kv_heads=2, dim_head=64, dim_ff=512, vocab_size=512,
            eps=1e-5, rope_theta=10000.0, rope_llama3=None)
TINY128 = dict(num_layers=2, dim_model=512, num_heads=4, num_kv_heads=1, dim_head=128, dim_ff=640, vocab_size=1000,
               eps=1e-5, rope_theta=500000.0, rope_llama3=dict(factor=8.0, low=1.0, high=4.0, orig=8192.0))


def _run(cfg, quant, dtype, sym=False, use_pdl=True, use_graph=True, steps=6, tied=False, seed=0, fuse=2):
    from zhilight_b200.llama import LlamaDecoder
    sd = omodel.make_state_dict(cfg, quant, 128, sym, seed=seed, tied=tied, dtype=dtype)
    dec = LlamaDecoder(quant_type=quant, group_size=128, sym=sym, dtype=dtype, max_batch=3, max_seq=64,
                       use_pdl=use_pdl, use_graph=use_graph, fuse=fuse, **cfg)
    dec.load_state_dict(sd)
    orc = omodel.OracleLlama(cfg, sd, quant, 128, sym, dtype, fuse_norm=fuse >= 1)
    rng = np.random.default_rng(seed)
    # three tasks at different positions (ragged batch, like the dynamic batcher produces)
    pos = np.array([0, 0, 0], dtype=np.int32)
    tok = rng.integers(0, cfg["vocab_size"], size=3).astype(np.int32)
    outs = []
    for s in range(steps):
        b = 3 if s % 3 != 2 else 2                      # batch size changes between steps
        nxt, logits = dec.decode(tok[:b], pos[:b], want_logits=True)
        ref = orc.decode(tok[:b], pos[:b], tasks=list(range(b)))
        outs.append((nxt.copy(), logits.copy(), ref))
        tok[:b] = rng.integers(0, cfg["vocab_size"], size=b)      # teacher forcing with random tokens
        pos[:b] += 1
    dec.close()
    return outs


@pytest.mark.parametrize("cfg", [TINY, TINY128], ids=["d64", "d128-llama3rope"])
@pytest.mark.parametrize("sym", [False, True])
@pytest.mark.parametrize("fuse", [0, 1, 2, 3])
def test_gptq_decode_matches_oracle(lib, cuda, cfg, sym, fuse):
    for nxt, logits, ref in _run(cfg, 5, "f16", sym=sym, fuse=fuse):
        # north_star: logits within 1e-3 rel for fp16 -- measured as relative L2 over the vocabulary
        assert rel_l2(logits, ref) <= 2e-3
        for b in range(len(nxt)):
            order = np.argsort(ref[b])
            if ref[b][order[-1]] - ref[b][order[-2]] > 1e-2:
                assert nxt[b] == order[-1]


def test_awq_decode_matches_oracle(lib, cuda):
    for nxt, logits, ref in _run(TINY, 6, "f16"):
        assert rel_l2(logits, ref) <= 2e-3


@pytest.mark.parametrize("dtype,tol", [("f16", 2e-3), ("bf16", 2e-2)])
def test_dense_decode_matches_oracle(lib, cuda, dtype, tol):
    """BASELINE config 2 path (Llama-3.2-1B bf16: no quant, tied lm_head, d=64 attention)."""
    for nxt, logits, ref in _run(TINY, 0, dtype, tied=True):
        assert rel_l2(logits, ref) <= tol


@pytest.mark.parametrize("fuse", [0, 2])
def test_graph_and_pdl_do_not_change_results(lib, cuda, fuse):
    a = _run(TINY, 5, "f16", use_pdl=False, use_graph=False, fuse=fuse)
    b = _run(TINY, 5, "f16", use_pdl=True, use_graph=False, fuse=fuse)
    c = _run(TINY, 5, "f16", use_pdl=True, use_graph=True, fuse=fuse)
    for (na, la, _), (nb, lb, _), (nc, lc, _) in zip(a, b, c):
        np.testing.assert_array_equal(la, lb)
        np.testing.assert_array_equal(la, lc)
        np.testing.assert_array_equal(na, nc)


def test_device_resident_stepping_matches_host_stepping(lib, cuda):
    """bench.py times the device-resident loop (`value`) and the host-fed loop (`e2e`); both must decode
    the same greedy sequence."""
    from zhilight_b200.llama import LlamaDecoder
    sd = omodel.make_state_dict(TINY, 5, 128, False, seed=3)
    finals = []
    for mode in ("host", "device"):
        dec = LlamaDecoder(quant_type=5, max_batch=2, max_seq=64, **TINY)
        dec.load_state_dict(sd)
        tok = np.array([7, 400], dtype=np.int32)
        pos = np.array([0, 0], dtype=np.int32)
        if mode == "host":
            for _ in range(8):
                tok = dec.decode(tok, pos)
                pos = pos + 1
        else:
            dec.set_state(tok, pos)
            for _ in range(8):
                dec.step_device(2)
            tok, pos = dec.get_state(2)
        finals.append((tok.copy(), pos.copy()))
        dec.close()
    np.testing.assert_array_equal(finals[0][0], finals[1][0])
    np.testing.assert_array_equal(finals[0][1], finals[1][1])


@pytest.mark.parametrize("fuse", [2])
def test_long_context_crosses_attention_buckets(lib, cuda, fuse):
    """Graphs are keyed by (batch, attention-length bucket): decode across the 256 -> 512 boundary."""
    from zhilight_b200.llama import LlamaDecoder
    sd = omodel.make_state_dict(TINY, 5, 128, False, seed=5)
    dec = LlamaDecoder(quant_type=5, max_batch=1, max_seq=600, fuse=fuse, **TINY)
    dec.load_state_dict(sd)
    orc = omodel.OracleLlama(TINY, sd, 5, 128, False, "f16", fuse_norm=True)
    rng = np.random.default_rng(0)
    toks = rng.integers(0, TINY["vocab_size"], size=300).astype(np.int32)
    for p in range(300):
        nxt, logits = dec.decode(toks[p:p + 1], np.array([p], np.int32), want_logits=True)
        if p in (0, 254, 255, 256, 257, 299):
            ref = orc.decode(toks[p:p + 1], [p])
            assert rel_l2(logits, ref) <= 3e-3, p
        else:
            orc.decode(toks[p:p + 1], [p])
    dec.close()


LAYER8B = dict(num_layers=3, dim_model=4096, num_heads=32, num_kv_heads=8, dim_head=128, dim_ff=14336, vocab_size=2048,
               eps=1e-5, rope_theta=500000.0, rope_llama3=dict(factor=8.0, low=1.0, high=4.0, orig=8192.0))


# W4: chunks of more than 16 tokens run the tcgen05 kernel (w rounded to fp16 once, fp32 accumulate in TMEM) behind a
# stand-alone RMSNorm, not the exact-integer M <= 16 kernel with the fused norm
@pytest.mark.parametrize("chunk", [32, 64])
@pytest.mark.parametrize("quant,dtype,tol,cfg", [(5, "f16", 5e-3, TINY128), (5, "f16", 5e-3, TINY), (0, "f16", 3e-3, TINY),
                                                 (0, "bf16", 2e-2, TINY)], ids=["gptq-d128", "gptq-d64", "f16", "bf16"])
def test_chunked_prefill_matches_token_by_token_oracle(lib, cuda, quant, dtype, tol, cfg, chunk):
    """zl_llama_prefill (chunks of `chunk` tokens through the M = chunk GEMMs and causal len_q = chunk attention) must
    leave the same KV state and produce the same next-token logits as feeding the prompt one token at a time."""
    from zhilight_b200.llama import LlamaDecoder
    sd = omodel.make_state_dict(cfg, quant, 128, False, seed=9, dtype=dtype)
    dec = LlamaDecoder(quant_type=quant, dtype=dtype, max_batch=2, max_seq=128, prefill_chunk=chunk, **cfg)
    dec.load_state_dict(sd)
    orc = omodel.OracleLlama(cfg, sd, quant, 128, False, dtype, fuse_norm=True)
    rng = np.random.default_rng(4)
    prompt = rng.integers(0, cfg["vocab_size"], size=70).astype(np.int32)      # chunks of 32, 32, 6 / 64, 6
    other = rng.integers(0, cfg["vocab_size"], size=5).astype(np.int32)
    # task 0 gets a short prompt first so that task 1's prefill runs beside existing state
    n0, l0 = dec.prefill(0, other, want_logits=True)
    n1, l1 = dec.prefill(1, prompt, want_logits=True)
    for p, t in enumerate(other):
        r0 = orc.decode(np.array([t]), [p], tasks=[0])
    for p, t in enumerate(prompt):
        r1 = orc.decode(np.array([t]), [p], tasks=[1])
    assert rel_l2(l0, r0) <= tol and rel_l2(l1, r1) <= tol
    # continue decoding both tasks from the prefilled KV state
    tok = np.array([int(np.argmax(r0[0])), int(np.argmax(r1[0]))], dtype=np.int32)
    pos = np.array([len(other), len(prompt)], dtype=np.int32)
    for _ in range(3):
        nxt, logits = dec.decode(tok, pos, want_logits=True)
        ref = orc.decode(tok, pos, tasks=[0, 1])
        assert rel_l2(logits, ref) <= tol
        tok = np.argmax(ref, axis=1).astype(np.int32)
        pos += 1
    dec.close()


def test_prefill_needs_configuration(lib, cuda):
    from zhilight_b200 import _lib
    from zhilight_b200.llama import LlamaDecoder
    dec = LlamaDecoder(quant_type=0, max_batch=1, max_seq=64, **TINY)
    dec.init_synthetic(0)
    with pytest.raises(_lib.ZLError):
        dec.prefill(0, np.arange(4, dtype=np.int32))
    dec.close()


@pytest.mark.parametrize("quant,dtype,tol", [(2, "f16", 6e-3), (2, "bf16", 2e-2), (7, "f16", 6e-3), (7, "bf16", 2e-2)])
def test_w8a8_decode_matches_oracle(lib, cuda, quant, dtype, tol):
    """Whole-model W8A8 decode: AutoInt8 (QuantType 2: per-row int8 weights made at load, per-token int8 activations,
    exact s32 GEMM) and FP8 (QuantType 7: e4m3 weights + per-tensor scale, dynamic per-tensor e4m3 activations).  The
    Linears themselves are bit-exact / 1e-3 (tests/test_w8_gpu.py); over a whole model a fp16 rounding difference
    upstream can flip an activation's quantisation bucket, hence the looser bound on logits."""
    for nxt, logits, ref in _run(TINY, quant, dtype, steps=4):
        assert np.isfinite(logits).all()
        assert rel_l2(logits, ref) <= tol


@pytest.mark.parametrize("cfg", [TINY128, TINY], ids=["d128", "d64-2kvheads"])
def test_dual_stream_prefill_matches_single_stream(lib, cuda, monkeypatch, cfg):
    """SURVEY 8-a16: the two-half / two-stream prefill pipeline (compute stream + reduce stream, events) must produce
    the same KV state and logits as the single-stream chunked prefill; on one GPU the 'reduce' is the residual add."""
    from zhilight_b200.llama import LlamaDecoder
    sd = omodel.make_state_dict(cfg, 5, 128, False, seed=13)
    rng = np.random.default_rng(6)
    prompt = rng.integers(0, cfg["vocab_size"], size=84).astype(np.int32)       # chunks 32, 32, 20 -> halves 16/16, 16/4
    outs = []
    for dual in ("0", "1"):
        monkeypatch.setenv("ZL_PREFILL_DUAL", dual)
        dec = LlamaDecoder(quant_type=5, max_batch=1, max_seq=128, prefill_chunk=32,
                           fuse=int(os.environ.get("ZL_TEST_FUSE", "2")), **cfg)
        dec.load_state_dict(sd)
        nxt, logits = dec.prefill(0, prompt[:int(os.environ.get("ZL_TEST_PROMPT", "84"))], want_logits=True)
        tok, pos = np.array([nxt], np.int32), np.array([int(os.environ.get("ZL_TEST_PROMPT", "84"))], np.int32)
        steps = [logits.copy()]
        for _ in range(3):
            t2, lg = dec.decode(tok, pos, want_logits=True)
            steps.append(lg.copy())
            tok, pos = t2, pos + 1
        dec.close()
        outs.append(steps)
    for a, b in zip(*outs):
        assert np.isfinite(a).all()
        # M = 32 chunks (tcgen05 kernel: weights rounded to fp16, stand-alone RMSNorm) vs two M = 16 halves (exact-integer
        # kernel, fused norm): fp16-level agreement
        assert rel_l2(b, a) <= 5e-3
    orc = omodel.OracleLlama(cfg, sd, 5, 128, False, "f16", fuse_norm=True)
    for p, t in enumerate(prompt[:int(os.environ.get("ZL_TEST_PROMPT", "84"))]):
        ref = orc.decode(np.array([t]), [p])
    assert rel_l2(outs[1][0], ref) <= 5e-3


def test_marlin_quant_type_is_served_by_the_gptq_kernels(lib, cuda):
    """QuantType 8 (GPTQ_Marlin) takes the same symmetric GPTQ checkpoint as QuantType 5 (linear.cpp:1418-1435)."""
    from zhilight_b200.llama import LlamaDecoder
    sd = omodel.make_state_dict(TINY, 5, 128, True, seed=17)
    outs = []
    for qt, sym in ((5, True), (8, False)):
        dec = LlamaDecoder(quant_type=qt, sym=sym, max_batch=2, max_seq=32, **TINY)
        dec.load_state_dict(sd)
        nxt, logits = dec.decode(np.array([3, 9], np.int32), np.array([0, 0], np.int32), want_logits=True)
        outs.append(logits.copy())
        dec.close()
    np.testing.assert_array_equal(outs[0], outs[1])


@pytest.mark.parametrize("cfg", [TINY, TINY128], ids=["d64", "d128"])
def test_qkv_bias_model_matches_oracle(lib, cuda, cfg):
    """Qwen2-style q/k/v biases (attention.cpp:105-109) through the fused qkv GEMM: the bias is gathered into packed-row
    order at load and added before RoPE, like the reference's Linear bias."""
    from zhilight_b200.llama import LlamaDecoder
    sd = omodel.make_state_dict(cfg, 5, 128, False, seed=21)
    rng = np.random.default_rng(5)
    d = cfg["dim_head"]
    for l in range(cfg["num_layers"]):
        for name, n in (("project_q", cfg["num_heads"] * d), ("project_k", cfg["num_kv_heads"] * d),
                        ("project_v", cfg["num_kv_heads"] * d)):
            sd["layers.%d.attn.%s.bias" % (l, name)] = (0.5 * rng.standard_normal(n)).astype(np.float16)
    orc = omodel.OracleLlama(cfg, sd, 5, 128, False, "f16", fuse_norm=True)
    for fuse in (0, 2):
        dec = LlamaDecoder(quant_type=5, max_batch=3, max_seq=64, fuse=fuse, **cfg)
        dec.load_state_dict(sd)
        o = omodel.OracleLlama(cfg, sd, 5, 128, False, "f16", fuse_norm=fuse >= 1)
        tok = np.array([3, 17, 101], dtype=np.int32)
        for step in range(4):
            pos = np.full(3, step, dtype=np.int32)
            nxt, logits = dec.decode(tok, pos, want_logits=True)
            ref = o.decode(tok, pos)
            assert rel_l2(logits, ref) <= 3e-3, (fuse, step)
            tok = np.argmax(ref, axis=1).astype(np.int32)
        dec.close()
    # and the biases matter: without them the logits differ visibly
    sd2 = {k: v for k, v in sd.items() if not k.endswith(".bias")}
    ref_nobias = omodel.OracleLlama(cfg, sd2, 5, 128, False, "f16", fuse_norm=True).decode(np.array([3]), [0])
    assert rel_l2(orc.decode(np.array([3]), [0]), ref_nobias) > 1e-2


LAYERS8B_SMALLV = dict(num_layers=2, dim_model=4096, num_heads=32, num_kv_heads=8, dim_head=128, dim_ff=14336, vocab_size=2048,
                       eps=1e-5, rope_theta=500000.0, rope_llama3=dict(factor=8.0, low=1.0, high=4.0, orig=8192.0))


@pytest.mark.parametrize("b,graph,pdl", [(20, True, True), (32, True, True), (32, False, True), (32, False, False), (17, True, False)])
def test_large_batch_decode_on_8b_shapes_matches_batch_1(lib, cuda, b, graph, pdl):
    """Batch 17..32 decode runs the tcgen05 GEMMs (split-k, qkv-RoPE / SwiGLU / residual epilogues) inside the CUDA graph
    with programmatic dependent launch on Llama-3.1-8B layer shapes: every task of a batch of identical tokens must
    reproduce the batch-1 logits (exact-integer kernel) to fp16 accuracy, with and without graph / PDL."""
    from zhilight_b200.llama import LlamaDecoder
    cfg = LAYERS8B_SMALLV

    def run(bb, feed):
        dec = LlamaDecoder(quant_type=5, group_size=128, sym=True, max_batch=bb, max_seq=64, use_graph=graph, use_pdl=pdl, **cfg)
        dec.init_synthetic(seed=3)
        res, fed = [], []
        tok = 7
        for step in range(4):
            if feed is not None:
                tok = feed[step]
            fed.append(tok)
            nxt, logits = dec.decode(np.full(bb, tok, dtype=np.int32), np.full(bb, step, dtype=np.int32), want_logits=True)
            res.append(logits.copy())
            tok = int(nxt[0])
        dec.close()
        return res, fed

    ref, fed = run(1, None)
    out, _ = run(b, fed)
    for step, (l1, lb) in enumerate(zip(ref, out)):
        assert np.isfinite(l1).all(), step
        assert np.isfinite(lb).all(), step
        for t in (0, b // 2, b - 1):
            assert rel_l2(lb[t], l1[0]) <= 5e-3, (step, t)


def test_prefill_chunk_128_on_8b_shapes_matches_decode_steps(lib, cuda, monkeypatch):
    """The TTFT path on Llama-3.1-8B layer shapes: a 256-token prompt in two 128-token chunks (M = 128 GEMMs, causal
    len_q = 128 attention on k_decode_attn) must leave the same KV state and last-position logits as 256 batch-1 decode
    steps of the same tokens, and three decode steps from either state must agree."""
    from zhilight_b200.llama import LlamaDecoder
    from tests.helpers import attention_plan
    cfg = LAYERS8B_SMALLV
    monkeypatch.delenv("ZL_PREFILL_DUAL", raising=False)       # single-stream chunks: len_q = 128 per attention call
    for keys in (128, 256):
        assert attention_plan(lib, 1, 128, cfg["num_heads"], cfg["num_kv_heads"], keys)[0] == 0
    prompt = np.random.default_rng(12).integers(0, cfg["vocab_size"], size=256).astype(np.int32)
    pre = LlamaDecoder(quant_type=5, group_size=128, sym=True, max_batch=1, max_seq=512, prefill_chunk=128, **cfg)
    pre.init_synthetic(seed=3)
    _, lp = pre.prefill(0, prompt, want_logits=True)
    dec = LlamaDecoder(quant_type=5, group_size=128, sym=True, max_batch=1, max_seq=512, **cfg)
    dec.init_synthetic(seed=3)
    for p, t in enumerate(prompt):
        _, ld = dec.decode(np.array([t], np.int32), np.array([p], np.int32), want_logits=True)
    assert np.isfinite(lp).all() and np.isfinite(ld).all()
    assert rel_l2(lp, ld) <= 5e-3
    tok, pos = np.array([int(np.argmax(ld[0]))], np.int32), np.array([len(prompt)], np.int32)
    for step in range(3):
        _, lp = pre.decode(tok, pos, want_logits=True)
        nd, ld = dec.decode(tok, pos, want_logits=True)
        assert np.isfinite(lp).all()
        assert rel_l2(lp, ld) <= 5e-3, step
        tok, pos = nd, pos + 1
    pre.close()
    dec.close()
