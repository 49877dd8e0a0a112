"""Seeded inputs of the golden cases (TEST INFRASTRUCTURE).

`oracle/gen_ref_golden.py` feeds them to the REFERENCE's own kernels (oracle/_ref/libzl_ref.so, on the B200 box)
and stores the outputs in tests/golden/ref_<case>.npz; `oracle/check_golden.py` regenerates the same inputs on
the CPU, runs the oracle and compares -- that is what pins the oracle to the reference.
"""
import hashlib

import numpy as np

from . import gptq, ops


def digest(a):
    """sha256 over shape, dtype and bytes: the stored stand-in of a large output that must match bit for bit."""
    a = np.ascontiguousarray(a)
    h = hashlib.sha256(("%s %s " % (a.shape, a.dtype.str)).encode())
    h.update(a.tobytes())
    return h.hexdigest()


def _rng(seed):
    return np.random.default_rng(seed)


def case_gptq_layout():
    k, n, g = 256, 64, 128
    qw, qz, sc, gi = gptq.make_gptq_checkpoint(k, n, g, False, seed=101)
    return dict(qweight=qw, qzeros=qz, scales=sc, K=k, N=n, G=k // g)


def case_awq_layout():
    k, n, g = 256, 64, 128
    r = _rng(102)
    qw = r.integers(0, 2 ** 32, size=(k, n // 8), dtype=np.uint64).astype(np.uint32).view(np.int32)
    qz = r.integers(0, 2 ** 32, size=(k // g, n // 8), dtype=np.uint64).astype(np.uint32).view(np.int32)
    sc = (0.005 + 0.015 * r.random((k // g, n))).astype(np.float16)
    return dict(qweight=qw, qzeros=qz, scales=sc, K=k, N=n, G=k // g)


def case_gemv(sym):
    k, n, g = 1024, 256, 128
    qw, qz, sc, gi = gptq.make_gptq_checkpoint(k, n, g, sym, seed=103 + int(sym))
    qw_km, qz_km, sc_km, _ = gptq.to_k_major(qw, qz, sc, gi, g)
    r = _rng(105)
    xs = {m: r.standard_normal((m, k)).astype(np.float16) for m in (1, 3, 16, 33)}
    bias = r.standard_normal(n).astype(np.float16)
    return dict(qw_km=qw_km.view(np.int32), qz_km=qz_km, sc_km=sc_km, xs=xs, bias=bias, K=k, N=n, G=k // g, sym=sym)


def case_gate_in():
    k, f, g = 512, 128, 128
    a = gptq.make_gptq_checkpoint(k, f, g, False, seed=106)
    b = gptq.make_gptq_checkpoint(k, f, g, False, seed=107)
    ka = gptq.to_k_major(a[0], a[1], a[2], a[3], g)
    kb = gptq.to_k_major(b[0], b[1], b[2], b[3], g)
    r = _rng(108)
    xs = {m: r.standard_normal((m, k)).astype(np.float16) for m in (1, 2)}
    return dict(gate=ka[:3], up=kb[:3], xs=xs, K=k, F=f, G=k // g)


def case_norm():
    r = _rng(109)
    t, d = 5, 1024
    return dict(a=r.standard_normal((t, d)).astype(np.float16), b=r.standard_normal((t, d)).astype(np.float16),
                w=(1 + 0.1 * r.standard_normal(d)).astype(np.float16), eps=1e-5, T=t, D=d)


def case_rope():
    r = _rng(110)
    t, hq, hkv, d = 6, 8, 2, 128
    pos = np.array([0, 1, 5, 100, 1000, 4000], dtype=np.int32)
    cos, sin = ops.rope_cos_sin(pos, d, 500000.0, dict(factor=8.0, low=1.0, high=4.0, orig=8192.0))
    return dict(qkv=r.standard_normal((t, (hq + 2 * hkv) * d)).astype(np.float16), cos=cos, sin=sin, T=t, hq=hq,
                hkv=hkv, d=d)


def case_attention(long):
    r = _rng(111 + int(long))
    hq, hkv, d = 8, 2, 128
    lens = [1600, 600] if long else [96, 33, 128]
    b = len(lens)
    q = r.standard_normal((b, 1, hq, d)).astype(np.float16)
    ks = [r.standard_normal((lb, hkv, d)).astype(np.float16) for lb in lens]
    vs = [r.standard_normal((lb, hkv, d)).astype(np.float16) for lb in lens]
    masks = []
    for lb in lens:
        m = np.ones((1, lb), np.int8)
        m[0, lb - 2:] = 0
        m[0, r.permutation(lb - 2)[: lb // 9]] = 0
        masks.append(m)
    return dict(q=q, ks=ks, vs=vs, masks=masks, lens=np.array(lens, np.int32), hq=hq, hkv=hkv, d=d,
                scale=float(1.0 / np.sqrt(d)))


def case_int8():
    r = _rng(113)
    m, k, ws = 4, 512, 4
    x = r.standard_normal((m, k)).astype(np.float16)
    parts = [r.standard_normal((8, 256)).astype(np.float16) for _ in range(ws)]
    return dict(x=x, parts=parts, WS=ws)


def case_w8():
    """W8A8 Linear pieces: per-token int8 quant + scale-back, layernorm_quant, per-tensor fp8 quant + fp8 GEMM."""
    r = _rng(127)
    m, k, n = 5, 512, 96
    x = (r.standard_normal((m, k)) * 1.7).astype(np.float16)
    x[3] = 0                                                   # all-zero token: absmax 0
    ln_w = (1.0 + 0.2 * r.standard_normal(k)).astype(np.float16)
    w_q = r.integers(-127, 128, size=(n, k)).astype(np.int8)
    w_s = (0.001 + 0.004 * r.random(n)).astype(np.float16)
    bias = (0.1 * r.standard_normal(n)).astype(np.float16)
    w_f8 = r.integers(0, 256, size=(n, k)).astype(np.uint8)
    w_f8[(w_f8 & 0x7F) == 0x7F] = 0x38                         # no NaN encodings (0x7f / 0xff)
    return dict(x=x, ln_w=ln_w, eps=1e-5, w_q=w_q, w_s=w_s, bias=bias, w_f8=w_f8, w_f8_scale=np.float32(0.0123))


ROPE_TABLE_VARIANTS = {
    "plain_d64": (64, 10000.0, None),
    "plain_d128": (128, 10000.0, None),
    "l3f8_d128": (128, 500000.0, dict(factor=8.0, low=1.0, high=4.0, orig=8192.0)),
    "l3f32_d64": (64, 500000.0, dict(factor=32.0, low=1.0, high=4.0, orig=8192.0)),
}


def case_rope_tables():
    """RopePreparer inputs (rope_preparer.cu:49-161): plain and llama3 (factor 8: Llama-3.1, factor 32: Llama-3.2)."""
    return dict(pos=np.array([0, 1, 2, 63, 4095, 8191, 8192, 100000], dtype=np.int32), variants=ROPE_TABLE_VARIANTS)


def case_marlin():
    """QuantType 8: symmetric (u4b8) g128 HF-GPTQ checkpoint as GPTQMarlin loads it (linear.cpp:1402-1435)."""
    k, n, g = 512, 256, 128
    qw, qz, sc, gi = gptq.make_gptq_checkpoint(k, n, g, True, seed=131)
    r = _rng(132)
    xs = {m: r.standard_normal((m, k)).astype(np.float16) for m in (1, 5, 17)}
    return dict(qweight=qw, qzeros=qz, scales=sc, g_idx=gi, xs=xs, K=k, N=n, G=k // g)


def case_kv8():
    """int8 KV cache (KV_CACHE_DTYPE=int8): fp16 K / V rows that all share one absmax (4.0) per (row, head) -- see
    tests/test_vs_reference_gpu.py for why: the reference's split kernel indexes its scales without the split offset."""
    r = _rng(141)
    hq, hkv, d = 8, 2, 128
    lens = [1100, 1300, 40]
    q = r.standard_normal((len(lens), 1, hq, d)).astype(np.float16)
    ks, vs, masks = [], [], []
    for lb in lens:
        k = np.clip(r.standard_normal((lb, hkv, d)), -4, 4).astype(np.float16)
        v = np.clip(r.standard_normal((lb, hkv, d)), -4, 4).astype(np.float16)
        k[:, :, 5] = 4.0
        v[:, :, 5] = 4.0
        ks.append(k)
        vs.append(v)
        m = np.ones((1, lb), np.int8)
        m[0, lb - 2:] = 0
        m[0, r.permutation(lb - 2)[: lb // 9]] = 0
        masks.append(m)
    return dict(q=q, ks=ks, vs=vs, masks=masks, lens=np.array(lens, np.int32), hq=hq, hkv=hkv, d=d,
                scale=float(1.0 / np.sqrt(d)))
