"""Compare the CPU oracle with the golden outputs of the reference's own kernels (TEST INFRASTRUCTURE).

tests/golden/ref_<case>.npz were produced by oracle/gen_ref_golden.py on a B200 from the reference kernels
recompiled for sm_100.  Integer stages must match bit for bit; float stages within the stated tolerance
(the reference's fp16 8-wide partial sums are emulated where that matters)."""
import os

import numpy as np

from . import golden_cases as gc
from . import gptq, ops

ULP16 = 2.0 ** -10


def _rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def _close_ulp(a, b, ulps=1.0, atol=1e-6):
    np.testing.assert_allclose(np.asarray(a, np.float32), np.asarray(b, np.float32), rtol=ulps * ULP16, atol=atol)


def check_layout(g, awq):
    c = gc.case_awq_layout() if awq else gc.case_gptq_layout()
    qw, qz, sc, _ = gptq.to_k_major(c["qweight"], c["qzeros"], c["scales"], None, 128, is_awq=awq)
    np.testing.assert_array_equal(g["qw_km"].view(np.uint32), qw)
    np.testing.assert_array_equal(g["qz_km"], qz)
    np.testing.assert_array_equal(g["sc_km"], sc)
    np.testing.assert_array_equal(g["w16"], gptq.dequant_k_major_f16(qw, qz, sc))


def check_gemv(g, sym):
    c = gc.case_gemv(sym)
    w = gptq.dequant_k_major_f32(c["qw_km"], c["qz_km"], c["sc_km"], sym)
    for m, x in c["xs"].items():
        ref = g["y%d" % m].astype(np.float32)
        refb = g["yb%d" % m].astype(np.float32)
        exact = gptq.gemm_f32(x, w)
        # the reference accumulates 8 products in fp16: ~1e-3 away from exact fp32
        assert _rel(ref, exact) < 4e-3, (m, _rel(ref, exact))
        assert _rel(refb, gptq.gemm_f32(x, w, c["bias"])) < 4e-3
        if m <= 3:   # the emulation follows the kernel's exact operation order (python loops: small m only)
            emu = gptq.gemv_ref_numerics(x, c["qw_km"], c["qz_km"], c["sc_km"], sym).astype(np.float32)
            _close_ulp(emu, ref, ulps=2.0, atol=2e-3)
            assert _rel(emu, ref) < 3e-4, (m, _rel(emu, ref))


def check_gate_in(g):
    c = gc.case_gate_in()
    wg = gptq.dequant_k_major_f32(*c["gate"])
    wu = gptq.dequant_k_major_f32(*c["up"])
    for m, x in c["xs"].items():
        exact = ops.silu(gptq.gemm_f32(x, wg)) * gptq.gemm_f32(x, wu)
        assert _rel(g["y%d" % m], exact) < 6e-3
        unf = ops.silu_mul(gptq.gemm_f32(x, wg), gptq.gemm_f32(x, wu), "f16")
        assert _rel(g["unfused%d" % m], unf) < 6e-3


def check_norm(g):
    c = gc.case_norm()
    a, b, w = c["a"], c["b"], c["w"]
    _close_ulp(g["y"], ops.rmsnorm(a, w, c["eps"]))
    s, y_fuse = ops.add_rmsnorm_fused(a, b, w, c["eps"])
    np.testing.assert_array_equal(g["s"].astype(np.float32), s)
    _close_ulp(g["y_fuse"], y_fuse)
    np.testing.assert_array_equal(g["add"].astype(np.float32), ops.residual_add(a, b))
    _close_ulp(g["y_after_add"], ops.add_then_rmsnorm(a, b, w, c["eps"])[1])
    _close_ulp(g["gate_mul"], ops.silu_mul(a, b))


def check_rope(g):
    c = gc.case_rope()
    q, k, v = ops.split_qkv_rope(c["qkv"], c["cos"], c["sin"], c["hq"], c["hkv"], c["d"])
    _close_ulp(g["q"], q, ulps=1.0, atol=2e-3)
    _close_ulp(g["k"], k, ulps=1.0, atol=2e-3)
    np.testing.assert_array_equal(g["v"].astype(np.float32), v)


def check_attention(g, long):
    c = gc.case_attention(long)
    ref = ops.decode_attention(c["q"], c["ks"], c["vs"], c["lens"], c["masks"], c["scale"], c["hq"] // c["hkv"])
    assert _rel(g["out"], ref) < 1e-3, _rel(g["out"], ref)
    np.testing.assert_allclose(g["out"].astype(np.float32), ref, atol=3e-3, rtol=3e-3)


def check_int8(g):
    c = gc.case_int8()
    q, s = ops.int8_quant_per_token(c["x"])
    assert np.abs(g["q"].astype(np.int32) - q.astype(np.int32)).max() <= 1
    assert (g["q"] != q).mean() < 1e-3
    np.testing.assert_allclose(g["s"], s, rtol=1e-6)
    ar = ops.allreduce_int8_reference(c["parts"])
    step = np.abs(ar).max() / 127.0
    np.testing.assert_allclose(g["allreduce"].astype(np.float32), ar, atol=1.01 * step)
    assert (np.abs(g["allreduce"].astype(np.float32) - ar) > 1e-6).mean() < 5e-3


def check_w8(g):
    c = gc.case_w8()
    for tag in ("f16", "bf16"):
        x = ops._t(c["x"], tag)
        q, sx = ops.int8_quant_per_token(x)
        np.testing.assert_array_equal(g["q_" + tag], q)                       # integer work: bit-exact
        np.testing.assert_array_equal(g["sx_" + tag], sx)
        acc = q.astype(np.int32) @ c["w_q"].astype(np.int32).T
        np.testing.assert_array_equal(g["acc_" + tag], acc)
        ws = ops._t(c["w_s"], tag)
        np.testing.assert_array_equal(g["back_" + tag], ops.int8_scale_back(acc, sx, ws, tag))
        np.testing.assert_array_equal(g["back_f32scale_" + tag], ops.int8_scale_back(acc, sx, ws, tag))
        y, lq, ls = ops.rmsnorm_quant(x, ops._t(c["ln_w"], tag), c["eps"], 1.0, tag)
        np.testing.assert_array_equal(g["ln_q_" + tag], lq)
        np.testing.assert_allclose(g["ln_s_" + tag], ls, rtol=2e-6)            # device rsqrtf vs exact 1/sqrt
        assert _rel(g["ln_y_" + tag], y) < (1e-3 if tag == "f16" else 4e-3)
        fq, fs = ops.fp8_quant_per_tensor(x, dtype=tag)
        np.testing.assert_array_equal(g["f8_s_" + tag], np.array([fs], np.float32))
        np.testing.assert_array_equal(ops.e4m3_decode(g["f8_q_" + tag]), fq)   # same e4m3 codes (as values)
        wv = ops.e4m3_decode(c["w_f8"])
        for key, bias in (("f8_y_", None), ("f8_y_bias_", ops._t(c["bias"], tag))):
            yo = ops.fp8_linear(x, wv, c["w_f8_scale"], tag, bias)
            assert _rel(g[key + tag], yo) < (1e-3 if tag == "f16" else 4e-3), (key, tag, _rel(g[key + tag], yo))


def check_rope_tables(g):
    c = gc.case_rope_tables()
    pos = c["pos"].astype(np.float64)
    for name, (d, theta, l3) in c["variants"].items():
        cos, sin = ops.rope_cos_sin(c["pos"], d, theta, l3)
        # fp32 angles: one ulp of inv_freq (numpy power vs the device's powf) moves the angle by pos * 6e-8 rad
        atol = (2e-6 + pos * 2.5e-7)[:, None]
        assert (np.abs(g["cos_" + name] - cos) <= atol).all(), name
        assert (np.abs(g["sin_" + name] - sin) <= atol).all(), name
        # position 0 and 1 pin the inverse frequencies themselves (incl. the llama3 wavelength branches)
        np.testing.assert_allclose(g["sin_" + name][1], sin[1], rtol=3e-6, atol=1e-9)


def check_marlin(g):
    c = gc.case_marlin()
    qw, qz, sc, _ = gptq.to_k_major(c["qweight"], c["qzeros"], c["scales"], c["g_idx"], 128)
    w = gptq.dequant_k_major_f32(qw, qz, sc, True)                  # zero fixed at 8 (u4b8)
    for m, x in c["xs"].items():
        assert _rel(g["y%d" % m], gptq.gemm_f32(x, w)) < 1e-3, m
    # gptq_marlin_repack only permutes nibbles
    nib = lambda a: np.sort(np.stack([(a.view(np.uint32) >> np.uint32(4 * i)) & np.uint32(15) for i in range(8)]).reshape(-1))
    np.testing.assert_array_equal(nib(g["repacked"]), nib(np.ascontiguousarray(c["qweight"])))


def check_kv8(g):
    c = gc.case_kv8()
    kd, vd = [], []
    for i, (k, v) in enumerate(zip(c["ks"], c["vs"])):
        kq, sk = ops.int8_quant_per_token(k.reshape(-1, c["d"]))        # same absmax / 127 rounding, codes offset by 128
        vq, sv = ops.int8_quant_per_token(v.reshape(-1, c["d"]))
        u8 = lambda q, shape: (q.astype(np.int32) + 128).astype(np.uint8).reshape(shape)
        assert gc.digest(u8(kq, k.shape)) == str(g["kq%d_digest" % i]), i
        assert gc.digest(u8(vq, v.shape)) == str(g["vq%d_digest" % i]), i
        np.testing.assert_array_equal(g["sk%d" % i].reshape(-1), sk)
        np.testing.assert_array_equal(g["sv%d" % i].reshape(-1), sv)
        kd.append((kq.astype(np.float32) * sk[:, None]).reshape(k.shape))
        vd.append((vq.astype(np.float32) * sv[:, None]).reshape(v.shape))
    ref = ops.decode_attention(c["q"], kd, vd, c["lens"], c["masks"], c["scale"], c["hq"] // c["hkv"], "f32")
    assert _rel(g["out"], ref) < 3e-3, _rel(g["out"], ref)          # the reference multiplies q.k in fp16


CHECKS = {
    "ref_gptq_layout": lambda g: check_layout(g, False),
    "ref_awq_layout": lambda g: check_layout(g, True),
    "ref_gemv_asym": lambda g: check_gemv(g, False),
    "ref_gemv_sym": lambda g: check_gemv(g, True),
    "ref_gate_in": check_gate_in,
    "ref_norm": check_norm,
    "ref_rope": check_rope,
    "ref_attention_short": lambda g: check_attention(g, False),
    "ref_attention_long": lambda g: check_attention(g, True),
    "ref_int8": check_int8,
    "ref_w8": check_w8,
    "ref_rope_tables": check_rope_tables,
    "ref_marlin": check_marlin,
    "ref_kv8": check_kv8,
}


def check_file(path):
    name = os.path.splitext(os.path.basename(path))[0]
    if name not in CHECKS:
        raise KeyError("no checker for golden file " + name)
    with np.load(path) as g:
        CHECKS[name](g)
