#!/usr/bin/env python
"""Run the REFERENCE's own kernels (oracle/_ref/libzl_ref.so) on the inputs of tests/test_vs_reference_gpu.py and store
what each of its tests compares with (TEST INFRASTRUCTURE; needs a GPU and the built shim library):

    python -m oracle.gen_vs_reference_golden OUT.npz       # then copy OUT.npz to tests/golden/vs_reference.npz

Keys are "<case>/<output>".  An output the tests compare bit for bit is stored as golden_cases.digest of its bytes; a
float output as its values in the output's own precision (bf16 as fp32), all of them when small, otherwise the fixed
seeded sample tests.helpers.sample_index picks, so that the file stays far below 1 MB.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle.gen_ref_golden import Ref  # noqa: E402
from tests import test_vs_reference_gpu as T  # noqa: E402
from tests.helpers import sample_index, tensor_digest  # noqa: E402

SAMPLE = 2048       # stored values of one large float output


class Recorder:
    def __init__(self):
        self.data = {}

    def exact(self, case, key, t):
        self.data[case + "/" + key] = np.array(tensor_digest(t))

    def values(self, case, key, t, n=SAMPLE):
        a = (t.float() if t.dtype == torch.bfloat16 else t).cpu().numpy().reshape(-1)
        self.data[case + "/" + key] = a[sample_index(a.size, n)]


def main(out_path):
    from zhilight_b200 import build, ops
    build.build()
    ref = Ref()
    dev = ref.dev
    rec = Recorder()
    ex, val = rec.exact, rec.values

    def layout(case, qw, qz, sc, awq=False, prefix=""):
        r = ref.gptq_to_k_major(qw, qz, sc, awq=awq)
        for key, t in zip(("qw_km", "qz_km", "sc_km"), r):
            ex(case, prefix + key, t)
        return r

    for sym in (False, True):
        qw, qz, sc, _ = T.ckpt_4096(sym)
        r = layout("layout_sym%d" % sym, qw, qz, sc)
        if not sym:
            ex("layout_sym0", "w16", ref.dequant_k_major(*r))
        for m in (1, 4, 16, 33):
            val("gemv_sym%d_m%d" % (sym, m), "y", ref.gemv(T.gemv_x(m, dev), *r, None, sym))

    qw, qz, sc = T.awq_checkpoint()
    layout("awq_layout", qw, qz, sc, awq=True)

    a, b, x = T.swiglu_inputs(dev)
    ga = layout("swiglu", *a[:3], prefix="gate_")
    ub = layout("swiglu", *b[:3], prefix="up_")
    val("swiglu", "y", ref.gate_in(x, ga, ub))

    for dtype in (torch.float16, torch.bfloat16):
        case = "norm_rope_%s" % str(dtype).split(".")[-1]
        a, b, w, qkv, pos, (hq, hkv, dh) = T.norm_rope_inputs(dtype, dev)
        val(case, "rmsnorm", ref.rmsnorm(a, w, 1e-5))
        s, y = ref.rmsnorm_fuse_add(a, b, w, 1e-5)
        ex(case, "fuse_add_s", s)
        val(case, "fuse_add_y", y)
        ex(case, "element_add", ref.element_add(a, b))
        cos, sin = ops.rope_cos_sin(pos, dh, 500000.0, dict(factor=8.0, low=1.0, high=4.0, orig=8192.0))
        ex(case, "rope_cos", cos)
        ex(case, "rope_sin", sin)
        q, k, v = ref.rope_qk_cache(cos, sin, qkv, hq, hkv, dh)
        val(case, "rope_q", q)
        val(case, "rope_k", k)
        ex(case, "rope_v", v)

    for lens in ([4096, 123], [300, 1024, 77], [2048, 2048]):
        q, ks, vs, mask, lens_t, hkv = T.attention_inputs(lens, dev)
        out = ref.attention(q, lens_t, ks, vs, mask, q.shape[-1] ** -0.5, hkv)
        val("attention_" + "_".join(map(str, lens)), "out", out, n=out.numel())

    for dt in (torch.float16, torch.bfloat16):
        tag = str(dt).split(".")[-1]
        x, w_q, w_s = T.int8_linear_inputs(dt, dev)
        r_q, r_s = ref.quant_calc_scale_dt(x)
        acc = (r_q.cpu().int() @ w_q.cpu().int().T).to(dev)
        ex("int8_linear_" + tag, "q", r_q)
        ex("int8_linear_" + tag, "s", r_s)
        ex("int8_linear_" + tag, "y", ref.quant_scale_back(acc, r_s, w_s, dt))

        x, w = T.rmsnorm_quant_inputs(dt, dev)
        ry, rq, rs = ref.layernorm_quant(x, w, 1e-5)
        ex("rmsnorm_quant_" + tag, "q", rq)
        val("rmsnorm_quant_" + tag, "s", rs, n=rs.numel())
        val("rmsnorm_quant_" + tag, "y", ry)

        x, w8, sw = T.fp8_inputs(dt, dev)
        rq, rs = ref.fp8_quant(x)
        ex("fp8_linear_" + tag, "s", rs)
        ex("fp8_linear_" + tag, "q", rq)
        val("fp8_linear_" + tag, "y", ref.fp8_gemm(rq, rs, w8, sw, None, dt))

    pos = torch.tensor(T.ROPE_POS, dtype=torch.int32, device=dev)
    for (theta, l3), name in zip(T.ROPE_VARIANTS, T.ROPE_IDS):
        for d in (64, 128):
            c, s = ref.rope_cos_sin(pos, d, theta, l3)
            val("rope_tables_%s_d%d" % (name, d), "cos", c, n=c.numel())
            val("rope_tables_%s_d%d" % (name, d), "sin", s, n=s.numel())

    for k, n in ((4096, 4096), (4096, 14336)):
        qw, qz, sc = T.sym_checkpoint(k, n, 5)
        for m in (1, 16, 32, 64):
            val("marlin_k%d_n%d_m%d" % (k, n, m), "y", ref.marlin_gemm(T.marlin_x(m, k, dev), ref.t(qw), ref.t(sc)))
    qw, _, _ = T.sym_checkpoint(256, 128, 9)
    rec.data["marlin_repack/repacked"] = ref.marlin_repack(ref.t(qw)).cpu().numpy()

    for m in (1, 8, 32):
        qw, qz, sc, x = T.awq_native_inputs(m, dev)
        val("awq_native_m%d" % m, "y", ref.awq_gemm(x, ref.t(qw), ref.t(sc), ref.t(qz)))

    k, v = T.kv_append_inputs(dev)
    t, hkv, d = k.shape
    kq, ks = ref.quant_u8(k.view(t * hkv, d))
    vq, vs = ref.quant_u8(v.view(t * hkv, d))
    ex("kv_append", "kq", kq.view(t, hkv, d))
    ex("kv_append", "vq", vq.view(t, hkv, d))
    ex("kv_append", "ks", ks.view(t, hkv))
    ex("kv_append", "vs", vs.view(t, hkv))

    for lens in ([1600, 600], [2000], [1100, 1300, 40]):
        case = "kv8_attention_" + "_".join(map(str, lens))
        q, ks, vs, mask, lens_t = T.kv8_shared_scale_inputs(lens, dev)
        hkv, d = ks[0].shape[1], ks[0].shape[2]
        kq, vq, sk, sv = [], [], [], []
        for i, (k, v) in enumerate(zip(ks, vs)):
            a, s = ref.quant_u8(k.view(-1, d))
            b, s2 = ref.quant_u8(v.view(-1, d))
            kq.append(a.view(k.shape))
            sk.append(s.view(k.shape[0], hkv))
            vq.append(b.view(v.shape))
            sv.append(s2.view(v.shape[0], hkv))
            for key, x in (("kq%d" % i, kq[-1]), ("vq%d" % i, vq[-1]), ("sk%d" % i, sk[-1]), ("sv%d" % i, sv[-1])):
                ex(case, key, x)
        out = ref.attention_kv8(q, lens_t, kq, vq, sk, sv, mask, 1.0 / np.sqrt(d), hkv)
        val(case, "out", out, n=out.numel())

    np.savez_compressed(out_path, **rec.data)
    print("wrote %d outputs to %s (%d bytes)" % (len(rec.data), out_path, os.path.getsize(out_path)))


if __name__ == "__main__":
    main(sys.argv[1])
    sys.stdout.flush()
    os._exit(0)      # bmengine statics are torn down after the CUDA driver at interpreter exit
