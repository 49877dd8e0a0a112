#!/usr/bin/env python
"""Run the REFERENCE's own kernels (oracle/_ref/libzl_ref.so, built by oracle/Makefile.ref from /root/reference
sources, recompiled for sm_100) on the seeded inputs of oracle/golden_cases.py and store their outputs as
tests/golden/ref_<case>.npz.  TEST INFRASTRUCTURE; needs a GPU (run through gpurun):

    python -m oracle.gen_ref_golden gpurun_out/golden      # then copy *.npz into tests/golden/

The fixtures are small (a few hundred KB) and are committed together with this script.
"""
import ctypes
import os
import sys

import numpy as np
import torch

from . import golden_cases as gc

HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(HERE, "_ref", "libzl_ref.so")


class Ref:
    """ctypes front end of oracle/ref_shim.cu (device pointers in, device pointers out)."""

    def __init__(self, mem_bytes=2 << 30, lib_path=None):
        self.lib = ctypes.CDLL(lib_path or LIB)
        self.lib.zlref_last_error.restype = ctypes.c_char_p
        self.dev = torch.device("cuda:0")
        self._chk(self.lib.zlref_init(0, ctypes.c_size_t(mem_bytes)))

    def _chk(self, rc):
        if rc != 0:
            raise RuntimeError("reference shim: " + self.lib.zlref_last_error().decode())

    def t(self, a):
        return torch.from_numpy(np.ascontiguousarray(a)).to(self.dev)

    @staticmethod
    def p(t):
        return ctypes.c_void_p(t.data_ptr()) if t is not None else None

    # ---- rope tables, Marlin, native AWQ (round 2) ----
    def rope_cos_sin(self, pos, d, theta, llama3=None):
        t = pos.numel()
        cos = torch.empty((t, d), dtype=torch.float32, device=self.dev)
        sin = torch.empty_like(cos)
        l3 = llama3 or {}
        self._chk(self.lib.zlref_rope_cos_sin(self.p(pos), t, d, ctypes.c_float(theta), int(llama3 is not None),
                                              ctypes.c_float(l3.get("factor", 1.0)), ctypes.c_float(l3.get("low", 1.0)),
                                              ctypes.c_float(l3.get("high", 4.0)), int(l3.get("orig", 8192)),
                                              self.p(cos), self.p(sin)))
        return cos, sin

    def marlin_repack(self, qweight_hf):
        k8, n = qweight_hf.shape
        out = torch.empty((k8 * 8 // 16, 2 * n), dtype=torch.int32, device=self.dev)
        self._chk(self.lib.zlref_marlin_repack(self.p(qweight_hf), n, k8 * 8, self.p(out)))
        return out

    def marlin_gemm(self, x, qweight_hf, scales_hf):
        """x (M, K) f16; HF GPTQ qweight (K/8, N) int32 (symmetric, u4b8), scales (K/g, N) f16 -> (M, N) f16."""
        m, k = x.shape
        n = qweight_hf.shape[1]
        out = torch.empty((m, n), dtype=torch.float16, device=self.dev)
        self._chk(self.lib.zlref_marlin_gemm(self.p(x), self.p(qweight_hf), self.p(scales_hf), m, n, k, scales_hf.shape[0],
                                             self.p(out)))
        return out

    def awq_gemm(self, x, qweight, scales, qzeros):
        """native awq_gemm (split-k 32): qweight (K, N/8) int32, scales (K/g, N) f16, qzeros (K/g, N/8) int32."""
        m, k = x.shape
        n = scales.shape[1]
        out = torch.empty((m, n), dtype=torch.float16, device=self.dev)
        self._chk(self.lib.zlref_awq_gemm(self.p(x), self.p(qweight), self.p(scales), self.p(qzeros), m, n, k, scales.shape[0],
                                          self.p(out)))
        return out

    # ---- int8 KV cache ----
    def quant_u8(self, x):
        """int8_op::quant_calc_scale(x, 127, 128): (M, K) -> uint8 codes, fp32 scales"""
        m, k = x.shape
        q = torch.empty((m, k), dtype=torch.uint8, device=self.dev)
        s = torch.empty(m, dtype=torch.float32, device=self.dev)
        self._chk(self.lib.zlref_quant_calc_scale_u8(self.p(x), m, k, 0 if x.dtype == torch.float16 else 1, self.p(q), self.p(s)))
        return q, s

    def attention_kv8(self, q, lens, ks, vs, sks, svs, mask, scale, hkv, out_dtype=torch.float16):
        b, len_q, hq, d = q.shape
        tab = lambda ts: torch.tensor([t.data_ptr() for t in ts], dtype=torch.int64, device=self.dev)
        ka, va, ska, sva = tab(ks), tab(vs), tab(sks), tab(svs)
        out = torch.empty(q.shape, dtype=out_dtype, device=self.dev)
        self._chk(self.lib.zlref_mqa_rag_buffer_quant(self.p(q), self.p(lens), self.p(ka), self.p(va), self.p(ska), self.p(sva),
                                                      self.p(mask), ctypes.c_size_t(mask.numel()), ctypes.c_float(scale),
                                                      int(lens.max().item()), b, len_q, hq, hkv, d,
                                                      0 if out_dtype == torch.float16 else 1, self.p(out)))
        return out

    # ---- layout ----
    def gptq_to_k_major(self, qweight, qzeros, scales, awq=False):
        lib, p = self.lib, self.p
        if awq:
            k, n8 = qweight.shape
            n = n8 * 8
            qin = self.t(qweight)
            qw = torch.empty((k // 8, n), dtype=torch.int32, device=self.dev)
            self._chk(lib.zlref_shuffle_awq(p(qin), k, n, 1, p(qw)))
            qz = self.t(qzeros)
            self._chk(lib.zlref_un_shuffle(p(qz), qz.shape[0], qz.shape[1]))
        else:
            k8, n = qweight.shape
            k = k8 * 8
            qw = self.t(qweight)
            self._chk(lib.zlref_gptq_shuffle(p(qw), k, n))
            qz = self.t(qzeros)
            self._chk(lib.zlref_increase_zero(p(qz), qz.shape[0], qz.shape[1]))
        g = qz.shape[0]
        z8 = torch.empty((g, n), dtype=torch.uint8, device=self.dev)
        self._chk(lib.zlref_q4_to_q8(p(qz), g, n // 8, p(z8)))
        qw_km = torch.empty((n, k // 8), dtype=torch.int32, device=self.dev)
        qz_km = torch.empty((n, g), dtype=torch.uint8, device=self.dev)
        sc = self.t(scales)
        sc_km = torch.empty((n, g), dtype=torch.float16, device=self.dev)
        self._chk(lib.zlref_transpose(p(qw), k // 8, n, 4, p(qw_km)))
        self._chk(lib.zlref_transpose(p(z8), g, n, 1, p(qz_km)))
        self._chk(lib.zlref_transpose(p(sc), g, n, 2, p(sc_km)))
        return qw_km, qz_km, sc_km

    def dequant_k_major(self, qw_km, qz_km, sc_km):
        n, k8 = qw_km.shape
        out = torch.empty((n, k8 * 8), dtype=torch.float16, device=self.dev)
        self._chk(self.lib.zlref_dequant_k_major(self.p(qw_km), self.p(qz_km), self.p(sc_km), n, k8 * 8, sc_km.shape[1],
                                                 self.p(out)))
        return out

    def gemv(self, x, qw_km, qz_km, sc_km, bias=None, sym=False):
        m, k = x.shape
        n = qw_km.shape[0]
        out = torch.empty((m, n), dtype=torch.float16, device=self.dev)
        self._chk(self.lib.zlref_gptq_gemm_k_major(self.p(x), self.p(qw_km), self.p(qz_km), self.p(sc_km), self.p(bias),
                                                   int(sym), m, n, k, sc_km.shape[1], self.p(out)))
        return out

    def gate_in(self, x, gate, up, sym=False):
        m, k = x.shape
        n = gate[0].shape[0]
        out = torch.empty((m, n), dtype=torch.float16, device=self.dev)
        self._chk(self.lib.zlref_gemm_fuse_gate_in(self.p(x), self.p(gate[0]), self.p(gate[1]), self.p(gate[2]),
                                                   self.p(up[0]), self.p(up[1]), self.p(up[2]), int(sym), m, n, k,
                                                   gate[2].shape[1], self.p(out)))
        return out

    def rmsnorm(self, x, w, eps):
        out = torch.empty_like(x)
        self._chk(self.lib.zlref_rmsnorm(self.p(x), self.p(w), x.shape[0], x.shape[1], ctypes.c_float(eps),
                                         0 if x.dtype == torch.float16 else 1, self.p(out)))
        return out

    def rmsnorm_fuse_add(self, a, b, w, eps):
        s, out = torch.empty_like(a), torch.empty_like(a)
        self._chk(self.lib.zlref_rmsnorm_fuse_add(self.p(a), self.p(b), self.p(w), a.shape[0], a.shape[1],
                                                  ctypes.c_float(eps), 0 if a.dtype == torch.float16 else 1, self.p(s),
                                                  self.p(out)))
        return s, out

    def element_add(self, a, b):
        out = torch.empty_like(a)
        self._chk(self.lib.zlref_element_add_scale(self.p(a), self.p(b), ctypes.c_size_t(a.numel()), ctypes.c_float(1.0),
                                                   0 if a.dtype == torch.float16 else 1, self.p(out)))
        return out

    def gate_mul(self, gate, up):
        g = gate.clone()
        self._chk(self.lib.zlref_gate_mul_inplace(self.p(g), self.p(up), g.shape[0], g.shape[1],
                                                  0 if g.dtype == torch.float16 else 1))
        return g

    def rope_qk_cache(self, cos, sin, qkv, hq, hkv, d):
        t = qkv.shape[0]
        q = torch.empty((t, hq * d), dtype=qkv.dtype, device=self.dev)
        k = torch.empty((t, hkv * d), dtype=qkv.dtype, device=self.dev)
        v = torch.empty_like(k)
        self._chk(self.lib.zlref_rope_qk_cache(self.p(cos), self.p(sin), self.p(qkv), t, hq, hkv, d,
                                               0 if qkv.dtype == torch.float16 else 1, self.p(q), self.p(k), self.p(v)))
        return q, k, v

    def attention(self, q, lens, ks, vs, mask_flat, scale, hkv, algo_id=-1):
        b, len_q, hq, d = q.shape
        ka = torch.tensor([t.data_ptr() for t in ks], dtype=torch.int64, device=self.dev)
        va = torch.tensor([t.data_ptr() for t in vs], dtype=torch.int64, device=self.dev)
        out = torch.empty_like(q)
        self._chk(self.lib.zlref_mqa_rag_buffer(self.p(q), self.p(lens), self.p(ka), self.p(va), self.p(mask_flat),
                                                ctypes.c_size_t(mask_flat.numel()), ctypes.c_float(scale),
                                                int(lens.max().item()), b, len_q, hq, hkv, d,
                                                0 if q.dtype == torch.float16 else 1, algo_id, self.p(out)))
        return out

    def quant_calc_scale_dt(self, x):
        m, k = x.shape
        q = torch.empty((m, k), dtype=torch.int8, device=self.dev)
        s = torch.empty(m, dtype=torch.float32, device=self.dev)
        self._chk(self.lib.zlref_quant_calc_scale(self.p(x), m, k, 0 if x.dtype == torch.float16 else 1, self.p(q),
                                                  self.p(s)))
        return q, s

    def quant_calc_scale(self, x):
        m, k = x.shape
        q = torch.empty((m, k), dtype=torch.int8, device=self.dev)
        s = torch.empty(m, dtype=torch.float32, device=self.dev)
        self._chk(self.lib.zlref_quant_calc_scale(self.p(x), m, k, 0, self.p(q), self.p(s)))
        return q, s

    def quant_scale_back(self, acc, sx, sy, dtype):
        m, n = acc.shape
        code = {torch.float16: 0, torch.bfloat16: 1, torch.float32: 2}
        out = torch.empty((m, n), dtype=dtype, device=self.dev)
        self._chk(self.lib.zlref_quant_scale_back(self.p(acc), self.p(sx), self.p(sy), code[sy.dtype], m, n, code[dtype],
                                                  self.p(out)))
        return out

    def layernorm_quant(self, x, w, eps, scale=1.0):
        t, d = x.shape
        y = torch.empty_like(x)
        q = torch.empty((t, d), dtype=torch.int8, device=self.dev)
        s = torch.empty(t, dtype=torch.float32, device=self.dev)
        self._chk(self.lib.zlref_layernorm_quant(self.p(x), self.p(w), t, d, ctypes.c_float(eps), ctypes.c_float(scale),
                                                 0 if x.dtype == torch.float16 else 1, self.p(y), self.p(q), self.p(s)))
        return y, q, s

    def fp8_quant(self, x):
        m, k = x.shape
        q = torch.empty((m, k), dtype=torch.uint8, device=self.dev)
        s = torch.empty(1, dtype=torch.float32, device=self.dev)
        self._chk(self.lib.zlref_fp8_dynamic_scaled_quant(self.p(x), m, k, 0 if x.dtype == torch.float16 else 1,
                                                          self.p(q), self.p(s)))
        return q, s

    def fp8_gemm(self, xq, sx, wq, sw, bias, dtype):
        m, k = xq.shape
        n = wq.shape[0]
        out = torch.empty((m, n), dtype=dtype, device=self.dev)
        self._chk(self.lib.zlref_fp8_gemm(self.p(xq), self.p(sx), self.p(wq), self.p(sw), self.p(bias), m, n, k,
                                          0 if dtype == torch.float16 else 1, self.p(out)))
        return out

    def quant_group_32(self, x):
        m = x.numel() // 32
        q = torch.empty(m * 32, dtype=torch.int8, device=self.dev)
        s = torch.empty(m, dtype=x.dtype, device=self.dev)
        self._chk(self.lib.zlref_quant_group_32(self.p(x), ctypes.c_size_t(m), 0, self.p(q), self.p(s)))
        return q.view(m, 32), s

    def dequant_sum_quant_g32(self, my, q_others, s_others):
        ws = q_others.shape[0] + 1
        m = my.numel() // 32
        q = torch.empty((m, 32), dtype=torch.int8, device=self.dev)
        s = torch.empty(m, dtype=my.dtype, device=self.dev)
        self._chk(self.lib.zlref_dequant_sum_quant_g32(self.p(my), self.p(q_others), self.p(s_others), ws,
                                                       ctypes.c_size_t(m), 0, self.p(q), self.p(s)))
        return q, s

    def dequant_group_32(self, q, s):
        m = q.numel() // 32
        out = torch.empty((m, 32), dtype=s.dtype, device=self.dev)
        self._chk(self.lib.zlref_dequant_group_32(self.p(q), self.p(s), ctypes.c_size_t(m), 0, self.p(out)))
        return out


def allreduce_int8_with_reference_kernels(ref, parts):
    """model_context.cpp:244-326 with the reference's three kernels, the exchanges done in numpy."""
    ws = len(parts)
    numel = parts[0].size
    m = numel // ws // 32
    sent = []
    for r in range(ws):
        q, s = ref.quant_group_32(ref.t(parts[r].reshape(ws * m, 32)))
        sent.append((q.view(ws, m, 32), s.view(ws, m)))
    q_sum, s_sum = [], []
    for r in range(ws):
        qo = torch.stack([sent[(r + i + 1) % ws][0][r] for i in range(ws - 1)]).contiguous()
        so = torch.stack([sent[(r + i + 1) % ws][1][r] for i in range(ws - 1)]).contiguous()
        my = ref.t(parts[r].reshape(ws, m, 32)[r])
        q, s = ref.dequant_sum_quant_g32(my, qo, so)
        q_sum.append(q)
        s_sum.append(s)
    out = ref.dequant_group_32(torch.cat(q_sum).contiguous(), torch.cat(s_sum).contiguous())
    return out.cpu().numpy().reshape(parts[0].shape)


def main(out_dir, lib_path=None):
    os.makedirs(out_dir, exist_ok=True)
    ref = Ref(lib_path=lib_path)
    n = lambda t: t.cpu().numpy()

    c = gc.case_gptq_layout()
    qw_km, qz_km, sc_km = ref.gptq_to_k_major(c["qweight"], c["qzeros"], c["scales"])
    np.savez(os.path.join(out_dir, "ref_gptq_layout.npz"), qw_km=n(qw_km), qz_km=n(qz_km), sc_km=n(sc_km),
             w16=n(ref.dequant_k_major(qw_km, qz_km, sc_km)))

    c = gc.case_awq_layout()
    qw_km, qz_km, sc_km = ref.gptq_to_k_major(c["qweight"], c["qzeros"], c["scales"], awq=True)
    np.savez(os.path.join(out_dir, "ref_awq_layout.npz"), qw_km=n(qw_km), qz_km=n(qz_km), sc_km=n(sc_km),
             w16=n(ref.dequant_k_major(qw_km, qz_km, sc_km)))

    for sym in (False, True):
        c = gc.case_gemv(sym)
        outs = {}
        for m, x in c["xs"].items():
            outs["y%d" % m] = n(ref.gemv(ref.t(x), ref.t(c["qw_km"]), ref.t(c["qz_km"]), ref.t(c["sc_km"]), None, sym))
            outs["yb%d" % m] = n(ref.gemv(ref.t(x), ref.t(c["qw_km"]), ref.t(c["qz_km"]), ref.t(c["sc_km"]),
                                          ref.t(c["bias"]), sym))
        np.savez(os.path.join(out_dir, "ref_gemv_%s.npz" % ("sym" if sym else "asym")), **outs)

    c = gc.case_gate_in()
    gate = [ref.t(a.view(np.int32) if a.dtype == np.uint32 else a) for a in c["gate"]]
    up = [ref.t(a.view(np.int32) if a.dtype == np.uint32 else a) for a in c["up"]]
    outs = {}
    for m, x in c["xs"].items():
        outs["y%d" % m] = n(ref.gate_in(ref.t(x), gate, up))
        g = ref.gemv(ref.t(x), gate[0], gate[1], gate[2])
        u = ref.gemv(ref.t(x), up[0], up[1], up[2])
        outs["unfused%d" % m] = n(ref.gate_mul(g, u))
    np.savez(os.path.join(out_dir, "ref_gate_in.npz"), **outs)

    c = gc.case_norm()
    a, b, w = ref.t(c["a"]), ref.t(c["b"]), ref.t(c["w"])
    s, y_fuse = ref.rmsnorm_fuse_add(a, b, w, c["eps"])
    np.savez(os.path.join(out_dir, "ref_norm.npz"), y=n(ref.rmsnorm(a, w, c["eps"])), s=n(s), y_fuse=n(y_fuse),
             add=n(ref.element_add(a, b)), y_after_add=n(ref.rmsnorm(ref.element_add(a, b), w, c["eps"])),
             gate_mul=n(ref.gate_mul(a, b)))

    c = gc.case_rope()
    q, k, v = ref.rope_qk_cache(ref.t(c["cos"]), ref.t(c["sin"]), ref.t(c["qkv"]), c["hq"], c["hkv"], c["d"])
    np.savez(os.path.join(out_dir, "ref_rope.npz"), q=n(q), k=n(k), v=n(v))

    for long in (False, True):
        c = gc.case_attention(long)
        ks, vs = [ref.t(x) for x in c["ks"]], [ref.t(x) for x in c["vs"]]
        mask = ref.t(np.concatenate([m.reshape(-1) for m in c["masks"]]))
        out = ref.attention(ref.t(c["q"]), ref.t(c["lens"]), ks, vs, mask, c["scale"], c["hkv"])
        np.savez(os.path.join(out_dir, "ref_attention_%s.npz" % ("long" if long else "short")), out=n(out))

    c = gc.case_int8()
    q, s = ref.quant_calc_scale(ref.t(c["x"]))
    np.savez(os.path.join(out_dir, "ref_int8.npz"), q=n(q), s=n(s),
             allreduce=allreduce_int8_with_reference_kernels(ref, c["parts"]))
    c = gc.case_w8()
    outs = {}
    for tag, dt in (("f16", torch.float16), ("bf16", torch.bfloat16)):
        x = ref.t(c["x"]).to(dt)
        q, sx = ref.quant_calc_scale_dt(x)
        acc = (q.cpu().int() @ torch.from_numpy(c["w_q"]).int().T).to(ref.dev)
        sw = ref.t(c["w_s"]).to(dt)
        outs["q_" + tag], outs["sx_" + tag], outs["acc_" + tag] = n(q), n(sx), n(acc)
        outs["back_" + tag] = n(ref.quant_scale_back(acc, sx, sw, dt).float())
        outs["back_f32scale_" + tag] = n(ref.quant_scale_back(acc, sx, sw.float(), dt).float())
        y, lq, ls = ref.layernorm_quant(x, ref.t(c["ln_w"]).to(dt), c["eps"])
        outs["ln_y_" + tag], outs["ln_q_" + tag], outs["ln_s_" + tag] = n(y.float()), n(lq), n(ls)
        fq, fs = ref.fp8_quant(x)
        outs["f8_q_" + tag], outs["f8_s_" + tag] = n(fq), n(fs)
        sw8 = ref.t(np.array([c["w_f8_scale"]], np.float32))
        outs["f8_y_" + tag] = n(ref.fp8_gemm(fq, fs, ref.t(c["w_f8"]), sw8, None, dt).float())
        outs["f8_y_bias_" + tag] = n(ref.fp8_gemm(fq, fs, ref.t(c["w_f8"]), sw8, ref.t(c["bias"]).to(dt), dt).float())
    np.savez(os.path.join(out_dir, "ref_w8.npz"), **outs)

    c = gc.case_rope_tables()
    outs = {}
    for name, (d, theta, l3) in c["variants"].items():
        cos, sin = ref.rope_cos_sin(ref.t(c["pos"]), d, theta, l3)
        outs["cos_" + name], outs["sin_" + name] = n(cos), n(sin)
    np.savez(os.path.join(out_dir, "ref_rope_tables.npz"), **outs)

    c = gc.case_kv8()
    outs = {}
    kq, vq, sk, sv = [], [], [], []
    for i, (k, v) in enumerate(zip(c["ks"], c["vs"])):
        a, s = ref.quant_u8(ref.t(k.reshape(-1, c["d"])))
        kq.append(a.view(k.shape)); sk.append(s.view(k.shape[0], c["hkv"]))
        b, s2 = ref.quant_u8(ref.t(v.reshape(-1, c["d"])))
        vq.append(b.view(v.shape)); sv.append(s2.view(v.shape[0], c["hkv"]))
        # the uint8 codes as digests: the whole cache would make the fixture larger than 1 MB
        outs["kq%d_digest" % i], outs["vq%d_digest" % i] = np.array(gc.digest(n(kq[-1]))), np.array(gc.digest(n(vq[-1])))
        outs["sk%d" % i], outs["sv%d" % i] = n(sk[-1]), n(sv[-1])
    mask = ref.t(np.concatenate([m.reshape(-1) for m in c["masks"]]))
    outs["out"] = n(ref.attention_kv8(ref.t(c["q"]), ref.t(c["lens"]), kq, vq, sk, sv, mask, c["scale"], c["hkv"]).float())
    np.savez(os.path.join(out_dir, "ref_kv8.npz"), **outs)

    if not hasattr(ref.lib, "zlref_marlin_gemm"):     # the drop-in library has no counterpart of the reference-only shim
        print("wrote goldens to", out_dir)
        return

    c = gc.case_marlin()
    outs = {"repacked": n(ref.marlin_repack(ref.t(c["qweight"])))}
    for m, x in c["xs"].items():
        outs["y%d" % m] = n(ref.marlin_gemm(ref.t(x), ref.t(c["qweight"]), ref.t(c["scales"])))
    np.savez(os.path.join(out_dir, "ref_marlin.npz"), **outs)
    print("wrote goldens to", out_dir)


if __name__ == "__main__":
    # usage: gen_ref_golden.py [out_dir] [shim library]   (default: the reference's own kernels, oracle/_ref/libzl_ref.so;
    # oracle/_ref/libzl_dropin.so runs the same calls through integration/zl_nn_dropin.cpp -> libzhilight_b200.so)
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, "..", "gpurun_out", "golden"),
         sys.argv[2] if len(sys.argv) > 2 else None)
    sys.stdout.flush()
    os._exit(0)      # bmengine statics are torn down after the CUDA driver at interpreter exit
