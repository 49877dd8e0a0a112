"""Torch-tensor front end of the C-ABI (plumbing only: torch supplies device memory and streams).

Every function takes CUDA tensors, passes raw pointers to libzhilight_b200.so on the current stream and
returns torch tensors.  Names / argument meaning mirror the reference operator each one replaces.
"""
import ctypes

import torch

from . import _lib

F16, BF16, F32 = 0, 1, 2
EPI_NONE, EPI_SWIGLU, EPI_RESIDUAL, EPI_QKV_ROPE = 0, 1, 2, 3


def _dt(t):
    if t.dtype == torch.float16:
        return F16
    if t.dtype == torch.bfloat16:
        return BF16
    if t.dtype == torch.float32:
        return F32
    raise _lib.ZLError(-2, "unsupported dtype %s" % t.dtype)


def _p(t):
    if t is None:
        return None
    if not t.is_cuda:
        raise _lib.ZLError(-1, "zhilight_b200 ops need CUDA tensors (no CPU fallback)")
    if not t.is_contiguous():
        raise _lib.ZLError(-1, "tensor must be contiguous")
    return ctypes.c_void_p(t.data_ptr())


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


# ------------------------------------------------------------------ load-time transforms
def gptq_shuffle(qweight, q_perm=None):
    """nn::gptq::gptq_shuffle -- in place on (K/8, N) int32."""
    k8, n = qweight.shape
    scratch = torch.empty_like(qweight) if q_perm is not None else None
    _lib.call("zl_gptq_shuffle", _p(qweight), _p(q_perm), _p(scratch), k8 * 8, n, _stream())
    return qweight


def gptq_increase_zero(qzeros):
    _lib.call("zl_gptq_increase_zero", _p(qzeros), qzeros.numel(), _stream())
    return qzeros


def gptq_subtract8(words):
    _lib.call("zl_gptq_subtract8", _p(words), words.numel(), _stream())
    return words


def q4_to_q8(qzeros):
    r, c8 = qzeros.shape
    out = torch.empty((r, c8 * 8), dtype=torch.uint8, device=qzeros.device)
    _lib.call("zl_q4_to_q8", _p(qzeros), _p(out), qzeros.numel(), _stream())
    return out


def awq_un_shuffle(qzeros):
    _lib.call("zl_awq_un_shuffle", _p(qzeros), qzeros.shape[0], qzeros.shape[1], _stream())
    return qzeros


def awq_shuffle(qweight, use_exllama=True):
    k, n8 = qweight.shape
    out = torch.empty((k // 8, n8 * 8), dtype=qweight.dtype, device=qweight.device)
    _lib.call("zl_awq_shuffle", _p(qweight), _p(out), k, n8 * 8, int(use_exllama), _stream())
    return out


def transpose_2d(x):
    r, c = x.shape
    out = torch.empty((c, r), dtype=x.dtype, device=x.device)
    _lib.call("zl_transpose_2d", _p(x), _p(out), r, c, x.element_size(), _stream())
    return out


def gptq_to_k_major(qweight, qzeros, scales, is_awq=False):
    """Int4GPTQ::preprocess_weight + transpose_weight (linear.cpp:1139-1160, 1085-1099) on device.
    Consumes copies of the HF tensors; returns (qweight_km (N,K/8) i32, qzeros_km (N,G) u8, scales_km (N,G) f16)."""
    if is_awq:
        qw = awq_shuffle(qweight.contiguous(), True)
        qz = awq_un_shuffle(qzeros.clone())
    else:
        qw = gptq_shuffle(qweight.clone())
        qz = gptq_increase_zero(qzeros.clone())
    z8 = q4_to_q8(qz)
    return transpose_2d(qw), transpose_2d(z8), transpose_2d(scales.contiguous())


def gptq_dequant_k_major(qweight_km, qzeros_km, scales_km):
    n, k8 = qweight_km.shape
    g = scales_km.shape[1]
    out = torch.empty((n, k8 * 8), dtype=torch.float16, device=qweight_km.device)
    _lib.call("zl_gptq_dequant_k_major", _p(qweight_km), _p(qzeros_km), _p(scales_km), _p(out), n, k8 * 8,
              (k8 * 8) // g, _stream())
    return out


def w4_pack(qweight_km, qzeros_km, scales_km, group_size=128, sym=False, row_map=None, variant=0):
    n_src, k8 = qweight_km.shape
    n = n_src if row_map is None else row_map.numel()
    k = k8 * 8
    nbytes = _lib.load().zl_w4_packed_bytes(n, k, group_size)
    if nbytes == 0:
        raise _lib.ZLError(-2, "unsupported ZLW4 shape N=%d K=%d group=%d" % (n, k, group_size))
    packed = torch.empty(nbytes, dtype=torch.uint8, device=qweight_km.device)
    _lib.call("zl_w4_pack_v", _p(qweight_km), _p(qzeros_km), _p(scales_km), _p(row_map), _p(packed), n, k, group_size,
              int(sym), int(variant), _stream())
    return packed


def w4_unpack(packed, n, k, group_size=128, variant=0):
    dev = packed.device
    qw = torch.empty((n, k // 8), dtype=torch.int32, device=dev)
    qz = torch.empty((n, k // group_size), dtype=torch.uint8, device=dev)
    sc = torch.empty((n, k // group_size), dtype=torch.float16, device=dev)
    _lib.call("zl_w4_unpack_v", _p(packed), _p(qw), _p(qz), _p(sc), n, k, group_size, int(variant), _stream())
    return qw, qz, sc


def swiglu_row_map(f, device):
    p = torch.arange(2 * f, device=device, dtype=torch.int32)
    tile, r = p // 16, p % 16
    return torch.where(r < 8, tile * 8 + r, f + tile * 8 + (r - 8)).to(torch.int32).contiguous()


# ------------------------------------------------------------------ compute
def w4a16_gemm(x, packed, n, k, group_size=128, bias=None, residual=None, epilogue=EPI_NONE, pdl=False, out=None):
    """nn::gptq::gptq_gemm_k_major (GEMV path) on the ZLW4 layout."""
    if x.dtype != torch.float16:
        raise _lib.ZLError(-2, "A must be half")      # q_gemm_k_major.cu:989
    m = x.shape[0]
    n_out = n // 2 if epilogue == EPI_SWIGLU else n
    if out is None:
        out = torch.empty((m, n_out), dtype=torch.float16, device=x.device)
    _lib.call("zl_w4a16_gemm", _p(x), x.stride(0), _p(packed), _p(bias), _p(residual), _p(out), m, n, k, group_size,
              epilogue, int(pdl), _stream())
    return out


def _dp(t):
    return t.data_ptr() if t is not None else None


def qkv_rope_row_map(n_heads_total, dim_head, device):
    m = torch.empty(n_heads_total * dim_head, dtype=torch.int32, device=device)
    _lib.call("zl_qkv_rope_row_map", _p(m), n_heads_total, dim_head, _stream())
    return m


def gather_rows_16(src, row_map):
    dst = torch.empty(row_map.numel(), dtype=src.dtype, device=src.device)
    _lib.call("zl_gather_rows_16", _p(src), _p(row_map), _p(dst), row_map.numel(), _stream())
    return dst


def w4a16_gemm_fused(x, packed, n, k, group_size=128, bias=None, residual=None, epilogue=EPI_NONE, pdl=False, out=None,
                     ln_weight=None, eps=1e-5, rope=None, variant=0):
    """zl_w4a16_gemm_fused.  rope = dict(cos, sin, token_batch, placement, k_bufs, v_bufs, num_heads, num_kv_heads,
    dim_head) for EPI_QKV_ROPE (returns q); bias must be in packed-row order."""
    if x.dtype != torch.float16:
        raise _lib.ZLError(-2, "A must be half")
    m = x.shape[0]
    a = _lib.W4FusedArgs()
    a.x, a.ldx, a.packed, a.bias, a.residual = x.data_ptr(), x.stride(0), packed.data_ptr(), _dp(bias), _dp(residual)
    a.M, a.N, a.K, a.group_size, a.epilogue, a.pdl = m, n, k, group_size, epilogue, int(pdl)
    a.ln_weight, a.eps = _dp(ln_weight), eps
    a.variant = int(variant)
    keep = []
    if epilogue == EPI_QKV_ROPE:
        r = rope
        q = torch.empty((m, r["num_heads"] * r["dim_head"]), dtype=torch.float16, device=x.device)
        ka, va = _ptr_table(r["k_bufs"], x.device), _ptr_table(r["v_bufs"], x.device)
        keep += [ka, va]
        a.cos, a.sin, a.q_out = r["cos"].data_ptr(), r["sin"].data_ptr(), q.data_ptr()
        a.token_batch, a.placement = r["token_batch"].data_ptr(), r["placement"].data_ptr()
        a.k_addrs, a.v_addrs = ka.data_ptr(), va.data_ptr()
        a.num_heads, a.num_kv_heads, a.dim_head = r["num_heads"], r["num_kv_heads"], r["dim_head"]
        ret = q
    else:
        n_out = n // 2 if epilogue == EPI_SWIGLU else n
        if out is None:
            out = torch.empty((m, n_out), dtype=torch.float16, device=x.device)
        a.y = out.data_ptr()
        ret = out
    _lib.call("zl_w4a16_gemm_fused", ctypes.byref(a), _stream())
    if keep:
        torch.cuda.current_stream().synchronize()
    return ret


def dense_gemm_skinny(x, w, bias=None, out_dtype=None, pdl=False):
    m, k = x.shape
    n = w.shape[0]
    od = x.dtype if out_dtype is None else out_dtype
    out = torch.empty((m, n), dtype=od, device=x.device)
    _lib.call("zl_dense_gemm_skinny", _p(x), x.stride(0), _p(w), _p(bias), _p(out), m, n, k, _dt(x), _dt(out),
              int(pdl), _stream())
    return out


W8_INT8, W8_FP8 = 0, 1


def int8_quant_per_token(x, pdl=False):
    """int8_op::quant_calc_scale: returns (q int8 (M,K), scale f32 (M))."""
    m, k = x.shape
    q = torch.empty((m, k), dtype=torch.int8, device=x.device)
    scale = torch.empty((m,), dtype=torch.float32, device=x.device)
    _lib.call("zl_int8_quant_per_token", _p(x), x.stride(0), _p(q), _p(scale), m, k, _dt(x), int(pdl), _stream())
    return q, scale


def rmsnorm_quant(x, weight, eps, scale=1.0, pdl=False):
    """int8_op::layernorm_quant: returns (y, q int8, qscale f32 (T))."""
    t, d = x.shape
    y = torch.empty_like(x)
    q = torch.empty((t, d), dtype=torch.int8, device=x.device)
    qs = torch.empty((t,), dtype=torch.float32, device=x.device)
    _lib.call("zl_rmsnorm_quant", _p(x), _p(weight), _p(y), _p(q), _p(qs), t, d, eps, scale, _dt(x), int(pdl),
              _stream())
    return y, q, qs


def fp8_quant_per_tensor(x, pdl=False):
    """nn::fp8::dynamic_scaled_quant: returns (q uint8 holding e4m3 bits, scale f32 (1))."""
    q = torch.empty(x.shape, dtype=torch.uint8, device=x.device)
    scale = torch.empty((1,), dtype=torch.float32, device=x.device)
    _lib.call("zl_fp8_quant_per_tensor", _p(x), _p(q), _p(scale), x.numel(), _dt(x), int(pdl), _stream())
    return q, scale


def w8a8_gemm(xq, x_scale, w, w_scale, out_dtype, kind=W8_INT8, bias=None, pdl=False):
    m, k = xq.shape
    n = w.shape[0]
    y = torch.empty((m, n), dtype=out_dtype, device=xq.device)
    ws_dt = 2 if w_scale.dtype == torch.float32 else _dt(w_scale)
    _lib.call("zl_w8a8_gemm", _p(xq), _p(x_scale), _p(w), _p(w_scale), ws_dt, _p(bias), _p(y), m, n, k, kind,
              _dt(y), int(pdl), _stream())
    return y


def int8_linear(x, w_q, w_scale, bias=None, pdl=False):
    """Int8Linear::forward (linear.cpp:560-636) in two launches instead of three."""
    q, s = int8_quant_per_token(x, pdl)
    return w8a8_gemm(q, s, w_q, w_scale, x.dtype, W8_INT8, bias, pdl)


def fp8_linear(x, w_fp8, w_scale, bias=None, pdl=False):
    """Fp8Linear::forward (linear.cpp:1660-1695)."""
    q, s = fp8_quant_per_tensor(x, pdl)
    return w8a8_gemm(q, s, w_fp8, w_scale, x.dtype, W8_FP8, bias, pdl)


def rmsnorm(x, weight, eps, scale=1.0, pdl=False):
    t, d = x.shape
    y = torch.empty_like(x)
    _lib.call("zl_rmsnorm", _p(x), _p(weight), _p(y), t, d, eps, scale, _dt(x), int(pdl), _stream())
    return y


def add_rmsnorm(a, b, weight, eps, scale=1.0, mode=0, pdl=False):
    t, d = a.shape
    out_sum = torch.empty_like(a)
    y = torch.empty_like(a)
    _lib.call("zl_add_rmsnorm", _p(a), _p(b), _p(weight), _p(out_sum), _p(y), t, d, eps, scale, mode, _dt(a),
              int(pdl), _stream())
    return out_sum, y


def element_add_scale(a, b, scale=1.0):
    c = torch.empty_like(a)
    _lib.call("zl_element_add_scale", _p(a), _p(b), _p(c), a.numel(), scale, _dt(a), _stream())
    return c


def gate_mul(gate, up, act="silu"):
    t, f = gate.shape
    out = torch.empty((t, f), dtype=gate.dtype, device=gate.device)
    # strided views are fine here: the C entry point takes row strides
    _lib.call("zl_gate_mul", ctypes.c_void_p(gate.data_ptr()), gate.stride(0),
              ctypes.c_void_p(up.data_ptr()) if up is not None else None, up.stride(0) if up is not None else 0, _p(out), f, t, f, 0 if act == "silu" else 1, _dt(gate), _stream())
    return out


def activation(x, act):
    """Linear::activate: silu / gelu in fp32, rounded to T."""
    return gate_mul(x, None, act)


def rope_cos_sin(pos, dim_head, theta, llama3=None, neox=True):
    t = pos.numel()
    cos = torch.empty((t, dim_head), dtype=torch.float32, device=pos.device)
    sin = torch.empty_like(cos)
    l3 = llama3 or {}
    _lib.call("zl_rope_cos_sin", _p(pos), _p(cos), _p(sin), t, dim_head, float(theta),
              float(l3.get("factor", 0.0)), float(l3.get("low", 1.0)), float(l3.get("high", 4.0)),
              float(l3.get("orig", 8192.0)), int(neox), _stream())
    return cos, sin


def rope_qk_cache(cos, sin, qkv, num_heads, num_kv_heads, dim_head, neox=True):
    t = qkv.shape[0]
    q = torch.empty((t, num_heads * dim_head), dtype=qkv.dtype, device=qkv.device)
    k = torch.empty((t, num_kv_heads * dim_head), dtype=qkv.dtype, device=qkv.device)
    v = torch.empty_like(k)
    _lib.call("zl_rope_qk_cache", _p(cos), _p(sin), _p(qkv), _p(q), _p(k), _p(v), t, num_heads, num_kv_heads,
              dim_head, int(neox), _dt(qkv), _stream())
    return q, k, v


def _ptr_table(tensors, device):
    return torch.tensor([t.data_ptr() for t in tensors], dtype=torch.int64, device=device)


def copy_to_rag_buffer2(placement, buf_lens, k_src, v_src, k_bufs, v_bufs, bshd=True):
    b, len_q, hkv, d = k_src.shape
    ka, va = _ptr_table(k_bufs, k_src.device), _ptr_table(v_bufs, k_src.device)
    _lib.call("zl_copy_to_rag_buffer2", _p(placement), _p(buf_lens), _p(k_src), _p(v_src), _p(ka), _p(va), b, len_q,
              hkv, d, int(bshd), _dt(k_src), _stream())
    torch.cuda.current_stream().synchronize()      # keep the pointer tables alive until the copy ran


def qkv_rope_append(cos, sin, qkv, token_batch, placement, k_bufs, v_bufs, num_heads, num_kv_heads, dim_head,
                    buf_lens=None, neox=True, bshd=True, pdl=False):
    t = qkv.shape[0]
    q = torch.empty((t, num_heads * dim_head), dtype=qkv.dtype, device=qkv.device)
    ka, va = _ptr_table(k_bufs, qkv.device), _ptr_table(v_bufs, qkv.device)
    _lib.call("zl_qkv_rope_append", _p(cos), _p(sin), _p(qkv), _p(q), _p(token_batch), _p(placement), _p(ka), _p(va),
              t, num_heads, num_kv_heads, dim_head, int(neox), int(bshd), _p(buf_lens), _dt(qkv), int(pdl), _stream())
    torch.cuda.current_stream().synchronize()
    return q


def decode_attention(q, buf_lens, k_bufs, v_bufs, mask, scale, max_len_buf, num_kv_heads, bshd=True, pdl=False):
    """nn::multi_query_attention_rag_buffer: q (B, len_q, H_q, d); k_bufs/v_bufs lists of per-task tensors."""
    b, len_q, hq, d = q.shape
    out = torch.empty_like(q)
    ws_bytes = _lib.load().zl_decode_attention_workspace_bytes(b, len_q, hq, d, max_len_buf)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=q.device)
    ka, va = _ptr_table(k_bufs, q.device), _ptr_table(v_bufs, q.device)
    _lib.call("zl_decode_attention", _p(q), _p(buf_lens), _p(ka), _p(va), _p(mask), float(scale), max_len_buf,
              _p(out), b, len_q, hq, num_kv_heads, d, int(bshd), _p(ws), ws_bytes, _dt(q), int(pdl), _stream())
    torch.cuda.current_stream().synchronize()
    return out


def decode_attention_kv8(q, buf_lens, k_bufs, v_bufs, sk_bufs, sv_bufs, mask, scale, max_len_buf, num_kv_heads, out_dtype=None,
                         pdl=False):
    """int8 KV cache attention: q (B, len_q, H_q, d) f16; k/v lists of (len_buf, H_kv, d) uint8; sk/sv lists of
    (len_buf, H_kv) fp32 scales."""
    b, len_q, hq, d = q.shape
    out = torch.empty(q.shape, dtype=out_dtype or q.dtype, device=q.device)
    ws_bytes = _lib.load().zl_decode_attention_workspace_bytes(b, len_q, hq, d, max_len_buf)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=q.device)
    tabs = [_ptr_table(x, q.device) for x in (k_bufs, v_bufs, sk_bufs, sv_bufs)]
    _lib.call("zl_decode_attention_kv8", _p(q), _p(buf_lens), _p(tabs[0]), _p(tabs[1]), _p(tabs[2]), _p(tabs[3]), _p(mask),
              float(scale), max_len_buf, _p(out), b, len_q, hq, num_kv_heads, d, _p(ws), ws_bytes, _dt(out), int(pdl),
              _stream())
    torch.cuda.current_stream().synchronize()
    return out


def kv_int8_quant_append(k_src, v_src, token_batch, placement, k_bufs, v_bufs, sk_bufs, sv_bufs):
    """k_src / v_src (T, H_kv, d) -> uint8 codes + fp32 scales scattered into the per-task caches."""
    t, hkv, d = k_src.shape
    tabs = [_ptr_table(x, k_src.device) for x in (k_bufs, v_bufs, sk_bufs, sv_bufs)]
    _lib.call("zl_kv_int8_quant_append", _p(k_src), _p(v_src), _p(token_batch), _p(placement), _p(tabs[0]), _p(tabs[1]),
              _p(tabs[2]), _p(tabs[3]), t, hkv, d, _dt(k_src), 0, _stream())
    torch.cuda.current_stream().synchronize()


def embedding(ids, table):
    t = ids.numel()
    out = torch.empty((t, table.shape[1]), dtype=table.dtype, device=table.device)
    _lib.call("zl_embedding", _p(ids), _p(table), _p(out), t, table.shape[1], table.shape[0], _dt(table), 0, _stream())
    return out


def argmax(logits):
    t, v = logits.shape
    out = torch.empty(t, dtype=torch.int32, device=logits.device)
    nb = _lib.load().zl_argmax_workspace_bytes(t)
    ws = torch.empty(nb, dtype=torch.uint8, device=logits.device)
    _lib.call("zl_argmax", _p(logits), _p(out), t, v, _p(ws), nb, 0, _stream())
    return out


def sample_params(tasks, device, vocab):
    """zl_sample_params_t records on `device` (a uint8 tensor) from a list of dicts with the keys of
    LlamaDecoder.set_sampling (temperature, top_p, top_k, repetition_penalty, presence_penalty, seed), validated as
    random_util.cu:121-122 asserts (temperature > 0, 0 <= top_p <= 1, 0 <= top_k < vocab)."""
    recs = (_lib.SampleParams * len(tasks))()
    for i, t in enumerate(tasks):
        r = recs[i]
        r.temperature = float(t.get("temperature", 1.0))
        r.top_p = float(t.get("top_p", 1.0))
        r.top_k = int(t.get("top_k", 0))
        r.repetition_penalty = float(t.get("repetition_penalty", 1.0))
        r.presence_penalty = float(t.get("presence_penalty", 0.0))
        r.seed = int(t.get("seed", 0)) & 0xFFFFFFFFFFFFFFFF
        if not (r.temperature > 0 and 0 <= r.top_p <= 1 and 0 <= r.top_k < vocab and r.repetition_penalty > 0):
            raise _lib.ZLError(-1, "invalid sampling parameters %r" % (t,))
    raw = bytes(recs)
    return torch.frombuffer(bytearray(raw), dtype=torch.uint8).to(device)


def sample(logits, params, seen_bits, draw_counters, row_task=None):
    """zl_sample: one pick per row of fp32 logits (T, V).  params: sample_params(...) of the tasks; seen_bits: int32
    (tasks, ceil(V/32)) seen-token bits; draw_counters: int32 (tasks); row_task: int32 (T) task of each row (default
    row i -> task i).  Updates seen_bits and draw_counters in place like the decode driver; returns int32 (T)."""
    t, v = logits.shape
    if row_task is None:
        row_task = torch.arange(t, dtype=torch.int32, device=logits.device)
    for x, dt in ((logits, torch.float32), (seen_bits, torch.int32), (draw_counters, torch.int32), (row_task, torch.int32)):
        if x.dtype != dt:
            raise _lib.ZLError(-1, "sample: expected %s, got %s" % (dt, x.dtype))
    if seen_bits.shape[-1] != (v + 31) // 32:
        raise _lib.ZLError(-1, "seen_bits must hold ceil(V/32) words per task")
    out = torch.empty(t, dtype=torch.int32, device=logits.device)
    nb = _lib.load().zl_sample_workspace_bytes(t, v)
    ws = torch.empty(max(nb, 1), dtype=torch.uint8, device=logits.device)
    _lib.call("zl_sample", _p(logits), t, v, _p(row_task), _p(params), _p(seen_bits), _p(draw_counters), _p(out), _p(ws),
              nb, 0, _stream())
    return out


def sample_uniform(seed, draw_index):
    """The u in (0, 1] zl_sample draws for (seed, draw_index) (host computation, no GPU needed)."""
    lib = _lib.load()
    return float(lib.zl_sample_uniform(int(seed) & 0xFFFFFFFFFFFFFFFF, int(draw_index)))
