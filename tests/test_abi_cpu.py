"""CPU-only checks of the drop-in boundary: the C-ABI library builds, loads, exports every symbol the
header declares, and rejects bad arguments with error codes (no compute call needs a GPU here)."""
import ctypes
import os

import numpy as np
import pytest

from tests.helpers import attention_plan
from zhilight_b200 import _lib


def test_library_exports_every_declared_symbol(lib):
    protos = _lib.parse_header()
    assert len(protos) >= 40
    for name in protos:
        assert hasattr(lib, name), name


def test_header_cites_reference_for_compute_entry_points():
    src = open(_lib.HEADER).read()
    for must in ("q_gemm_k_major.cu", "attention_kernel.cu", "rotary_embedding_fuse_cache.cu", "layernorm.cu",
                 "ragged_buffer_kernel.cu", "linear.cpp", "utils.cu"):
        assert must in src, must


def test_version_and_error_string(lib):
    assert lib.zl_version() >= 100
    rc = lib.zl_gptq_increase_zero(None, 0, None)
    assert rc == -1
    assert b"invalid argument" in lib.zl_last_error()


def test_packed_bytes(lib):
    assert lib.zl_w4_packed_bytes(4096, 4096, 128) == (4096 // 32) * 32 * 2128
    assert lib.zl_w4_packed_bytes(4096, 4096, 64) == 0          # unsupported group size
    assert lib.zl_w4_packed_bytes(100, 4096, 128) == 0          # N % 32


def test_argument_validation_without_gpu(lib):
    p = ctypes.c_void_p(16)
    # group size != 128 is reported as unsupported before any CUDA call
    assert lib.zl_w4a16_gemm(p, 4096, p, None, None, p, 1, 4096, 4096, 64, 0, 0, None) == -2
    # misaligned leading dimension
    assert lib.zl_w4a16_gemm(p, 4097, p, None, None, p, 1, 4096, 4096, 128, 0, 0, None) == -1
    # residual epilogue without residual pointer
    assert lib.zl_w4a16_gemm(p, 4096, p, None, None, p, 1, 4096, 4096, 128, 2, 0, None) == -1
    assert lib.zl_decode_attention(p, p, p, p, None, 1.0, 128, p, 1, 1, 32, 8, 96, 1, None, 0, 0, 0, None) == -2
    assert lib.zl_rmsnorm(p, p, p, 1, 4095, 1e-5, 1.0, 0, 0, None) == -2


def test_ops_refuse_cpu_tensors():
    import torch
    from zhilight_b200 import ops
    with pytest.raises(_lib.ZLError):
        ops.rmsnorm(torch.zeros(1, 64, dtype=torch.float16), torch.ones(64, dtype=torch.float16), 1e-5)


def test_missing_library_fails_loudly(monkeypatch, tmp_path):
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", str(tmp_path / "nope.so"))
    with pytest.raises(_lib.ZLError):
        _lib.load()


@pytest.mark.parametrize("n_tiles,G,ctas", [(224, 32, 148), (48, 32, 148), (32, 32, 128), (32, 112, 148), (1, 8, 4), (7, 5, 3),
                                            (300, 3, 148), (16, 128, 148)])
def test_tcgen05_stream_k_schedule_covers_every_unit_once(n_tiles, G, ctas):
    """The tcgen05 W4 kernel's scheduling code (TcSched in w4a16_tc.cu, exported as zl_w4_tc_schedule): every
    (128-row tile, 128-k group) unit belongs to exactly one piece, a tile's pieces are contiguous in k and counted correctly,
    partial pieces come first in a CTA's order (at most two) and never share a workspace slot."""
    import ctypes
    lib = _lib.load()
    lib.zl_w4_tc_schedule.restype = ctypes.c_int
    covered = np.zeros((n_tiles, G), np.int32)
    pieces_of = {}
    slots = set()
    for cta in range(ctas):
        out = (ctypes.c_int * (5 * 512))()
        n = lib.zl_w4_tc_schedule(n_tiles, G, ctas, cta, out, 512)
        assert n >= 1
        partial_seen_after_whole = False
        seen_whole = False
        n_partial = 0
        for i in range(n):
            tile, g0, g1, nparts, slot = (out[5 * i + j] for j in range(5))
            assert 0 <= tile < n_tiles and 0 <= g0 < g1 <= G
            covered[tile, g0:g1] += 1
            pieces_of.setdefault(tile, []).append((g0, g1, nparts, cta))
            whole = g0 == 0 and g1 == G
            if whole:
                assert slot == -1 and nparts == 1
                seen_whole = True
            else:
                n_partial += 1
                assert i < 2, "partial pieces are processed first"
                assert not seen_whole or i == 1
                assert 0 <= slot < 2 * ctas and slot // 2 == cta and slot not in slots
                slots.add(slot)
        assert n_partial <= 2
    assert (covered == 1).all()
    for tile, ps in pieces_of.items():
        ps.sort()
        assert all(p[2] == len(ps) for p in ps), (tile, ps)
        assert ps[0][0] == 0 and ps[-1][1] == G and all(a[1] == b[0] for a, b in zip(ps, ps[1:]))
        assert [p[3] for p in ps] == list(range(ps[0][3], ps[0][3] + len(ps))), "pieces in k order belong to consecutive CTAs"


def test_decode_attention_plan_fits_every_kernel(lib):
    """zl_decode_attention_plan is the launch decision of zl_decode_attention.  Both kernels size their shared memory for a
    fixed number of keys per CTA and trust the host to keep round16(ceil(len_buf / splits)) within it: 256 for the
    warp-per-32-keys kernel, 1024 for k_decode_attn.  The splits must also cover the context and fit the workspace that
    zl_decode_attention_workspace_bytes reports."""
    d = 128
    heads = [(8, 8), (32, 8), (40, 8), (28, 4), (64, 8), (48, 4), (32, 2)]      # m_query 1, 4, 5, 7, 8, 12, 16
    lens = [1, 15, 16, 17, 255, 256, 257, 1023, 1024, 1025, 16384, 16385, 65536, 70000, 131072]
    max_keys = {0: 1024, 1: 256}
    for b in range(1, 65):
        for len_q in (1, 3, 64, 128):
            for hq, hkv in heads:
                for max_len in lens:
                    kernel, splits = attention_plan(lib, b, len_q, hq, hkv, max_len)
                    case = (b, len_q, hq, hkv, max_len, kernel, splits)
                    assert kernel in max_keys and splits >= 1, case
                    chunk = (-(-max_len // splits) + 15) // 16 * 16
                    assert chunk <= max_keys[kernel], case
                    assert splits * chunk >= max_len, case
                    if splits > 1:
                        need = b * len_q * hq * splits * (d + 2) * 4
                        assert lib.zl_decode_attention_workspace_bytes(b, len_q, hq, d, max_len) >= need, case


@pytest.mark.parametrize("b,len_q,max_len,splits", [
    (1, 128, 128, 1), (1, 128, 256, 1),              # 8B prefill, chunk 128: both chunks of a 256-token prompt
    (32, 1, 2048, 2),                                # batch 32 decode at context 2048
    (8, 1, 8192, 8),                                 # batch 8, context 8192
    (1, 1, 20000, 37), (1, 1, 70000, 69),            # batch 1, long context (more splits than a short context allows)
    (32, 1, 513, 2), (32, 1, 4096, 4)])              # batch 32 decode past 512 tokens
def test_decode_attention_plan_of_benchmarked_shapes(lib, b, len_q, max_len, splits):
    """The shapes the project reports numbers for (Llama-3.1-8B heads, 32 / 8) run on k_decode_attn (kernel 0)."""
    assert attention_plan(lib, b, len_q, 32, 8, max_len) == (0, splits)
    bad = ctypes.c_int()
    assert lib.zl_decode_attention_plan(b, len_q, 32, 7, max_len, ctypes.byref(bad), ctypes.byref(bad)) == -1
