"""GPU parity against the REFERENCE's own kernels (its hot-path .cu files recompiled for sm_100 behind a thin shim,
oracle/_ref/libzl_ref.so) on identical inputs -- north_star: "outputs match the reference's own kernels on identical
inputs (bit-exact for GPTQ unpack/index, within 1e-3 rel for fp16)".

The reference's outputs on the seeded inputs built here are stored in tests/golden/vs_reference.npz
(oracle/gen_vs_reference_golden.py ran them on a B200): a bit-exact output as the digest of its bytes, a float output
as its values, or as a fixed seeded sample of them where the whole output is large.  Where a reference output fed
the next reference call, our own result is checked bit for bit against it and takes its place."""
import os

import numpy as np
import pytest
import torch

from oracle import gptq
from tests.helpers import rel_l2, sample_index, tensor_digest

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "vs_reference.npz")


class Stored:
    """The reference's outputs of one case as stored in GOLDEN."""

    def __init__(self, data, case):
        self.data, self.case = data, case

    def _get(self, key):
        return self.data[self.case + "/" + key]

    def assert_same(self, key, t):
        """bit for bit: shape, dtype and bytes"""
        assert tensor_digest(t) == str(self._get(key)), "%s/%s differs from the reference" % (self.case, key)

    def values(self, key):
        return self._get(key).astype(np.float32)

    def pick(self, key, a):
        """the elements of `a` (flattened) at the positions the stored values of `key` were taken from"""
        a = np.asarray(a, np.float32).reshape(-1)
        return a[sample_index(a.size, self._get(key).size)]


@pytest.fixture(scope="module")
def ref(cuda):
    with np.load(GOLDEN) as f:
        data = dict(f)
    return lambda case: Stored(data, case)


def to_dev(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


# ---- inputs (oracle/gen_vs_reference_golden.py feeds the same ones to the reference) ----
def ckpt_4096(sym):
    return gptq.make_gptq_checkpoint(4096, 4096, 128, sym, seed=0)


def awq_checkpoint():
    k, n, g = 1024, 512, 128
    rng = np.random.default_rng(1)
    qw = rng.integers(0, 2 ** 32, size=(k, n // 8), dtype=np.uint64).astype(np.uint32).view(np.int32)
    qz = rng.integers(0, 2 ** 32, size=(k // g, n // 8), dtype=np.uint64).astype(np.uint32).view(np.int32)
    sc = (0.01 * rng.random((k // g, n))).astype(np.float16)
    return qw, qz, sc


def gemv_x(m, dev):
    return torch.randn(m, 4096, generator=torch.Generator().manual_seed(0)).half().to(dev)


def swiglu_inputs(dev):
    k = 4096
    a = gptq.make_gptq_checkpoint(k, 1024, 128, False, seed=2)
    b = gptq.make_gptq_checkpoint(k, 1024, 128, False, seed=3)
    x = torch.randn(2, k, generator=torch.Generator().manual_seed(1)).half().to(dev)
    return a, b, x


def norm_rope_inputs(dtype, dev):
    g = torch.Generator().manual_seed(3)
    t, d = 7, 4096
    a = torch.randn(t, d, generator=g).to(dtype).to(dev)
    b = torch.randn(t, d, generator=g).to(dtype).to(dev)
    w = (1 + 0.1 * torch.randn(d, generator=g)).to(dtype).to(dev)
    hq, hkv, dh = 32, 8, 128
    qkv = torch.randn(t, (hq + 2 * hkv) * dh, generator=g).to(dtype).to(dev)
    pos = torch.tensor([0, 1, 2, 100, 1000, 5000, 8191], dtype=torch.int32, device=dev)
    return a, b, w, qkv, pos, (hq, hkv, dh)


def attention_inputs(lens, dev):
    hq, hkv, d = 16, 4, 128
    g = torch.Generator().manual_seed(4)
    b = len(lens)
    q = torch.randn(b, 1, hq, d, generator=g).half().to(dev)
    ks = [torch.randn(lb, hkv, d, generator=g).half().to(dev) for lb in lens]
    vs = [torch.randn(lb, hkv, d, generator=g).half().to(dev) for lb in lens]
    masks = []
    for lb in lens:
        m = torch.ones(lb, dtype=torch.int8)
        m[lb - 3:] = 0
        masks.append(m)
    mask = torch.cat(masks).to(dev)
    lens_t = torch.tensor(lens, dtype=torch.int32, device=dev)
    return q, ks, vs, mask, lens_t, hkv


def int8_linear_inputs(dt, dev):
    m, n, k = 7, 1536, 4096
    g = torch.Generator().manual_seed(3)
    x = (torch.randn(m, k, generator=g) * 1.3).to(dt).to(dev)
    w_q = torch.randint(-127, 128, (n, k), generator=g, dtype=torch.int8).to(dev)
    w_s = (0.0005 + 0.003 * torch.rand(n, generator=g)).to(dt).to(dev)
    return x, w_q, w_s


def rmsnorm_quant_inputs(dt, dev):
    t, d = 5, 4096
    g = torch.Generator().manual_seed(4)
    x = torch.randn(t, d, generator=g).to(dt).to(dev)
    w = (1 + 0.2 * torch.randn(d, generator=g)).to(dt).to(dev)
    return x, w


def fp8_inputs(dt, dev):
    m, n, k = 8, 2048, 4096
    g = torch.Generator().manual_seed(5)
    x = (torch.randn(m, k, generator=g) * 2).to(dt).to(dev)
    w8 = (torch.randn(n, k, generator=g) * 0.5).to(torch.float8_e4m3fn).view(torch.uint8).to(dev)
    sw = torch.tensor([0.01], dtype=torch.float32, device=dev)
    return x, w8, sw


ROPE_POS = [0, 1, 2, 63, 4095, 8191, 8192, 100000]


def sym_checkpoint(k, n, seed):
    rng = np.random.default_rng(seed)
    qw = rng.integers(0, 2 ** 32, size=(k // 8, n), dtype=np.uint64).astype(np.uint32).view(np.int32)
    sc = (0.002 + 0.004 * rng.random((k // 128, n))).astype(np.float16)
    qz = np.full((k // 128, n // 8), 0x77777777, dtype=np.uint32).view(np.int32)      # stored 7 -> zero 8 (u4b8)
    return qw, qz, sc


def marlin_x(m, k, dev):
    return torch.randn(m, k, generator=torch.Generator().manual_seed(m)).half().to(dev)


def awq_native_inputs(m, dev):
    k, n, g = 2048, 1024, 128
    rng = np.random.default_rng(3)
    qw = rng.integers(0, 2 ** 32, size=(k, n // 8), dtype=np.uint64).astype(np.uint32).view(np.int32)
    qz = rng.integers(0, 2 ** 32, size=(k // g, n // 8), dtype=np.uint64).astype(np.uint32).view(np.int32)
    sc = (0.002 + 0.004 * rng.random((k // g, n))).astype(np.float16)
    x = torch.randn(m, k, generator=torch.Generator().manual_seed(7)).half().to(dev)
    return qw, qz, sc, x


def kv_append_inputs(dev):
    hkv, d, t = 2, 128, 7
    g = torch.Generator().manual_seed(3)
    k = (torch.randn(t, hkv, d, generator=g) * 2).half().to(dev)
    v = torch.randn(t, hkv, d, generator=g).half().to(dev)
    return k, v


def kv8_case(dev, lens, hq, hkv, d, seed):
    g = torch.Generator().manual_seed(seed)
    b = len(lens)
    q = torch.randn(b, 1, hq, d, generator=g).half().to(dev)
    ks = [torch.randn(lb, hkv, d, generator=g).half().to(dev) for lb in lens]
    vs = [torch.randn(lb, hkv, d, generator=g).half().to(dev) for lb in lens]
    masks = []
    for lb in lens:
        m = torch.ones(lb, dtype=torch.int8)
        m[lb - 3:] = 0
        m[torch.randperm(lb - 3, generator=g)[: lb // 11]] = 0
        masks.append(m)
    return q, ks, vs, torch.cat(masks).to(dev), torch.tensor(lens, dtype=torch.int32, device=dev)


def kv8_shared_scale_inputs(lens, dev):
    """caches whose rows all share one absmax (4.0) per head -- see test_decode_attention_kv8_vs_reference_quant_kernel"""
    q, ks, vs, mask, lens_t = kv8_case(dev, lens, 8, 2, 128, 17)
    for t in ks + vs:                      # one common absmax per (row, head): identical scales along the buffer
        t.clamp_(-4.0, 4.0)
        t[:, :, 5] = 4.0
    return q, ks, vs, mask, lens_t


# ---- the tests ----
def test_load_pipeline_bit_exact_vs_reference(lib, ref, cuda):
    from zhilight_b200 import ops
    r = ref("layout_sym0")
    qw, qz, sc, gi = ckpt_4096(False)
    o_qw, o_qz, o_sc = ops.gptq_to_k_major(to_dev(qw, cuda), to_dev(qz, cuda), to_dev(sc, cuda))
    r.assert_same("qw_km", o_qw)
    r.assert_same("qz_km", o_qz)
    r.assert_same("sc_km", o_sc)
    r.assert_same("w16", ops.gptq_dequant_k_major(o_qw, o_qz, o_sc))


def test_awq_pipeline_bit_exact_vs_reference(lib, ref, cuda):
    from zhilight_b200 import ops
    r = ref("awq_layout")
    qw, qz, sc = awq_checkpoint()
    o = ops.gptq_to_k_major(to_dev(qw, cuda), to_dev(qz, cuda), to_dev(sc, cuda), is_awq=True)
    for key, b in zip(("qw_km", "qz_km", "sc_km"), o):
        r.assert_same(key, b)


@pytest.mark.parametrize("sym", [False, True])
@pytest.mark.parametrize("m", [1, 4, 16, 33])
def test_w4a16_vs_reference_gemv(lib, ref, cuda, sym, m):
    """BASELINE config 1 shape.  The reference accumulates 8 products in fp16, we accumulate in fp32: the two
    must agree to ~1e-3 (L2) and ours must be the closer one to the exact result."""
    from zhilight_b200 import ops
    k = n = 4096
    qw, qz, sc, gi = ckpt_4096(sym)
    r_qw, r_qz, r_sc = ops.gptq_to_k_major(to_dev(qw, cuda), to_dev(qz, cuda), to_dev(sc, cuda))
    lay = ref("layout_sym%d" % sym)              # the k-major weights the reference GEMV ran on
    lay.assert_same("qw_km", r_qw)
    lay.assert_same("qz_km", r_qz)
    lay.assert_same("sc_km", r_sc)
    x = gemv_x(m, cuda)
    r = ref("gemv_sym%d_m%d" % (sym, m))
    y_ref = r.values("y")
    packed = ops.w4_pack(r_qw, r_qz, r_sc, 128, sym)
    y = ops.w4a16_gemm(x, packed, n, k).float().cpu().numpy()
    o_qw, o_qz, o_sc, _ = gptq.to_k_major(qw, qz, sc, gi, 128)
    exact = gptq.gemm_f32(x.cpu().numpy(), gptq.dequant_k_major_f32(o_qw, o_qz, o_sc, sym))
    ys, exact_s = r.pick("y", y), r.pick("y", exact)
    assert rel_l2(ys, y_ref) <= 2e-3
    assert rel_l2(y, exact) <= 1e-3
    assert rel_l2(ys, exact_s) <= rel_l2(y_ref, exact_s) + 1e-4


def test_swiglu_vs_reference_fused_gate_in(lib, ref, cuda):
    from zhilight_b200 import ops
    k, f = 4096, 1024
    a, b, x = swiglu_inputs(cuda)
    r = ref("swiglu")
    ga = ops.gptq_to_k_major(*(to_dev(t, cuda) for t in a[:3]))
    ub = ops.gptq_to_k_major(*(to_dev(t, cuda) for t in b[:3]))
    for key, t in zip(("gate_qw_km", "gate_qz_km", "gate_sc_km", "up_qw_km", "up_qz_km", "up_sc_km"), ga + ub):
        r.assert_same(key, t)
    y_ref = r.values("y")
    fused = [torch.cat([p, q]).contiguous() for p, q in zip(ga, ub)]
    packed = ops.w4_pack(fused[0], fused[1], fused[2], 128, False, ops.swiglu_row_map(f, cuda))
    y = ops.w4a16_gemm(x, packed, 2 * f, k, epilogue=ops.EPI_SWIGLU).float().cpu().numpy()
    assert rel_l2(r.pick("y", y), y_ref) <= 4e-3


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
def test_norm_rope_vs_reference(lib, ref, cuda, dtype):
    from zhilight_b200 import ops
    a, b, w, qkv, pos, (hq, hkv, dh) = norm_rope_inputs(dtype, cuda)
    r = ref("norm_rope_%s" % str(dtype).split(".")[-1])
    ulp = 2 ** -10 if dtype == torch.float16 else 2 ** -7
    f32 = lambda t: t.float().cpu().numpy()
    np.testing.assert_allclose(r.pick("rmsnorm", f32(ops.rmsnorm(a, w, 1e-5))), r.values("rmsnorm"), rtol=ulp, atol=1e-6)
    s, y = ops.add_rmsnorm(a, b, w, 1e-5, mode=1)
    r.assert_same("fuse_add_s", s)
    np.testing.assert_allclose(r.pick("fuse_add_y", f32(y)), r.values("fuse_add_y"), rtol=ulp, atol=1e-6)
    r.assert_same("element_add", ops.element_add_scale(a, b, 1.0))
    cos, sin = ops.rope_cos_sin(pos, dh, 500000.0, dict(factor=8.0, low=1.0, high=4.0, orig=8192.0))
    r.assert_same("rope_cos", cos)                # the tables the reference's rope was given
    r.assert_same("rope_sin", sin)
    q, k, v = ops.rope_qk_cache(cos, sin, qkv, hq, hkv, dh)
    np.testing.assert_allclose(r.pick("rope_q", f32(q)), r.values("rope_q"), rtol=ulp, atol=1e-3)
    np.testing.assert_allclose(r.pick("rope_k", f32(k)), r.values("rope_k"), rtol=ulp, atol=1e-3)
    r.assert_same("rope_v", v)


@pytest.mark.parametrize("lens", [[4096, 123], [300, 1024, 77], [2048, 2048]])
def test_decode_attention_vs_reference(lib, ref, cuda, lens):
    """src/nn/tests/test_attention_rag_buffer.cpp shape: 4 kv-heads x m_query 4, lens {4096, 123}."""
    from zhilight_b200 import ops
    q, ks, vs, mask, lens_t, hkv = attention_inputs(lens, cuda)
    d = q.shape[-1]
    r = ref("attention_" + "_".join(map(str, lens)))
    out = ops.decode_attention(q, lens_t, ks, vs, mask, d ** -0.5, max(lens), hkv)
    assert rel_l2(r.pick("out", out.float().cpu().numpy()), r.values("out")) <= 1e-3


@pytest.mark.parametrize("dt", [torch.float16, torch.bfloat16])
def test_int8_linear_bit_exact_vs_reference_kernels(lib, ref, cuda, dt):
    """Int8Linear = quant_calc_scale -> s32 GEMM -> quant_scale_back (linear.cpp:560-636).  The s32 GEMM is exact
    integer arithmetic (torch int matmul stands in for cuBLASLt); both ends are the reference's own kernels."""
    from zhilight_b200 import ops
    x, w_q, w_s = int8_linear_inputs(dt, cuda)
    r = ref("int8_linear_%s" % str(dt).split(".")[-1])
    q, s = ops.int8_quant_per_token(x)
    r.assert_same("q", q)
    r.assert_same("s", s)
    y = ops.int8_linear(x, w_q, w_s)
    r.assert_same("y", y)             # quant_scale_back of the exact s32 product of q and w_q


@pytest.mark.parametrize("dt", [torch.float16, torch.bfloat16])
def test_rmsnorm_quant_vs_reference(lib, ref, cuda, dt):
    from zhilight_b200 import ops
    x, w = rmsnorm_quant_inputs(dt, cuda)
    r = ref("rmsnorm_quant_%s" % str(dt).split(".")[-1])
    y, q, s = ops.rmsnorm_quant(x, w, 1e-5)
    r.assert_same("q", q)
    np.testing.assert_allclose(r.pick("s", s.cpu().numpy()), r.values("s"), rtol=1e-6, atol=0)
    assert rel_l2(r.pick("y", y.float().cpu().numpy()), r.values("y")) < 1e-3


@pytest.mark.parametrize("dt", [torch.float16, torch.bfloat16])
def test_fp8_linear_vs_reference(lib, ref, cuda, dt):
    """dynamic_scaled_quant codes must be identical; the GEMM is cuBLASLt fp8 in the reference (fp32 accumulate,
    different summation order): <= 1e-3 rel."""
    from zhilight_b200 import ops
    x, w8, sw = fp8_inputs(dt, cuda)
    r = ref("fp8_linear_%s" % str(dt).split(".")[-1])
    q, s = ops.fp8_quant_per_tensor(x)
    r.assert_same("s", s)
    r.assert_same("q", q)
    y = ops.w8a8_gemm(q, s, w8, sw, dt, kind=ops.W8_FP8).float().cpu().numpy()
    assert rel_l2(r.pick("y", y), r.values("y")) < (1e-3 if dt == torch.float16 else 4e-3)


# ---- round 2: rope tables, Marlin, native AWQ against the reference's own kernels ----
LLAMA3_8 = dict(factor=8.0, low=1.0, high=4.0, orig=8192)
LLAMA3_32 = dict(factor=32.0, low=1.0, high=4.0, orig=8192)
ROPE_VARIANTS = [(10000.0, None), (500000.0, LLAMA3_8), (500000.0, LLAMA3_32)]
ROPE_IDS = ["plain", "llama3-f8", "llama3-f32"]


@pytest.mark.parametrize("d", [64, 128])
@pytest.mark.parametrize("theta,l3", ROPE_VARIANTS, ids=ROPE_IDS)
def test_rope_cos_sin_vs_reference_rope_preparer(lib, ref, cuda, d, theta, l3):
    """zl_rope_cos_sin against RopePreparer / KERNEL_rope_cos_sin(_llama3) (src/nn/position/rope_preparer.cu:49-161).
    Both evaluate the same fp32 expression, so the tables agree to the last bits even at position 100000 where a
    1-ulp change of inv_freq already moves cos by 1e-2: every llama3-rope model depends on this table."""
    from zhilight_b200 import ops
    pos = torch.tensor(ROPE_POS, dtype=torch.int32, device=cuda)
    r = ref("rope_tables_%s_d%d" % (ROPE_IDS[[v[1] for v in ROPE_VARIANTS].index(l3)], d))
    c_ref, s_ref = r.values("cos"), r.values("sin")
    c, s = ops.rope_cos_sin(pos, d, theta, l3)
    c, s = r.pick("cos", c.cpu().numpy()), r.pick("sin", s.cpu().numpy())
    np.testing.assert_allclose(c, c_ref, rtol=0, atol=2e-6)
    np.testing.assert_allclose(s, s_ref, rtol=0, atol=2e-6)
    assert float((c == c_ref).mean()) > 0.99 and float((s == s_ref).mean()) > 0.99


@pytest.mark.parametrize("m", [1, 16, 32, 64])
@pytest.mark.parametrize("k,n", [(4096, 4096), (4096, 14336)])
def test_quant_type_8_vs_reference_marlin_kernel(lib, ref, cuda, k, n, m):
    """QuantType 8 (GPTQ_Marlin): our kernels on a symmetric g128 checkpoint against the reference's gptq_marlin_gemm
    (src/nn/quant/marlin/gptq_marlin.cu:2034-2192) fed by gptq_marlin_repack + the scale permutation of
    GPTQMarlin::post_load (linear.cpp:1402-1428).  Marlin multiplies fp16 dequantised weights with fp32 accumulation;
    M <= 16 runs our exact-integer kernel, M > 16 the tcgen05 kernel: both within 1e-3 (L2) of it and of the fp32 oracle."""
    from zhilight_b200 import ops
    qw, qz, sc = sym_checkpoint(k, n, 5)
    x = marlin_x(m, k, cuda)
    r = ref("marlin_k%d_n%d_m%d" % (k, n, m))
    y_ref = r.values("y")
    o_qw, o_qz, o_sc = ops.gptq_to_k_major(to_dev(qw, cuda), to_dev(qz, cuda), to_dev(sc, cuda))
    packed = ops.w4_pack(o_qw, o_qz, o_sc, 128, True, variant=1)
    y = ops.w4a16_gemm_fused(x, packed, n, k, variant=1).float().cpu().numpy()
    k_qw, k_qz, k_sc, _ = gptq.to_k_major(qw, qz, sc, np.arange(k) // 128, 128)
    exact = gptq.gemm_f32(x.cpu().numpy(), gptq.dequant_k_major_f32(k_qw, k_qz, k_sc, True))
    assert rel_l2(r.pick("y", y), y_ref) <= 1e-3
    assert rel_l2(y, exact) <= 1e-3 and rel_l2(y_ref, r.pick("y", exact)) <= 1e-3


def test_marlin_repack_is_a_permutation_of_the_checkpoint(lib, ref, cuda):
    """gptq_marlin_repack (gptq_marlin_repack.cu:258-318) only permutes nibbles: same multiset per 16 x 64 tile."""
    k, n = 256, 128
    qw, _, _ = sym_checkpoint(k, n, 9)
    r = ref("marlin_repack")._get("repacked").view(np.uint32)
    assert r.shape == (k // 16, 2 * n)
    nib = lambda a: np.sort(np.stack([(a >> (4 * i)) & 15 for i in range(8)]).reshape(-1))
    np.testing.assert_array_equal(nib(r), nib(qw.view(np.uint32)))


@pytest.mark.parametrize("m", [1, 8, 32])
def test_awq_native_gemm_vs_ours(lib, ref, cuda, m):
    """QuantType 6 through the reference's native awq_gemm (src/nn/quant/awq/gemm_kernels.cu:404-468, split-k 32) against
    our AWQ path (shuffle_awq / un_shuffle into the k-major layout, then the W4A16 kernels): same w = (q - z) * s."""
    from zhilight_b200 import ops
    qw, qz, sc, x = awq_native_inputs(m, cuda)
    n = sc.shape[1]
    r = ref("awq_native_m%d" % m)
    o_qw, o_qz, o_sc = ops.gptq_to_k_major(to_dev(qw, cuda), to_dev(qz, cuda), to_dev(sc, cuda), is_awq=True)
    packed = ops.w4_pack(o_qw, o_qz, o_sc, 128, False, variant=1)
    y = ops.w4a16_gemm_fused(x, packed, n, x.shape[1], variant=1).float().cpu().numpy()
    # awq_gemm sums 32 fp16 partial tensors (KERNEL_sum_dim0): it is the noisier side
    assert rel_l2(r.pick("y", y), r.values("y")) <= 3e-3


# ---- int8 KV cache: quantising append and the split-KV quant attention kernel ----
def quantise_buffer(ops, k, v):
    """our cache-side quantisation of one task's whole K / V buffers: uint8 codes and fp32 scales per (row, head)"""
    lb, hkv, d = k.shape
    kq = torch.zeros(lb, hkv, d, dtype=torch.uint8, device=k.device)
    vq = torch.zeros_like(kq)
    sk = torch.zeros(lb, hkv, dtype=torch.float32, device=k.device)
    sv = torch.zeros_like(sk)
    ops.kv_int8_quant_append(k, v, torch.zeros(lb, dtype=torch.int32, device=k.device),
                             torch.arange(lb, dtype=torch.int32, device=k.device), [kq], [vq], [sk], [sv])
    return kq, vq, sk, sv


def test_kv_int8_quant_append_bit_exact_vs_reference(lib, ref, cuda):
    """codes and scales of our cache-side quantisation == int8_op::quant_calc_scale(x, 127, 128) (quant_kernel.cu:15-47)"""
    from zhilight_b200 import ops
    hkv, d, t = 2, 128, 7
    k, v = kv_append_inputs(cuda)
    r = ref("kv_append")
    tb = torch.tensor([0, 1, 0, 1, 0, 1, 0], dtype=torch.int32, device=cuda)
    pl = torch.tensor([0, 0, 1, 1, 2, 2, 3], dtype=torch.int32, device=cuda)
    kb = [torch.zeros(4, hkv, d, dtype=torch.uint8, device=cuda) for _ in range(2)]
    vb = [torch.zeros(4, hkv, d, dtype=torch.uint8, device=cuda) for _ in range(2)]
    sk = [torch.zeros(4, hkv, dtype=torch.float32, device=cuda) for _ in range(2)]
    sv = [torch.zeros(4, hkv, dtype=torch.float32, device=cuda) for _ in range(2)]
    ops.kv_int8_quant_append(k, v, tb, pl, kb, vb, sk, sv)
    tokens = [(int(tb[i]), int(pl[i])) for i in range(t)]     # the cache rows token by token, in token order
    for key, bufs in (("kq", kb), ("vq", vb), ("ks", sk), ("vs", sv)):
        r.assert_same(key, torch.stack([bufs[b_][p_] for b_, p_ in tokens]))


@pytest.mark.parametrize("lens", [[1600, 600], [2000], [1100, 1300, 40]])
def test_decode_attention_kv8_vs_reference_quant_kernel(lib, ref, cuda, lens):
    """zl_decode_attention_kv8 against KERNEL_mqa_rag_buffer_split_kv_quant (attention_kernel.cu:804-880) on the same uint8
    caches and scales (the reference only takes its quant kernel above 1024 keys, with < 1024 keys per split).

    The reference kernel offsets the K / V pointers of split s by s * len_split rows but NOT the scale pointers
    (attention_kernel.cu:847-851: scale_key = scale_key_addrs[b] + head_kv), i.e. every split after the first multiplies
    its logits and probabilities with the scales of the FIRST split's tokens.  Measured here on a B200: 0.2-0.4 relative
    error against the fp32 evaluation of the same cache.  The comparison therefore uses caches whose rows all share one
    scale per head (every row carries one element of magnitude 4.0), where that indexing is harmless; with per-row scales
    our kernel is checked against the fp32 evaluation (next test and the assertions on `exact` here).
    The reference multiplies q.k in fp16 (quant_attention.cuh:60-70): both within 2e-3, ours within 1e-3 of exact."""
    from zhilight_b200 import ops
    hq, hkv, d = 8, 2, 128
    q, ks, vs, mask, lens_t = kv8_shared_scale_inputs(lens, cuda)
    r = ref("kv8_attention_" + "_".join(map(str, lens)))
    kq, vq, sk, sv = [], [], [], []
    for i, (k, v) in enumerate(zip(ks, vs)):
        a, b, s, s2 = quantise_buffer(ops, k, v)
        for key, t in (("kq%d" % i, a), ("vq%d" % i, b), ("sk%d" % i, s), ("sv%d" % i, s2)):
            r.assert_same(key, t)              # the caches the reference kernel ran on
        kq.append(a)
        vq.append(b)
        sk.append(s)
        sv.append(s2)
    assert float(sk[0].max() - sk[0].min()) == 0.0
    scale = 1.0 / np.sqrt(d)
    y_ref = r.values("out")
    y = ops.decode_attention_kv8(q, lens_t, kq, vq, sk, sv, mask, scale, max(lens), hkv).float().cpu().numpy()
    # fp32 evaluation of the same quantised cache
    from oracle import ops as oops
    kd = [((a.float() - 128) * s[:, :, None]).cpu().numpy() for a, s in zip(kq, sk)]
    vd = [((a.float() - 128) * s[:, :, None]).cpu().numpy() for a, s in zip(vq, sv)]
    off = np.cumsum([0] + lens)
    masks = [mask[off[i]:off[i + 1]].cpu().numpy().reshape(1, -1) for i in range(len(lens))]
    exact = oops.decode_attention(q.cpu().numpy(), kd, vd, lens, masks, scale, hq // hkv, "f32")
    ys, exact_s = r.pick("out", y), r.pick("out", exact)
    assert rel_l2(y, exact) <= 1e-3
    assert rel_l2(ys, y_ref) <= 2e-3
    assert rel_l2(ys, exact_s) <= rel_l2(y_ref, exact_s) + 2e-4       # at least as close to the exact result as the reference


def test_decode_attention_kv8_per_row_scales_long_context(lib, cuda):
    """per-row scales (what a real cache holds) over split contexts: against the fp32 evaluation of the quantised cache"""
    from zhilight_b200 import ops
    from oracle import ops as oops
    hq, hkv, d = 8, 2, 128
    lens = [1600, 600, 2100]
    g = torch.Generator().manual_seed(23)
    q = torch.randn(3, 1, hq, d, generator=g).half().to(cuda)
    kq = [torch.randint(0, 256, (lb, hkv, d), generator=g, dtype=torch.uint8).to(cuda) for lb in lens]
    vq = [torch.randint(0, 256, (lb, hkv, d), generator=g, dtype=torch.uint8).to(cuda) for lb in lens]
    sk = [(0.002 + 0.004 * torch.rand(lb, hkv, generator=g)).to(cuda) for lb in lens]
    sv = [(0.005 + 0.02 * torch.rand(lb, hkv, generator=g)).to(cuda) for lb in lens]
    lens_t = torch.tensor(lens, dtype=torch.int32, device=cuda)
    mask = (torch.rand(sum(lens), generator=g) > 0.1).to(torch.int8).to(cuda)
    scale = 1.0 / np.sqrt(d)
    y = ops.decode_attention_kv8(q, lens_t, kq, vq, sk, sv, mask, scale, max(lens), hkv).float().cpu().numpy()
    kd = [((a.float() - 128) * s[:, :, None]).cpu().numpy() for a, s in zip(kq, sk)]
    vd = [((a.float() - 128) * s[:, :, None]).cpu().numpy() for a, s in zip(vq, sv)]
    off = np.cumsum([0] + lens)
    masks = [mask[off[i]:off[i + 1]].cpu().numpy().reshape(1, -1) for i in range(len(lens))]
    exact = oops.decode_attention(q.cpu().numpy(), kd, vd, lens, masks, scale, hq // hkv, "f32")
    assert rel_l2(y, exact) <= 1e-3


def test_decode_attention_kv8_short_context_and_gqa4(lib, cuda):
    """below the reference's split threshold (its quant kernel is never taken there) and with m_query = 4: against the fp32
    evaluation of the quantised cache"""
    from zhilight_b200 import ops
    from oracle import ops as oops
    hq, hkv, d = 8, 2, 128
    lens = [130, 17, 512]
    g = torch.Generator().manual_seed(5)
    q = torch.randn(3, 1, hq, d, generator=g).half().to(cuda)
    kq = [torch.randint(0, 256, (lb, hkv, d), generator=g, dtype=torch.uint8).to(cuda) for lb in lens]
    vq = [torch.randint(0, 256, (lb, hkv, d), generator=g, dtype=torch.uint8).to(cuda) for lb in lens]
    sk = [(0.01 + 0.01 * torch.rand(lb, hkv, generator=g)).to(cuda) for lb in lens]
    sv = [(0.01 + 0.01 * torch.rand(lb, hkv, generator=g)).to(cuda) for lb in lens]
    lens_t = torch.tensor(lens, dtype=torch.int32, device=cuda)
    mask = torch.ones(sum(lens), dtype=torch.int8, device=cuda)
    scale = 1.0 / np.sqrt(d)
    y = ops.decode_attention_kv8(q, lens_t, kq, vq, sk, sv, mask, scale, max(lens), hkv).float().cpu().numpy()
    kd = [((a.float() - 128) * s[:, :, None]).cpu().numpy() for a, s in zip(kq, sk)]
    vd = [((a.float() - 128) * s[:, :, None]).cpu().numpy() for a, s in zip(vq, sv)]
    masks = [np.ones((1, lb), np.int8) for lb in lens]
    exact = oops.decode_attention(q.cpu().numpy(), kd, vd, lens, masks, scale, hq // hkv, "f32")
    assert rel_l2(y, exact) <= 1e-3
