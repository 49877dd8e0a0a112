"""GPU parity of k_decode_attn (decode_attn.cu: S = K.Q^T and P.V on the tensor cores, split-KV + LSE combine) and of the
int8-KV kernel (decode_attn_kv8.cu) against a float64 evaluation of the same attention.

k_decode_attn serves every shape with more work than the warp-per-32-keys kernel takes: prefill chunks, batch decode past
a few hundred tokens, long contexts.  Each case first asks zl_decode_attention_plan which kernel its shape selects, so a
later change of the thresholds fails here instead of silently testing the other kernel.  Tolerances are those of
test_attention_gpu.py, over the whole output and, at 4x, over every (task, query, head) row: a misplaced head, split or
V column cannot hide in the global norm."""
import numpy as np
import pytest
import torch

from tests.helpers import attention_plan, rel_l2

pytestmark = pytest.mark.gpu

TOL = {torch.float16: 1e-3, torch.bfloat16: 6e-3}
DTYPES = [pytest.param(torch.float16, id="f16"), pytest.param(torch.bfloat16, id="bf16")]
KERNEL_TC = 0


def attention_f64(q, ks, vs, lens, masks, scale):
    """float64 restatement of the kernels' contract (oracle.ops.decode_attention): logit = mask ? scale q.k : -inf,
    max seeded -1e20, sum seeded 1e-20, out = sum_k p v.  q (B, len_q, H_q, d); ks / vs per task (len_b, H_kv, d);
    masks per task (len_q, len_b) or None.  Vectorised over the queries and heads of each kv head."""
    q = np.asarray(q, np.float64)
    b, len_q, hq, d = q.shape
    out = np.zeros_like(q)
    for bi, lb in enumerate(lens):
        hkv = ks[bi].shape[1]
        m_query = hq // hkv
        valid = np.ones((len_q, lb), bool) if masks is None or masks[bi] is None else np.asarray(masks[bi]) != 0
        for hk in range(hkv):
            k = np.asarray(ks[bi][:lb, hk], np.float64)                     # (lb, d)
            v = np.asarray(vs[bi][:lb, hk], np.float64)
            qh = q[bi, :, hk * m_query:(hk + 1) * m_query]                  # (len_q, m, d)
            logit = np.einsum("qmd,kd->qmk", qh, k) * scale
            logit = np.where(valid[:, None, :], logit, -np.inf)
            mx = np.maximum(logit.max(axis=-1, keepdims=True), -1e20)
            e = np.exp(logit - mx)
            p = e / (e.sum(axis=-1, keepdims=True) + 1e-20)
            out[bi, :, hk * m_query:(hk + 1) * m_query] = np.einsum("qmk,kd->qmd", p, v)
    return out


def check(out, ref, dtype, tol=None):
    """global and per-(task, query, head) relative L2 of the kernel output against the float64 result rounded to dtype"""
    tol = tol or TOL[dtype]
    out = out.float().cpu().numpy().astype(np.float64)
    ref = torch.from_numpy(ref).to(dtype).double().numpy()
    assert np.isfinite(out).all()
    assert rel_l2(out, ref) <= tol
    rows = np.linalg.norm(out - ref, axis=-1) / np.maximum(np.linalg.norm(ref, axis=-1), 1e-30)
    worst = np.unravel_index(np.argmax(rows), rows.shape)
    assert rows[worst] <= 4 * tol, ("(task, query, head)", worst, float(rows[worst]))


def causal_masks(len_q, pos0):
    """query i of a prefill chunk starting at position pos0 sees keys <= pos0 + i"""
    return [(np.arange(pos0 + len_q)[None, :] <= pos0 + np.arange(len_q)[:, None]).astype(np.int8)]


def holey_masks(lens, len_q, g):
    """padding past the tokens and beam-tree style holes (as test_attention_gpu.py); every row keeps key 0"""
    masks = []
    for lb in lens:
        m = (torch.rand(len_q, lb, generator=g) > 0.15).to(torch.int8)
        m[:, lb - min(3, lb - 1):] = 0
        m[:, 0] = 1
        masks.append(m.numpy())
    return masks


class Case:
    """q / K / V drawn on the GPU from a seeded generator (long contexts are 10^8 elements); masks on the host."""

    def __init__(self, cuda, dtype, b_lens, hq, hkv, d, len_q=1, seed=0, bshd=True, masks=None, q_scale=1.0, v_scale=1.0):
        g = torch.Generator(device=cuda).manual_seed(seed)
        self.lens, self.hq, self.hkv, self.d, self.len_q, self.bshd, self.masks = b_lens, hq, hkv, d, len_q, bshd, masks
        self.q = (q_scale * torch.randn(len(b_lens), len_q, hq, d, generator=g, device=cuda)).to(dtype)
        shape = (lambda lb: (lb, hkv, d)) if bshd else (lambda lb: (hkv, lb, d))
        self.k = [torch.randn(*shape(lb), generator=g, device=cuda).to(dtype) for lb in b_lens]
        self.v = [(v_scale * torch.randn(*shape(lb), generator=g, device=cuda)).clamp(-3e4, 3e4).to(dtype)
                  for lb in b_lens]
        self.scale = 1.0 / np.sqrt(d)

    def run(self):
        from zhilight_b200 import ops
        cuda = self.q.device
        mask = None
        if self.masks is not None:
            mask = torch.from_numpy(np.concatenate([m.reshape(-1) for m in self.masks])).to(cuda)
        return ops.decode_attention(self.q, torch.tensor(self.lens, dtype=torch.int32, device=cuda), self.k, self.v, mask,
                                    self.scale, max(self.lens), self.hkv, bshd=self.bshd)

    def reference(self):
        host = lambda t: (t if self.bshd else t.permute(1, 0, 2)).float().cpu().numpy()    # exact; float64 per head
        return attention_f64(self.q.double().cpu().numpy(), [host(k) for k in self.k], [host(v) for v in self.v],
                             self.lens, self.masks, self.scale)

    def assert_plan(self, lib, splits=None):
        kernel, s = attention_plan(lib, len(self.lens), self.len_q, self.hq, self.hkv, max(self.lens))
        assert kernel == KERNEL_TC, "shape no longer selects k_decode_attn"
        if splits is not None:
            assert s == splits
        return s


def ragged_lens(b, longest, seed):
    """one task at `longest`, the rest spread over lengths where splits come out empty or partial"""
    edge = [1, 15, 16, 17, 255, 1023, 1024, 1025, 31, 33, 513, 1500]
    rng = np.random.default_rng(seed)
    rest = [edge[i] if i < len(edge) else int(rng.integers(1, longest + 1)) for i in range(b - 1)]
    return [longest] + [min(x, longest) for x in rest]


# ------------------------------------------------------------------------------------------- fp16 / bf16 cache


@pytest.mark.parametrize("dtype", DTYPES)
def test_batch_decode_ragged(lib, cuda, dtype):
    """B = 32 decode on Llama-3.1-8B heads, one task at 2048 keys (2 splits): tasks of 1..1025 keys leave the second split
    empty (k0 >= len_buf) or partial; random mask holes.  Two identical calls are bitwise equal."""
    lens = ragged_lens(32, 2048, 0)
    c = Case(cuda, dtype, lens, 32, 8, 128, seed=1, masks=holey_masks(lens, 1, torch.Generator().manual_seed(1)))
    c.assert_plan(lib, splits=2)
    out = c.run()
    check(out, c.reference(), dtype)
    assert torch.equal(out, c.run())


@pytest.mark.parametrize("dtype", DTYPES)
def test_head_dim_64(lib, cuda, dtype):
    """Llama-3.2-1B heads (32 / 8, d = 64), B = 16 at up to 1500 keys"""
    lens = ragged_lens(16, 1500, 2)
    c = Case(cuda, dtype, lens, 32, 8, 64, seed=2, masks=holey_masks(lens, 1, torch.Generator().manual_seed(2)))
    c.assert_plan(lib)
    check(c.run(), c.reference(), dtype)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("hq,hkv,b", [(8, 8, 16), (40, 8, 16), (28, 4, 32), (48, 4, 16), (32, 2, 32)],
                         ids=["mq1", "mq5", "mq7", "mq12", "mq16"])
def test_gqa_ratios(lib, cuda, dtype, hq, hkv, b):
    """m_query 1, 5, 7 (partial 8-head groups), 12 (a second head group of 4) and 16 (two full groups)"""
    lens = ragged_lens(b, 1500, 3)
    c = Case(cuda, dtype, lens, hq, hkv, 128, seed=3, masks=holey_masks(lens, 1, torch.Generator().manual_seed(3)))
    c.assert_plan(lib)
    check(c.run(), c.reference(), dtype)


@pytest.mark.parametrize("dtype", DTYPES)
def test_hsd_layout(lib, cuda, dtype):
    """(H_kv, len_buf, d) buffers (bshd = 0)"""
    lens = ragged_lens(16, 1500, 4)
    c = Case(cuda, dtype, lens, 32, 8, 128, seed=4, bshd=False,
             masks=holey_masks(lens, 1, torch.Generator().manual_seed(4)))
    c.assert_plan(lib)
    check(c.run(), c.reference(), dtype)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("b,length,splits", [(1, 20000, 37), (1, 70000, 69), (8, 8192, 8)])
def test_long_context(lib, cuda, dtype, b, length, splits):
    """batch 1 at 20000 and 70000 keys (more splits than kAttnMaxSplits = 64), batch 8 at 8192 keys; no mask"""
    c = Case(cuda, dtype, [length] * b, 32, 8, 128, seed=5)
    c.assert_plan(lib, splits=splits)
    check(c.run(), c.reference(), dtype)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("pos0,splits", [(0, 1), (1172, 2)])
def test_prefill_chunk_causal(lib, cuda, dtype, pos0, splits):
    """a 128-token prefill chunk of Llama-3.1-8B (B = 1, len_q = 128, 32 / 8 heads): query i sees keys <= pos0 + i, so
    every query row reads its own mask row"""
    c = Case(cuda, dtype, [pos0 + 128], 32, 8, 128, len_q=128, seed=6, masks=causal_masks(128, pos0))
    c.assert_plan(lib, splits=splits)
    check(c.run(), c.reference(), dtype)


@pytest.mark.parametrize("dtype", DTYPES)
def test_zero_query_averages_v(lib, cuda, dtype):
    """q = 0: every unmasked key has the same weight, the output is the mean of the unmasked V rows"""
    lens = ragged_lens(32, 2048, 7)
    masks = holey_masks(lens, 1, torch.Generator().manual_seed(7))
    c = Case(cuda, dtype, lens, 32, 8, 128, seed=7, masks=masks)
    c.q.zero_()
    c.assert_plan(lib)
    mean = np.stack([(v.double().cpu().numpy()[m[0] != 0]).mean(axis=0) for v, m in zip(c.v, masks)])  # (B, H_kv, d)
    ref = np.repeat(mean, 4, axis=1)[:, None]                                   # m_query = 4
    check(c.run(), ref, dtype)


@pytest.mark.parametrize("dtype", DTYPES)
def test_fully_masked_row_in_batch(lib, cuda, dtype):
    """one task whose mask row is all zeros: its output is zero, and no other task's output changes by a bit"""
    lens = ragged_lens(32, 2048, 8)
    masks = holey_masks(lens, 1, torch.Generator().manual_seed(8))
    c = Case(cuda, dtype, lens, 32, 8, 128, seed=8, masks=masks)
    c.assert_plan(lib)
    before = c.run()
    dead = 5                                    # 255 keys
    masks[dead][:] = 0
    out = c.run()
    assert torch.isfinite(out).all()
    assert out[dead].abs().max().item() == 0.0
    keep = [i for i in range(len(lens)) if i != dead]
    assert torch.equal(out[keep], before[keep])
    check(out, c.reference(), dtype)


def test_large_v_fp16(lib, cuda):
    """fp16 V up to |v| = 3e4 (near the fp16 limit): the P.V product stays finite and accurate"""
    lens = ragged_lens(32, 2048, 9)
    c = Case(cuda, torch.float16, lens, 32, 8, 128, seed=9, v_scale=1e4,
             masks=holey_masks(lens, 1, torch.Generator().manual_seed(9)))
    c.assert_plan(lib)
    assert max(v.abs().max().item() for v in c.v) == 3e4
    check(c.run(), c.reference(), torch.float16)


@pytest.mark.parametrize("dtype", DTYPES)
def test_sharp_logits(lib, cuda, dtype):
    """q scaled so that the logits have a standard deviation of about 10: a few keys carry nearly all the weight"""
    lens = ragged_lens(32, 2048, 10)
    c = Case(cuda, dtype, lens, 32, 8, 128, seed=10, q_scale=10.0,
             masks=holey_masks(lens, 1, torch.Generator().manual_seed(10)))
    c.assert_plan(lib)
    check(c.run(), c.reference(), dtype)


# ------------------------------------------------------------------------------------------- int8 KV cache


def kv8_run(cuda, lens, hq, hkv, d, out_dtype=torch.float16, len_q=1, masks=None, seed=0, sv_range=(0.005, 0.025)):
    """random uint8 codes and per-(token, kv head) scales; the reference is the float64 attention over the dequantised
    cache (code - 128) * scale"""
    from zhilight_b200 import ops
    g = torch.Generator(device=cuda).manual_seed(seed)
    b = len(lens)
    q = torch.randn(b, len_q, hq, d, generator=g, device=cuda).half()
    kq = [torch.randint(0, 256, (lb, hkv, d), generator=g, device=cuda, dtype=torch.uint8) for lb in lens]
    vq = [torch.randint(0, 256, (lb, hkv, d), generator=g, device=cuda, dtype=torch.uint8) for lb in lens]
    sk = [0.002 + 0.004 * torch.rand(lb, hkv, generator=g, device=cuda) for lb in lens]
    lo, hi = sv_range
    sv = [lo + (hi - lo) * torch.rand(lb, hkv, generator=g, device=cuda) for lb in lens]
    mask = None
    if masks is not None:
        mask = torch.from_numpy(np.concatenate([m.reshape(-1) for m in masks])).to(cuda)
    scale = 1.0 / np.sqrt(d)
    out = ops.decode_attention_kv8(q, torch.tensor(lens, dtype=torch.int32, device=cuda), kq, vq, sk, sv, mask, scale,
                                   max(lens), hkv, out_dtype=out_dtype)
    deq = lambda c, s: ((c.double() - 128) * s.double()[:, :, None]).float().cpu().numpy()   # exact in fp32
    ref = attention_f64(q.double().cpu().numpy(), [deq(a, s) for a, s in zip(kq, sk)],
                        [deq(a, s) for a, s in zip(vq, sv)], lens, masks, scale)
    return out, ref


@pytest.mark.parametrize("out_dtype", DTYPES)
def test_kv8_head_dim_64(lib, cuda, out_dtype):
    lens = [1600, 600, 2100]
    out, ref = kv8_run(cuda, lens, 32, 8, 64, out_dtype, masks=holey_masks(lens, 1, torch.Generator().manual_seed(11)),
                       seed=11)
    check(out, ref, out_dtype)


@pytest.mark.parametrize("hq,hkv", [(64, 8), (32, 2)], ids=["mq8", "mq16"])
def test_kv8_gqa_groups(lib, cuda, hq, hkv):
    lens = [1600, 600, 2100]
    out, ref = kv8_run(cuda, lens, hq, hkv, 128, torch.bfloat16,
                       masks=holey_masks(lens, 1, torch.Generator().manual_seed(12)), seed=12)
    check(out, ref, torch.bfloat16)


def test_kv8_prefill_rows_causal(lib, cuda):
    """len_q = 16 query rows, each with its own causal mask row"""
    out, ref = kv8_run(cuda, [1516], 32, 8, 128, len_q=16, masks=causal_masks(16, 1500), seed=13)
    check(out, ref, torch.float16)


@pytest.mark.parametrize("out_dtype", DTYPES)
def test_kv8_ragged_empty_splits(lib, cuda, out_dtype):
    """tasks of 1..1025 keys beside one of 2048 (8 splits): most of their splits are empty; mask holes"""
    lens = [2048, 1, 15, 16, 17, 255, 1025]
    out, ref = kv8_run(cuda, lens, 8, 2, 128, out_dtype, masks=holey_masks(lens, 1, torch.Generator().manual_seed(14)),
                       seed=14)
    check(out, ref, out_dtype)


@pytest.mark.parametrize("out_dtype", DTYPES)
def test_kv8_large_v_scale(lib, cuda, out_dtype):
    """V rows with |v| up to ~2e4 (scales ~157): the weight of the key with the largest logit is its V scale, which
    must not overflow fp16 on its way into the tensor cores"""
    lens = [2048, 1500]
    out, ref = kv8_run(cuda, lens, 32, 8, 128, out_dtype, masks=holey_masks(lens, 1, torch.Generator().manual_seed(15)),
                       seed=15, sv_range=(100.0, 160.0))
    check(out, ref, out_dtype)


def test_kv8_small_v_scale(lib, cuda):
    """V scales ~4e-8 (|v| ~ 5e-6, bf16 output): the weights are scaled up to fp16 normal numbers before the tensor cores"""
    lens = [2048, 1500]
    out, ref = kv8_run(cuda, lens, 32, 8, 128, torch.bfloat16, masks=holey_masks(lens, 1, torch.Generator().manual_seed(16)),
                       seed=16, sv_range=(2e-8, 6e-8))
    check(out, ref, torch.bfloat16)


def test_kv8_beyond_64_splits(lib, cuda):
    """70000 keys need 69 splits of at most 1024 keys"""
    out, ref = kv8_run(cuda, [70000], 32, 8, 128, seed=17)
    check(out, ref, torch.float16)
