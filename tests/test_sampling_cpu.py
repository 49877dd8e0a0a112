"""Sampling contract without a GPU: the Philox draw (oracle and library), hand-worked picks, argument validation."""
import ctypes

import numpy as np
import pytest

from oracle import sampling as S
from zhilight_b200 import _lib


@pytest.fixture(scope="module")
def lib():
    return _lib.load()


def test_philox_known_answers():
    """Random123 philox4x32_10 known-answer vectors."""
    cases = [
        ([0, 0, 0, 0], [0, 0], [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]),
        ([0xffffffff] * 4, [0xffffffff] * 2, [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]),
        ([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344], [0xa4093822, 0x299f31d0],
         [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]),
    ]
    for ctr, key, want in cases:
        assert S.philox4x32_10(ctr, key).tolist() == want


def test_uniform_mapping():
    w0 = 0x6627e8d5
    assert S.uniform(0, 0) == np.float32(((w0 >> 8) + 1) * 2.0 ** -24)
    u = S.uniform(np.arange(1000, dtype=np.uint64), 3)
    assert (u > 0).all() and (u <= 1).all()


def test_library_uniform_matches_oracle(lib):
    seeds = [0, 1, 2, 12345, 2 ** 32 - 1, 2 ** 32, 2 ** 32 + 7, 0xDEADBEEFCAFEF00D, 2 ** 64 - 1]
    draws = [0, 1, 2, 17, 1000, 2 ** 31, 2 ** 32 - 1]
    for s in seeds:
        for d in draws:
            got = lib.zl_sample_uniform(s, d)
            assert np.float32(got) == S.uniform(s, d), (s, d)


def test_oracle_ties_keep_index_order():
    l = np.array([1.0, 3.0, 3.0, 3.0, 0.0], np.float32)
    order, cum = S.sorted_cum(l, 1.0)
    assert order.tolist() == [1, 2, 3, 0, 4]
    e = np.exp(np.array([0, 0, 0, -2, -3.0]))
    np.testing.assert_allclose(cum, np.cumsum(e) / e.sum())
    # v just above the first boundary picks the second of the tied tokens
    P = 0.999999
    assert S.pick(l, u=(cum[0] + 1e-9) / (P * cum[-1]), top_p=P) == 2
    assert S.pick(l, u=(cum[1] + 1e-9) / (P * cum[-1]), top_p=P) == 3
    assert S.pick(l, u=0.5 * cum[0] / (P * cum[-1]), top_p=P) == 1


def test_oracle_top_k_one_and_tiny_top_p_are_greedy():
    rng = np.random.RandomState(0)
    l = rng.randn(1000).astype(np.float32)
    for u in (1e-7, 0.3, 1.0):
        assert S.pick(l, u=u, top_k=1) == int(np.argmax(l))
        assert S.pick(l, u=u, top_p=1e-6) == int(np.argmax(l))
        assert S.pick(l, u=u, top_p=0.0) == int(np.argmax(l))


def test_oracle_top_k_truncates():
    l = np.array([5.0, 4.0, 3.0, 2.0], np.float32)
    probs = S.truncated_distribution(l, top_k=2)
    e = np.exp(np.array([0.0, -1.0]))
    np.testing.assert_allclose(probs, [e[0] / e.sum(), e[1] / e.sum(), 0, 0], rtol=1e-12)
    # u = 1 lands on the last kept token
    assert S.pick(l, u=1.0, top_k=2) == 1


def test_oracle_penalty_branches():
    l = np.array([2.0, -2.0, 1.0, 0.5], np.float32)
    # repetition: positive divided, negative multiplied
    np.testing.assert_array_equal(S.penalise(l, [0, 1], repetition_penalty=2.0), np.float32([1.0, -4.0, 1.0, 0.5]))
    # presence replaces the repetition branch entirely
    np.testing.assert_array_equal(S.penalise(l, [0, 1], repetition_penalty=2.0, presence_penalty=0.25),
                                  np.float32([1.75, -2.25, 1.0, 0.5]))
    # a penalised greedy task: token 0 drops below token 2
    assert S.pick(l, seen=[0], repetition_penalty=4.0) == 2
    assert S.pick(l, seen=[0], presence_penalty=1.5) == 2
    assert S.pick(l, seen=[0], presence_penalty=0.5) == 0


def test_oracle_temperature():
    l = np.array([1.0, 0.0], np.float32)
    p_hot = S.truncated_distribution(l, temperature=100.0)
    p_cold = S.truncated_distribution(l, temperature=1e-3)
    assert abs(p_hot[0] - 0.5) < 0.01 and p_cold[0] == 1.0


def test_sampling_argument_validation_without_gpu(lib):
    p = ctypes.c_void_p(16)
    # no rows / missing pointers are rejected before any CUDA call
    assert lib.zl_sample(p, 0, 1000, p, p, p, p, p, None, 0, 0, None) == -1
    assert lib.zl_sample(None, 1, 1000, p, p, p, p, p, None, 0, 0, None) == -1
    assert lib.zl_sample(p, 1, 1000, p, None, p, p, p, None, 0, 0, None) == -1
    # vocabularies beyond the shared-memory slices are unsupported
    assert lib.zl_sample(p, 1, 1 << 20, p, p, p, p, p, None, 0, 0, None) == -2
    assert lib.zl_sample_workspace_bytes(64, 128256) == 0
    # the driver entry points refuse a missing model
    sp = _lib.SampleParams(1.0, 0.9, 1.0, 0.0, 50, 1)
    assert lib.zl_llama_set_sampling(None, 0, ctypes.byref(sp)) == -1
    assert lib.zl_llama_clear_sampling(None, 0) == -1


def test_sample_params_validation():
    from zhilight_b200 import ops
    for bad in ({"temperature": 0.0}, {"top_p": 1.5}, {"top_p": -0.1}, {"top_k": -1}, {"top_k": 1000}):
        with pytest.raises(_lib.ZLError):
            ops.sample_params([bad], "cpu", 1000)
    t = ops.sample_params([{"top_p": 0.9, "top_k": 50, "seed": 2 ** 40 + 3}], "cpu", 1000)
    assert t.numel() == ctypes.sizeof(_lib.SampleParams) == 32


def test_header_prototypes_parse():
    protos = _lib.parse_header()
    assert protos["zl_sample_uniform"][0] == "float"
    assert [n for _, n in protos["zl_sample"][1]][:5] == ["logits", "T", "V", "row_task", "params"]
    assert "zl_llama_set_sampling" in protos and "zl_llama_clear_sampling" in protos
