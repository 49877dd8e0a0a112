"""zl_sample (seeded top-k / top-p sampling with penalties) against the numpy contract in oracle/sampling.py, and the
decode driver's sampling state (zl_llama_set_sampling / clear_sampling)."""
import itertools

import numpy as np
import pytest

from oracle import model as omodel
from oracle import sampling as S

pytestmark = pytest.mark.gpu

TINY = dict(num_layers=2, dim_model=256, num_heads=4, num_kv_heads=2, dim_head=64, dim_ff=512, vocab_size=512,
            eps=1e-5, rope_theta=10000.0, rope_llama3=None)


def _bits(seen_sets, v):
    words = (v + 31) // 32
    b = np.zeros((len(seen_sets), words), np.uint32)
    for t, ss in enumerate(seen_sets):
        for tok in ss:
            b[t, tok >> 5] |= np.uint32(1 << (tok & 31))
    return b.view(np.int32)


def _row(rng, v, kind):
    if kind == 1:      # long runs of equal logits
        return (np.round(rng.standard_normal(v) * 2) / 2).astype(np.float32)
    if kind == 2:      # -inf entries
        l = (rng.standard_normal(v) * 3).astype(np.float32)
        l[rng.random(v) < 0.3] = -np.inf
        return l
    if kind == 3:      # every logit equal
        return np.full(v, 0.25, np.float32)
    return (rng.standard_normal(v) * 3).astype(np.float32)


def _run_sample(cuda, logits, tasks, seen_sets, draws):
    import torch
    from zhilight_b200 import ops
    t, v = logits.shape
    lg = torch.from_numpy(logits).to(cuda)
    params = ops.sample_params(tasks, cuda, v)
    seen = torch.from_numpy(_bits(seen_sets, v)).to(cuda)
    cnt = torch.from_numpy(np.asarray(draws, np.int32)).to(cuda)
    out = ops.sample(lg, params, seen, cnt)
    torch.cuda.synchronize()
    return out.cpu().numpy(), seen.cpu().numpy().view(np.uint32), cnt.cpu().numpy()


@pytest.mark.parametrize("V", [512, 1000, 50257, 128256, 152064])
def test_sample_matches_oracle(lib, cuda, V):
    rng = np.random.default_rng(V)
    combos = list(itertools.product([1e-3, 0.7, 1.0, 100.0], [0, 1, 50, V - 1], [1e-6, 0.5, 0.9, 1.0],
                                    [(1.3, 0.0), (1.0, 0.8)]))
    tasks, seen_sets, draws, rows = [], [], [], []
    for i, (temp, k, p, (rep, pres)) in enumerate(combos):
        tasks.append(dict(temperature=temp, top_k=k, top_p=p, repetition_penalty=rep, presence_penalty=pres,
                          seed=int(rng.integers(0, 2 ** 62)) * 2 + i % 2))
        seen_sets.append(set(rng.integers(0, V, size=int(rng.integers(0, 64))).tolist()))
        draws.append(int(rng.integers(0, 1000)))
        rows.append(_row(rng, V, i % 4 if i % 8 != 7 else 3))
    logits = np.stack(rows)
    out, seen_after, cnt_after = _run_sample(cuda, logits, tasks, seen_sets, draws)
    near = 0
    for i, t in enumerate(tasks):
        u = S.uniform(t["seed"], draws[i])
        exact = S.pick(logits[i], seen_sets[i], u, **t_args(t))
        ok, is_near = S.pick_window(logits[i], seen_sets[i], u, **t_args(t))
        near += is_near
        if is_near:
            assert out[i] in ok, (i, t, out[i], ok)
        else:
            assert out[i] == exact, (i, t, out[i], exact)
        assert (seen_after[i, out[i] >> 5] >> (out[i] & 31)) & 1
        assert cnt_after[i] == draws[i] + 1
    # v within 1e-6 of cum[V-1] of a boundary: bounded, and the count is what the tolerance covers
    assert near <= len(tasks) // 4, near


def t_args(t):
    return dict(temperature=t["temperature"], top_p=t["top_p"], top_k=t["top_k"],
                repetition_penalty=t["repetition_penalty"], presence_penalty=t["presence_penalty"])


@pytest.mark.parametrize("V", [1000, 128256])
def test_greedy_equivalence_bitwise(lib, cuda, V):
    """top_k = 1 at temperature 1 and non-random penalised tasks pick exactly what zl_argmax picks on the penalised
    logits, ties included."""
    import torch
    from zhilight_b200 import ops
    rng = np.random.default_rng(1)
    rows, tasks, seen_sets = [], [], []
    for i in range(32):
        rows.append(_row(rng, V, i % 4))
        ss = set(rng.integers(0, V, size=40).tolist())
        if i % 2:
            ss.add(int(np.argmax(rows[-1])))   # penalise the raw argmax
        seen_sets.append(ss)
        pen = [(1.5, 0.0), (1.0, 2.0), (1.0, 0.0)][i % 3]
        if i % 4 == 0:
            tasks.append(dict(top_k=1, seed=i, repetition_penalty=pen[0], presence_penalty=pen[1]))
        else:
            tasks.append(dict(seed=i, repetition_penalty=pen[0], presence_penalty=pen[1]))
    logits = np.stack(rows)
    out, _, _ = _run_sample(cuda, logits, tasks, seen_sets, [0] * len(tasks))
    penalised = np.stack([S.penalise(logits[i], seen_sets[i], t["repetition_penalty"], t["presence_penalty"])
                          for i, t in enumerate(tasks)])
    ref = ops.argmax(torch.from_numpy(penalised).to(cuda)).cpu().numpy()
    np.testing.assert_array_equal(out, ref)


@pytest.mark.parametrize("temperature,top_k,top_p", [(1.0, 0, 0.9), (0.5, 5, 1.0), (2.0, 8, 0.7), (1.0, 15, 0.999)])
def test_distribution_chi_square(lib, cuda, temperature, top_k, top_p):
    from scipy import stats
    V, T, calls = 16, 50000, 4
    l = np.linspace(2.0, -1.5, V).astype(np.float32)[np.random.RandomState(0).permutation(V)]
    l[3] = l[5]                              # a tie
    expected = S.truncated_distribution(l, temperature, top_p, top_k)
    import torch
    from zhilight_b200 import ops
    lg = torch.from_numpy(np.tile(l, (T, 1))).to(cuda)
    tasks = [dict(temperature=temperature, top_k=top_k, top_p=top_p, seed=1000 + i) for i in range(T)]
    params = ops.sample_params(tasks, cuda, V)
    seen = torch.zeros((T, 1), dtype=torch.int32, device=cuda)
    cnt = torch.zeros(T, dtype=torch.int32, device=cuda)
    counts = np.zeros(V, np.int64)
    for _ in range(calls):
        seen.zero_()                         # no penalties: the seen set plays no part
        out = ops.sample(lg, params, seen, cnt).cpu().numpy()
        counts += np.bincount(out, minlength=V)
    n = T * calls
    assert counts[expected == 0].sum() == 0
    keep = expected > 0
    chi = stats.chisquare(counts[keep], expected[keep] * n)
    assert chi.pvalue > 1e-4, (chi, counts, expected * n)
    assert (cnt.cpu().numpy() == calls).all()


# ---------------------------------------------------------------------------------------------------- decode driver
SAMPLE1 = dict(temperature=0.8, top_p=0.9, top_k=50, repetition_penalty=1.2, presence_penalty=0.0, seed=2 ** 33 + 5)


def _decoder(use_graph=True, prefill_chunk=16, max_batch=3, **kw):
    from zhilight_b200.llama import LlamaDecoder
    sd = omodel.make_state_dict(TINY, 5, 128, False, seed=3)
    dec = LlamaDecoder(quant_type=5, max_batch=max_batch, max_seq=64, use_graph=use_graph, prefill_chunk=prefill_chunk,
                       **TINY, **kw)
    dec.load_state_dict(sd)
    return dec


def _check_pick(tok, logits_row, seen, params, draw):
    u = S.uniform(params["seed"], draw)
    args = {k: params[k] for k in ("temperature", "top_p", "top_k", "repetition_penalty", "presence_penalty")}
    ok, _ = S.pick_window(logits_row, seen, u, **args)
    assert tok in ok, (tok, ok, draw)


def test_driver_decode_samples_only_the_sampling_task(lib, cuda):
    rng = np.random.default_rng(0)
    toks = rng.integers(0, 512, size=(8, 3)).astype(np.int32)
    base = _decoder()
    greedy = [base.decode(toks[s], np.full(3, s, np.int32)) for s in range(8)]
    base.close()
    dec = _decoder()
    dec.set_sampling(1, **SAMPLE1)
    seen = set()
    for s in range(8):
        nxt, lg = dec.decode(toks[s], np.full(3, s, np.int32), want_logits=True)
        assert nxt[0] == greedy[s][0] and nxt[2] == greedy[s][2]
        _check_pick(int(nxt[1]), lg[1], seen, SAMPLE1, s)
        seen.add(int(nxt[1]))
    dec.close()


@pytest.mark.parametrize("use_graph", [True, False])
def test_driver_step_device_and_prefill(lib, cuda, use_graph):
    start = np.array([7, 300, 42], np.int32)
    base = _decoder(use_graph=use_graph)
    base.set_state(start, np.zeros(3, np.int32))
    greedy = []
    for _ in range(10):
        base.step_device(3)
        greedy.append(base.get_state(3)[0].copy())
    base.close()
    dec = _decoder(use_graph=use_graph)
    dec.set_sampling(1, **SAMPLE1)
    dec.set_state(start, np.zeros(3, np.int32))
    seen = set()
    for s in range(10):
        dec.step_device(3)
        lg = dec.logits(3)
        tok = dec.get_state(3)[0]
        assert tok[0] == greedy[s][0] and tok[2] == greedy[s][2]
        _check_pick(int(tok[1]), lg[1], seen, SAMPLE1, s)
        seen.add(int(tok[1]))
    # prefill of the sampling task: draw 10 continues the same stream and seen set
    prompt = np.arange(20, dtype=np.int32) * 7 % 512
    nxt, lg = dec.prefill(1, prompt, 0, want_logits=True)
    _check_pick(nxt, lg[0], seen, SAMPLE1, 10)
    dec.close()


def test_driver_reseed_presence_clear_and_graph_reuse(lib, cuda):
    start = np.array([11, 12, 13], np.int32)

    def run(dec, n):
        dec.set_state(start, np.zeros(3, np.int32))
        out = []
        for _ in range(n):
            dec.step_device(3)
            out.append(dec.get_state(3)[0].copy())
        return np.stack(out)

    base = _decoder()
    greedy = run(base, 20)
    base.close()
    dec = _decoder()
    p = dict(SAMPLE1, temperature=1.5, top_p=1.0, top_k=0, repetition_penalty=1.0)   # a wide distribution
    dec.set_sampling(1, **p)
    a = run(dec, 12)
    dec.set_sampling(1, **p)                  # re-seeding replays the same sequence
    np.testing.assert_array_equal(run(dec, 12), a)
    kps_sample = dec.stats(3)[1]
    dec.set_sampling(1, **dict(p, presence_penalty=1e4))
    r = run(dec, 20)[:, 1]
    assert len(set(r.tolist())) == 20, r      # a large presence penalty never repeats a token
    dec.clear_sampling(1)
    np.testing.assert_array_equal(run(dec, 20), greedy)
    kps_greedy = dec.stats(3)[1]              # the greedy graph was captured last
    assert kps_greedy == kps_sample + 1       # two argmax kernels against one zl_sample launch
    # new parameter values reuse the sampling graph: a new capture would report the sampling graph's kernel count
    q = dict(SAMPLE1, seed=99, top_k=5)
    dec.set_sampling(1, **q)
    dec.set_state(start, np.zeros(3, np.int32))
    seen = set()
    for s in range(6):
        dec.step_device(3)
        lg = dec.logits(3)
        tok = dec.get_state(3)[0]
        _check_pick(int(tok[1]), lg[1], seen, q, s)
        seen.add(int(tok[1]))
        assert dec.stats(3)[1] == kps_greedy
    dec.close()


def test_tensor_parallel_sampling_is_unsupported(lib, cuda):
    from zhilight_b200 import _lib
    from zhilight_b200.llama import LlamaDecoder
    dec = LlamaDecoder(quant_type=5, max_batch=2, max_seq=32, tp_rank=0, tp_size=2, **TINY)
    with pytest.raises(_lib.ZLError) as e:
        dec.set_sampling(0, top_p=0.9)
    assert e.value.code == -2
    dec.close()
