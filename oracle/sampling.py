"""numpy restatement of the sampling pick (zl_sample, zhilight_b200/csrc/sample.cu) and of its random draw.

Per task, on one fp32 logits row, following the reference:
  penalties (generator/beam_util.cu:198-220) on the seen tokens, in fp32 like the kernel;
  random iff top_p < 1 or top_k > 0 (generator/batch_generator.h:106), else argmax (ties -> lowest index);
  p = softmax(l / T) (functions/softmax.cu:10-30: max-subtracted, sum seeded with 1e-20) in float64 over the fp32 l / T;
  cum = inclusive cumsum of p sorted descending, stable (ties in ascending index order, as cub's radix sort);
  P = min(top_p, cum[top_k-1]) if top_k > 0 else top_p; v = u * P * cum[V-1]; the first sorted position with cum >= v
  (generator/random_util.cu:83-106).
u comes from Philox4x32-10 (Random123 philox4x32_10) with key = seed, counter = {draw_index, 0, 0, 0}:
  u = ((w0 >> 8) + 1) * 2^-24.
"""
import numpy as np

_M0, _M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_W0, _W1 = np.uint32(0x9E3779B9), np.uint32(0xBB67AE85)
_MASK = np.uint64(0xFFFFFFFF)


def philox4x32_10(ctr, key):
    """ctr (..., 4) uint32, key (..., 2) uint32 -> (..., 4) uint32."""
    c = np.array(ctr, dtype=np.uint32)
    k = np.array(key, dtype=np.uint32)
    c0, c1, c2, c3 = (c[..., i].astype(np.uint64) for i in range(4))
    k0, k1 = k[..., 0].astype(np.uint32), k[..., 1].astype(np.uint32)
    with np.errstate(over="ignore"):
        for _ in range(10):
            p0 = _M0 * c0
            p1 = _M1 * c2
            hi0, lo0 = p0 >> np.uint64(32), p0 & _MASK
            hi1, lo1 = p1 >> np.uint64(32), p1 & _MASK
            c0, c1, c2, c3 = hi1 ^ c1 ^ k0.astype(np.uint64), lo1, hi0 ^ c3 ^ k1.astype(np.uint64), lo0
            k0 = k0 + _W0
            k1 = k1 + _W1
    return np.stack([c0, c1, c2, c3], axis=-1).astype(np.uint32)


def uniform(seed, draw_index):
    """u in (0, 1] for (seed, draw_index) (scalars or broadcastable arrays), as float32."""
    seed = np.asarray(seed, dtype=np.uint64)
    draw = np.asarray(draw_index, dtype=np.uint64)
    seed, draw = np.broadcast_arrays(seed, draw)
    ctr = np.zeros(seed.shape + (4,), dtype=np.uint32)
    ctr[..., 0] = (draw & _MASK).astype(np.uint32)
    key = np.stack([(seed & _MASK).astype(np.uint32), (seed >> np.uint64(32)).astype(np.uint32)], axis=-1)
    w0 = philox4x32_10(ctr, key)[..., 0]
    return (((w0 >> np.uint32(8)).astype(np.float64) + 1.0) * 2.0 ** -24).astype(np.float32)


def penalise(logits, seen, repetition_penalty=1.0, presence_penalty=0.0):
    """fp32 penalised copy of one row; seen: iterable of token ids (or a bool mask)."""
    l = np.array(logits, dtype=np.float32, copy=True)
    idx = np.flatnonzero(seen) if np.asarray(seen).dtype == bool else np.unique(np.asarray(list(seen), dtype=np.int64))
    if idx.size == 0:
        return l
    s = l[idx]
    if presence_penalty != 0:
        s = s - np.float32(presence_penalty)
    else:
        rep = np.float32(repetition_penalty)
        s = np.where(s < 0, s * rep, s / rep).astype(np.float32)
    l[idx] = s
    return l


def is_random(top_p=1.0, top_k=0):
    return top_p < 1 or top_k > 0


def sorted_cum(l, temperature):
    """(order, cum) of one penalised fp32 row: stable descending order of the fp32 l / T and the inclusive cumulative
    probabilities (float64) in that order."""
    x = (np.asarray(l, dtype=np.float32) / np.float32(temperature)).astype(np.float32)
    order = np.argsort(-x.astype(np.float64), kind="stable")
    xd = x.astype(np.float64)
    e = np.exp(xd - xd.max())
    p = e / (np.sum(e) + 1e-20)
    return order, np.cumsum(p[order])


def target(cum, u, top_p=1.0, top_k=0):
    P = min(float(top_p), float(cum[top_k - 1])) if top_k > 0 else float(top_p)
    return float(u) * P * float(cum[-1])


def pick(logits, seen=(), u=1.0, temperature=1.0, top_p=1.0, top_k=0, repetition_penalty=1.0, presence_penalty=0.0):
    """The token the contract picks for one row with draw u."""
    l = penalise(logits, seen, repetition_penalty, presence_penalty)
    if not is_random(top_p, top_k):
        return int(np.argmax(l))          # first maximum: ties -> lowest index
    order, cum = sorted_cum(l, temperature)
    v = target(cum, u, top_p, top_k)
    j = int(np.searchsorted(cum, v, side="left"))
    return int(order[min(j, len(order) - 1)])


def pick_window(logits, seen=(), u=1.0, temperature=1.0, top_p=1.0, top_k=0, repetition_penalty=1.0,
                presence_penalty=0.0, rel=1e-6):
    """Every token acceptable for this draw when v may be off by `rel` of cum[V-1]: the exact pick plus its sorted
    neighbours whose cumulative boundary lies within that distance of v.  -> (set of tokens, near_boundary flag)."""
    l = penalise(logits, seen, repetition_penalty, presence_penalty)
    if not is_random(top_p, top_k):
        return {int(np.argmax(l))}, False
    order, cum = sorted_cum(l, temperature)
    v = target(cum, u, top_p, top_k)
    tol = rel * float(cum[-1])
    lo = int(np.searchsorted(cum, v - tol, side="left"))
    hi = int(np.searchsorted(cum, v + tol, side="left"))
    n = len(order)
    toks = {int(order[min(j, n - 1)]) for j in range(lo, hi + 1)}
    return toks, hi > lo


def truncated_distribution(logits, temperature=1.0, top_p=1.0, top_k=0):
    """Exact probability of each token under the selection rule with u uniform on (0, 1] (no penalties)."""
    order, cum = sorted_cum(np.asarray(logits, dtype=np.float32), temperature)
    vmax = target(cum, 1.0, top_p, top_k)
    prev = np.concatenate([[0.0], cum[:-1]])
    # position j is picked for v in (prev_j, cum_j] intersected with (0, vmax]
    w = np.clip(np.minimum(cum, vmax) - prev, 0.0, None)
    if vmax <= 0:
        w = np.zeros_like(cum)
        w[0] = 1.0
    probs = np.zeros(len(order))
    probs[order] = w / w.sum()
    return probs
