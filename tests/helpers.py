"""Shared test helpers (numpy restatement of OUR ZLW4 tile layout + small utilities)."""
import numpy as np

from oracle import golden_cases, gptq

BLK = 2128


def km_shift(kk):
    return (kk >> 1) * 4 + (kk & 1) * 16


def phys_k(t, j, r, e):
    u = j * 4 + r * 2 + e
    return (u >> 3) * 32 + t * 8 + (u & 7)


def w4_pack_numpy(qw_km, qz_km, sc_km, sym=False, row_map=None):
    """Reference implementation of the ZLW4 packer (zhilight_b200/csrc/w4_layout.cuh) in numpy."""
    q = gptq.unpack_k_major(qw_km)                     # (Nsrc, K) natural k
    z = np.asarray(qz_km)
    s = np.asarray(sc_km, dtype=np.float16)
    if row_map is not None:
        q, z, s = q[row_map], z[row_map], s[row_map]
    n, k = q.shape
    g = k // 128
    out = np.zeros((n // 32, g, BLK), dtype=np.uint8)
    words = np.zeros((n // 32, g, 512), dtype=np.uint32)
    for tt in range(2):
        for hh in range(2):
            for lane in range(32):
                gg, t = lane >> 2, lane & 3
                for jj in range(4):
                    j = hh * 4 + jj
                    idx = ((tt * 2 + hh) * 32 + lane) * 4 + jj
                    w = np.zeros((n // 32, g), dtype=np.uint32)
                    for slot in range(8):
                        row = tt * 16 + gg + (8 if (slot >> 1) & 1 else 0)
                        kk = phys_k(t, j, slot >> 2, slot & 1)
                        vals = q.reshape(n // 32, 32, g, 128)[:, row, :, kk].astype(np.uint32)
                        w |= vals << np.uint32(km_shift(slot))
                    words[:, :, idx] = w
    out[:, :, :2048] = words.view(np.uint8).reshape(n // 32, g, 2048)
    sr = s.reshape(n // 32, 2, 2, 8, g)                # [st, tt, up, g8, G]
    zr = (np.full_like(z, 8) if sym else z).reshape(n // 32, 2, 2, 8, g)
    sc2 = np.stack([sr[:, :, 0], sr[:, :, 1]], axis=-1)            # [st, tt, g8, G, 2]
    sc2 = np.transpose(sc2, (0, 3, 1, 2, 4)).copy()                # [st, G, tt, g8, 2]
    out[:, :, 2048:2112] = sc2.view(np.uint8).reshape(n // 32, g, 64)
    zb = (zr[:, :, 0] & 15) | ((zr[:, :, 1] & 15) << 4)            # [st, tt, g8, G]
    out[:, :, 2112:2128] = np.transpose(zb, (0, 3, 1, 2)).reshape(n // 32, g, 16).astype(np.uint8)
    return out.reshape(-1)


def attention_plan(lib, b, len_q, hq, hkv, max_len):
    """(kernel, splits) that zl_decode_attention launches for this shape: kernel 0 = k_decode_attn, 1 = warp kernel"""
    import ctypes
    kernel, splits = ctypes.c_int(-1), ctypes.c_int(-1)
    assert lib.zl_decode_attention_plan(b, len_q, hq, hkv, max_len, ctypes.byref(kernel), ctypes.byref(splits)) == 0
    return kernel.value, splits.value


def rel_l2(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def tensor_digest(t):
    """golden_cases.digest of a torch tensor (bf16 hashed as its 16-bit patterns)."""
    import torch
    t = t.detach().contiguous().cpu()
    if t.dtype == torch.bfloat16:
        t = t.view(torch.int16)
    return golden_cases.digest(t.numpy())


def sample_index(size, n):
    """A fixed, seeded choice of n of `size` flat indices (all of them when n >= size)."""
    if n >= size:
        return np.arange(size)
    return np.sort(np.random.RandomState(0).choice(size, n, replace=False))


def to_bf16_bits(x):
    u = np.asarray(x, dtype=np.float32).view(np.uint32).astype(np.uint64)
    r = ((u >> 16) & 1) + 0x7FFF
    return ((u + r) >> 16).astype(np.uint16)


def from_bf16_bits(b):
    return (np.asarray(b, dtype=np.uint16).astype(np.uint32) << 16).view(np.float32)


def w4i_pack_numpy(qw_km, qz_km, sc_km, sym=False, row_map=None):
    """numpy restatement of the ZLW4I (integer-kernel) nibble order; meta identical to ZLW4."""
    base = w4_pack_numpy(qw_km, qz_km, sc_km, sym, row_map).reshape(-1, BLK).copy()
    q = gptq.unpack_k_major(qw_km)
    if row_map is not None:
        q = q[row_map]
    n, k = q.shape
    g = k // 128
    qr = q.reshape(n // 32, 32, g, 128)
    words = np.zeros((n // 32, g, 512), dtype=np.uint32)
    for tt in range(2):
        for hh in range(2):
            for lane in range(32):
                gg, t = lane >> 2, lane & 3
                for jj in range(4):
                    wi = hh * 4 + jj
                    j, p = wi >> 1, wi & 1
                    idx = ((tt * 2 + hh) * 32 + lane) * 4 + jj
                    w = np.zeros((n // 32, g), dtype=np.uint32)
                    for slot in range(8):
                        row = tt * 16 + gg + (8 if slot & 1 else 0)
                        kk = t * 32 + j * 8 + p * 4 + (slot >> 1)
                        w |= qr[:, row, :, kk].astype(np.uint32) << np.uint32(4 * slot)
                    words[:, :, idx] = w
    base = base.reshape(n // 32, g, BLK)
    base[:, :, :2048] = words.view(np.uint8).reshape(n // 32, g, 2048)
    return base.reshape(-1)
