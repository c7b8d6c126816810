"""Masked language-model batches in plain Python (no torch, no transformers): the rule of Engine.mlm_mask and of
akshar_mlm_mask (include/akshar_b200.h), which is transformers' DataCollatorForLanguageModeling(mlm=True)
`torch_mask_tokens` with its draws taken from Philox4x32-10 keyed by (seed, epoch, row, position) instead of the
collator's serial CPU generator.

1. Draws: one Philox4x32-10 block per position, key (seed mod 2^32, seed >> 32), counter (j, R mod 2^32, R >> 32, epoch)
   with R = row_base + n the row and j the position: (u_select, u_mask, u_random, r_id).
2. Thresholds t(q) = min(2^32, ceil(fl32(q) 2^32)), fl32 the rounding to float32: t1 = t(p), t2 = t(m),
   t3 = t(r / (1 - m)) (0 when m = 1 or r = 0).
3. selected = not special and u_select < t1; replaced = selected and u_mask < t2; random = selected, not replaced and
   u_random < t3.  labels = the id where selected, else -100; ids: mask_id where replaced, r_id V >> 32 where random.
`philox` works on Python ints, `philox_np` on numpy uint32 arrays (for large batches); both give the same words.
"""
import struct

import numpy as np

M0, M1, W0, W1 = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85
MASK32 = 0xFFFFFFFF


def philox(ctr, key):
    """Philox4x32-10 of counter ctr (4 words) under key (2 words) -> 4 words"""
    c0, c1, c2, c3 = ctr
    k0, k1 = key
    for _ in range(10):
        p0, p1 = M0 * c0, M1 * c2
        c0, c1, c2, c3 = (p1 >> 32) ^ c1 ^ k0, p1 & MASK32, (p0 >> 32) ^ c3 ^ k1, p0 & MASK32
        k0, k1 = (k0 + W0) & MASK32, (k1 + W1) & MASK32
    return c0, c1, c2, c3


def philox_np(c0, c1, c2, c3, k0, k1):
    """the same over arrays: c0..c3 uint32 arrays (broadcast), k0 / k1 ints -> 4 uint32 arrays"""
    c0, c1, c2, c3 = (np.asarray(c, np.uint64) for c in (c0, c1, c2, c3))
    c0, c1, c2, c3 = np.broadcast_arrays(c0, c1, c2, c3)
    k0, k1 = int(k0), int(k1)
    m32 = np.uint64(MASK32)
    s32 = np.uint64(32)
    for _ in range(10):
        p0, p1 = c0 * np.uint64(M0), c2 * np.uint64(M1)
        c0, c1, c2, c3 = (p1 >> s32) ^ c1 ^ np.uint64(k0), p1 & m32, (p0 >> s32) ^ c3 ^ np.uint64(k1), p0 & m32
        k0, k1 = (k0 + W0) & MASK32, (k1 + W1) & MASK32
    return tuple(c.astype(np.uint32) for c in (c0, c1, c2, c3))


def fl32(q):
    return struct.unpack('<f', struct.pack('<f', q))[0]


def threshold(q):
    """draw iff u < t: bernoulli(fl32(q)) of a u / 2^32 draw"""
    x = fl32(q) * 2 ** 32
    return min(2 ** 32, int(x) + (x != int(x)))


def thresholds(p, m, r):
    return threshold(p), threshold(m), 0 if m == 1 or r == 0 else threshold(r / (1 - m))


def draws(n_rows, width, seed, epoch, row_base):
    """the four words of every position of an [n_rows, width] batch, each a uint32 [n_rows, width] array"""
    R = (row_base + np.arange(n_rows, dtype=object)).astype(object)
    lo = np.array([int(x) & MASK32 for x in R], np.uint64).reshape(-1, 1)
    hi = np.array([int(x) >> 32 for x in R], np.uint64).reshape(-1, 1)
    j = np.arange(width, dtype=np.uint64).reshape(1, -1)
    return philox_np(j, lo, hi, np.uint64(epoch), seed & MASK32, seed >> 32)


def mask(input_ids, special_ids, V, mask_id, seed, p=0.15, m=0.8, r=0.1, epoch=0, row_base=0, pad_id=None):
    """-> (new input_ids, labels, counts (selected, replaced, random)) for an int64 [N, L] array; input_ids is not changed.
    Worked in blocks of rows, so that large batches need little memory"""
    ids = np.asarray(input_ids, np.int64)
    N, L = ids.shape
    t = [np.uint64(x) for x in thresholds(p, m, r)]
    specials = np.asarray(sorted(set(special_ids) | ({pad_id} if pad_id is not None else set())), np.int64)
    out, labels = ids.copy(), np.full_like(ids, -100)
    counts = np.zeros(3, np.int64)
    step = max(1, (1 << 20) // max(L, 1))
    for a in range(0, N, step):
        x = ids[a:a + step]
        u0, u1, u2, u3 = (w.astype(np.uint64) for w in draws(x.shape[0], L, seed, epoch, row_base + a))
        selected = ~np.isin(x, specials) & (u0 < t[0])
        replaced = selected & (u1 < t[1])
        rand = selected & ~replaced & (u2 < t[2])
        labels[a:a + step][selected] = x[selected]
        out[a:a + step][replaced] = mask_id
        out[a:a + step][rand] = ((u3[rand] * np.uint64(V)) >> np.uint64(32)).astype(np.int64)
        counts += (selected.sum(), replaced.sum(), rand.sum())
    return out, labels, tuple(int(c) for c in counts)
