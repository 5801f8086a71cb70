"""TEST INFRASTRUCTURE: a plain numpy reference of the in-kernel sampling noise (include/phk.h, phk_sample_tokens with
u == NULL, phk_head_sample, phk_sample_tail), written from the Random123 definition of Philox4x32, independent of the
CUDA sources.

Layout of the library:  key = (seed lo, seed hi), counter = (c lo, c hi, 0, 0),
    c = offset + row * ceil(V / 4) + v // 4   (mod 2^64),   entry v takes output word v % 4.
The head uses its token row; the masked-rows tail uses the compact row `sequence * k + j`, not the position.
Uniform: u = (2 * (w >> 9) + 1) / 2^24 (exact);  gumbel: -log(-log(u)) in float64."""
import numpy as np

M0, M1 = 0xD2511F53, 0xCD9E8D57          # Philox4x32 round multipliers
W0, W1 = 0x9E3779B9, 0xBB67AE85          # Weyl key increments
ROUNDS = 7                               # the library's round count
MASK32 = np.uint64(0xFFFFFFFF)
K_COUNT = 1 << 23                        # distinct uniforms: k = w >> 9


def philox4x32(ctr, key, rounds=ROUNDS):
    """ctr: uint32-valued array [..., 4]; key: (k0, k1).  Returns the four output words, uint32 [..., 4]."""
    c = np.asarray(ctr, dtype=np.uint64)
    c0, c1, c2, c3 = (c[..., i].copy() for i in range(4))
    k0, k1 = int(key[0]) & 0xFFFFFFFF, int(key[1]) & 0xFFFFFFFF
    for _ in range(rounds):
        p0 = np.uint64(M0) * c0
        p1 = np.uint64(M1) * c2
        n0 = (p1 >> np.uint64(32)) ^ c1 ^ np.uint64(k0)
        n2 = (p0 >> np.uint64(32)) ^ c3 ^ np.uint64(k1)
        c0, c1, c2, c3 = n0, p1 & MASK32, n2, p0 & MASK32
        k0, k1 = (k0 + W0) & 0xFFFFFFFF, (k1 + W1) & 0xFFFFFFFF
    return np.stack([c0, c1, c2, c3], axis=-1).astype(np.uint32)


def counter_bits(seed, ctr):
    """The four words of the 64-bit counters `ctr` (uint64 array) under the library's key of `seed`: uint32 [..., 4]."""
    ctr = np.asarray(ctr, dtype=np.uint64)
    c = np.stack([ctr & MASK32, ctr >> np.uint64(32), np.zeros_like(ctr), np.zeros_like(ctr)], axis=-1)
    s = int(seed) & (2 ** 64 - 1)
    return philox4x32(c, (s & 0xFFFFFFFF, s >> 32))


def stream_bits(seed, offset, n):
    """Word i % 4 of counter offset + i // 4, i < n (what phk_noise_probe returns with bits_in == NULL)."""
    q = (n + 3) // 4
    ctr = np.uint64(int(offset) & (2 ** 64 - 1)) + np.arange(q, dtype=np.uint64)   # wraps mod 2^64 like the kernels
    return counter_bits(seed, ctr).reshape(-1)[:n]


def row_bits(seed, offset, rows, V):
    """uint32 [len(rows), V]: the noise word of entry v of each token row (rows: array of row indices)."""
    per = (V + 3) // 4
    rows = np.asarray(rows, dtype=np.uint64)
    ctr = (np.uint64(int(offset) & (2 ** 64 - 1)) + rows[:, None] * np.uint64(per)
           + np.arange(per, dtype=np.uint64)[None, :])
    return counter_bits(seed, ctr).reshape(len(rows), per * 4)[:, :V]


def uniform(bits):
    return (2.0 * (np.asarray(bits, dtype=np.uint32) >> 9).astype(np.float64) + 1.0) / 2.0 ** 24


def gumbel64(bits):
    """-log(-log(u)) in float64.  -log(u) is taken as -log1p(-w) with the exact complement w = 1 - u, so that the
    values near u = 1 (the largest gumbels) are correct to float64 precision."""
    u = uniform(bits)
    return -np.log(-np.log1p(-(1.0 - u)))


def gumbel64_table():
    """float64 gumbel of every k = w >> 9 (2^23 entries)."""
    return gumbel64(np.arange(K_COUNT, dtype=np.uint32) << 9)


def scores(logits, temperature, g):
    return np.asarray(logits, dtype=np.float64) / max(float(temperature), 1e-10) + g


def ideal(logits, temperature, bits):
    """argmax(l / max(T, 1e-10) + gumbel64), lowest index on ties: the reference's gumbel_sample
    (phenaki_pytorch.py:83-93) on these uniforms."""
    return np.argmax(scores(logits, temperature, gumbel64(bits)), axis=-1)


def with_table(logits, temperature, bits, table):
    """The same decision with a supplied per-k gumbel table (table[w >> 9], e.g. the device's transform)."""
    g = np.asarray(table, dtype=np.float64)[np.asarray(bits, dtype=np.uint32) >> 9]
    return np.argmax(scores(logits, temperature, g), axis=-1)


def top2_gap(s):
    """Best score minus the second best, per row (inf for a single column)."""
    if s.shape[-1] == 1:
        return np.full(s.shape[:-1], np.inf)
    part = np.partition(s, -2, axis=-1)
    return part[..., -1] - part[..., -2]


def softmax64(logits):
    l = np.asarray(logits, dtype=np.float64)
    e = np.exp(l - l.max(axis=-1, keepdims=True))
    return e / e.sum(axis=-1, keepdims=True)
