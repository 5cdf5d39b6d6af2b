"""numpy restatement of the counter-based normals behind Corex.sample / sample_missing (lcx_normal_fill,
lowrank_kernels.cuh) -- test helper only.

Philox4x32-10 (Salmon, Moraes, Dror and Shaw, SC'11; Random123's round and key constants).  Normal j of stream
(seed, tag, row, draw) comes from the counter (j // 2, draw, row mod 2^32, row // 2^32 + 2^24 tag) under the key
(seed mod 2^32, seed // 2^32): two 53-bit uniforms in (0, 1], u1 from words 0/1 and u2 from words 2/3, then Box-Muller,
z_2t = sqrt(-2 ln u1) cospi(2 u2), z_2t+1 = sqrt(-2 ln u1) sinpi(2 u2).
"""
import numpy as np

_M0, _M1, _W0, _W1 = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85
_MASK = np.uint64(0xFFFFFFFF)


def philox4x32_10(ctr, key):
    """ctr (..., 4) and key (2,) of 32-bit values -> the (..., 4) output words as uint64 arrays."""
    ctr = np.asarray(ctr, dtype=np.uint64)
    c = [ctr[..., i] for i in range(4)]
    k0, k1 = np.uint64(int(key[0]) & 0xFFFFFFFF), np.uint64(int(key[1]) & 0xFFFFFFFF)
    for _ in range(10):
        p0 = np.uint64(_M0) * c[0]  # 32 x 32 bits: exact in uint64
        p1 = np.uint64(_M1) * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & _MASK, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & _MASK]
        k0 = (k0 + np.uint64(_W0)) & _MASK
        k1 = (k1 + np.uint64(_W1)) & _MASK
    return np.stack(c, axis=-1)


def stream_words(seed, tag, rows, draw, n_cols):
    """(len(rows), ceil(n_cols / 2), 4) Philox words behind normals 0..n_cols-1 of the streams (seed, tag, row, draw)."""
    rows = np.asarray(rows, dtype=np.uint64)
    t = np.arange((n_cols + 1) // 2, dtype=np.uint64)
    ctr = np.zeros((len(rows), len(t), 4), dtype=np.uint64)
    ctr[..., 0] = t[None, :]
    ctr[..., 1] = np.uint64(draw)
    ctr[..., 2] = (rows & _MASK)[:, None]
    ctr[..., 3] = (((rows >> np.uint64(32)) + np.uint64(tag << 24)) & _MASK)[:, None]
    seed = int(seed)
    return philox4x32_10(ctr, (seed & 0xFFFFFFFF, seed >> 32))


def uniform53(hi, lo):
    """((hi 2^21 + lo // 2^11) + 1) 2^-53: 53 bits, in (0, 1], exact."""
    v = ((hi << np.uint64(21)) | (lo >> np.uint64(11))) + np.uint64(1)
    return v.astype(np.float64) * 2.0 ** -53


def sincospi(x):
    """(sin(pi x), cos(pi x)) to about an ulp for x in [0, 2]: reduction by quarter turns is exact, so only |pi r| <= pi/4
    reaches np.sin / np.cos."""
    q = np.rint(2 * x)
    r = x - q / 2  # exact: x is a multiple of 2^-52, |r| <= 1/4
    s, c = np.sin(np.pi * r), np.cos(np.pi * r)
    q = q.astype(np.int64) % 4
    sin = np.select([q == 0, q == 1, q == 2], [s, c, -s], -c)
    cos = np.select([q == 0, q == 1, q == 2], [c, -s, -c], s)
    return sin, cos


def normals(seed, tag, rows, draw, n_cols):
    """(len(rows), n_cols) float64: normal j of stream (seed, tag, row, draw) for each row."""
    w = stream_words(seed, tag, rows, draw, n_cols)
    rad = np.sqrt(-2.0 * np.log(uniform53(w[..., 0], w[..., 1])))
    s, c = sincospi(2.0 * uniform53(w[..., 2], w[..., 3]))
    z = np.stack([rad * c, rad * s], axis=-1).reshape(len(rows), -1)
    return z[:, :n_cols]
