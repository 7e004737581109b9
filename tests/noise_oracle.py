"""CPU restatement of the keyed sampling noise (csrc/noise.cu, engine.keyed_normal): Philox4x32-10 in exact uint32 arithmetic
(numpy, vectorised over counters) and Box-Muller in float64 on the fp32 uniforms the kernel forms."""
import numpy as np

M0, M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
W0, W1 = 0x9E3779B9, 0xBB67AE85
MASK = np.uint64(0xFFFFFFFF)


def philox4x32_10(ctr, key):
    """ctr uint32 [..., 4], key uint32 [..., 2] (broadcast) -> uint32 [..., 4]."""
    c = [np.asarray(ctr, dtype=np.uint64)[..., j] for j in range(4)]
    k0 = np.asarray(key, dtype=np.uint64)[..., 0]
    k1 = np.asarray(key, dtype=np.uint64)[..., 1]
    for r in range(10):
        if r:
            k0 = (k0 + np.uint64(W0)) & MASK
            k1 = (k1 + np.uint64(W1)) & MASK
        p0, p1 = M0 * c[0], M1 * c[2]                  # < 2^64: exact in uint64
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & MASK, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & MASK]
    return np.stack(c, -1).astype(np.uint32)


def uniform01(w):
    """u = ((w >> 8) + 0.5) 2^-24 with the kernel's fp32 rounding (exact below 2^23, one correctly rounded addition above), in
    (0, 1]: the largest word rounds to u = 1."""
    return (((np.asarray(w, dtype=np.uint32) >> np.uint32(8)).astype(np.float32) + np.float32(0.5)) * np.float32(2.0 ** -24)).astype(np.float32)


def counters(keys, draw, slices, L):
    """uint32 [S, NB, L, 4] counters of slices `slices` for member keys `keys` (int64 [NB])."""
    k = np.asarray(keys, dtype=np.int64).astype(np.uint64)
    s = np.asarray(slices, dtype=np.uint64)
    i = np.arange(L, dtype=np.uint64)
    S, NB = s.size, k.size
    ctr = np.empty((S, NB, L, 4), dtype=np.uint64)
    ctr[..., 0] = (k & MASK)[None, :, None]
    ctr[..., 1] = (k >> np.uint64(32))[None, :, None]
    ctr[..., 2] = np.uint64(draw)
    ctr[..., 3] = ((s << np.uint64(21))[:, None, None] | i[None, None, :]) & MASK
    return ctr.astype(np.uint32)


def keyed_normal(seed, keys, L, draw, first_slice, n_slices):
    """float64 [n_slices, NB, L, 3]: what engine.keyed_normal computes, with float64 Box-Muller."""
    seed = int(seed)
    key = np.array([seed & 0xFFFFFFFF, seed >> 32], dtype=np.uint32)
    w = philox4x32_10(counters(keys, draw, np.arange(first_slice, first_slice + n_slices), L), key)
    u = uniform01(w).astype(np.float64)
    r01 = np.sqrt(-2.0 * np.log(u[..., 0]))
    r23 = np.sqrt(-2.0 * np.log(u[..., 2]))
    return np.stack([r01 * np.cos(2 * np.pi * u[..., 1]), r01 * np.sin(2 * np.pi * u[..., 1]), r23 * np.cos(2 * np.pi * u[..., 3])], -1)
