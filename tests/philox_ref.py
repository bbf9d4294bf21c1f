"""Vectorised numpy Philox4x32-10 and the keep-mask / Box-Muller draws of hvae_fill_noise (csrc/optim.cu), as a reference
for the device generator.  Counter {ctr_lo, ctr_hi, stream_id, 0}, key {seed_lo, seed_hi}."""
import numpy as np

M0, M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
W0, W1 = 0x9E3779B9, 0xBB67AE85
_LO = np.uint64(0xFFFFFFFF)
_32 = np.uint64(32)


def philox4x32(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 of counter words c0..c3 (arrays or scalars, broadcast) under key (k0, k1): four uint32 arrays."""
    c0, c1, c2, c3 = np.broadcast_arrays(*[np.asarray(c, dtype=np.uint64) & _LO for c in (c0, c1, c2, c3)])
    k0, k1 = int(k0) & 0xFFFFFFFF, int(k1) & 0xFFFFFFFF
    for _ in range(10):
        p0, p1 = M0 * c0, M1 * c2
        c0, c1, c2, c3 = (p1 >> _32) ^ c1 ^ np.uint64(k0), p1 & _LO, (p0 >> _32) ^ c3 ^ np.uint64(k1), p0 & _LO
        k0, k1 = (k0 + W0) & 0xFFFFFFFF, (k1 + W1) & 0xFFFFFFFF
    return [c.astype(np.uint32) for c in (c0, c1, c2, c3)]


def draws(n, seed, base, stream_id):
    """The n uint32 words hvae_fill_noise consumes: word 4i+k = output k of counter base + i (64-bit, wrapping)."""
    n4 = (n + 3) // 4
    ctr = (np.uint64(base & 0xFFFFFFFFFFFFFFFF) + np.arange(n4, dtype=np.uint64))       # wraps mod 2^64 as the kernel does
    r = philox4x32(ctr & _LO, ctr >> _32, stream_id & 0xFFFFFFFF, 0, seed & 0xFFFFFFFF, seed >> 32)
    return np.stack(r, axis=1).reshape(-1)[:n]


def keep_mask(n, keep, seed, base, stream_id):
    """uint8 mask: (r >> 8) * 2^-24 < keep, all in float32 (exact: r >> 8 < 2^24)."""
    r = draws(n, seed, base, stream_id)
    return ((r >> 8).astype(np.float32) * np.float32(2.0 ** -24) < np.float32(keep)).astype(np.uint8)


def normal_uniforms(n, seed, base, stream_id):
    """(u1, u2) of every Box-Muller pair the eps draw uses (stream id + 2^31), float32 values held in float64:
    u1 = ((r0 >> 8) + 1) * 2^-24 in (0, 1], u2 = (r1 >> 8) * 2^-24 in [0, 1)."""
    r = draws(2 * ((n + 1) // 2), seed, base, stream_id + 0x80000000).reshape(-1, 2)
    u1 = ((r[:, 0] >> 8).astype(np.float64) + 1.0) * 2.0 ** -24
    u2 = (r[:, 1] >> 8).astype(np.float64) * 2.0 ** -24
    return u1, u2


def normals64(n, seed, base, stream_id):
    """Box-Muller eps evaluated in float64 on the generator's uniforms: (eps [n], radius of each value [n])."""
    u1, u2 = normal_uniforms(n, seed, base, stream_id)
    rad = np.sqrt(-2.0 * np.log(u1))
    eps = np.stack([rad * np.cos(2.0 * np.pi * u2), rad * np.sin(2.0 * np.pi * u2)], axis=1).reshape(-1)[:n]
    return eps, np.repeat(rad, 2)[:n]
