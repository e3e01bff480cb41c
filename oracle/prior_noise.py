"""Test infrastructure (like everything under oracle/): the seeded prior noise of ev_prior_noise in numpy.

Philox4x32-10 as Random123 defines it (philox.h: round function, multipliers and Weyl key increments), vectorised over uint64
arrays; Box-Muller in float64, rounded once to float32; and the splitmix64 stream synthesise_corpus derives per-utterance
seeds from.  Independent of the package: it shares no code with emojivoice_b200/batch.py or csrc/noise.cu.

For seed s the key is (s mod 2^32, s >> 32).  Feature f and frame group q = t >> 2 give (w0, w1, w2, w3) = Philox(counter =
(q, f, 0, 0), key); with u = (w0 + 0.5) 2^-32, v = w1 2^-32, r = sqrt(-2 ln u): z[f, 4q] = r cos(2 pi v), z[f, 4q+1] = r sin(2 pi v),
and (w2, w3) give frames 4q+2 and 4q+3 the same way."""
import numpy as np

M32 = np.uint64(0xFFFFFFFF)
M64 = (1 << 64) - 1
PHILOX_M = (np.uint64(0xD2511F53), np.uint64(0xCD9E8D57))
PHILOX_W = (np.uint64(0x9E3779B9), np.uint64(0xBB67AE85))


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 of broadcastable uint32-valued arrays -> (w0, w1, w2, w3) as uint64 arrays holding 32-bit values."""
    c0, c1, c2, c3, k0, k1 = (np.asarray(v, dtype=np.uint64) & M32 for v in (c0, c1, c2, c3, k0, k1))
    for r in range(10):
        p0 = PHILOX_M[0] * c0                  # < 2^64: a 32 x 32-bit product, exact in uint64
        p1 = PHILOX_M[1] * c2
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & M32, (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & M32
        k0 = (k0 + PHILOX_W[0]) & M32
        k1 = (k1 + PHILOX_W[1]) & M32
    return c0, c1, c2, c3


def box_muller(a, b):
    """Two uint32 words -> two N(0, 1) samples in float64: u = (a + 0.5) 2^-32 >= 2^-33, v = b 2^-32."""
    u = (np.asarray(a, dtype=np.float64) + 0.5) * 2.0 ** -32
    v = np.asarray(b, dtype=np.float64) * 2.0 ** -32
    r = np.sqrt(-2.0 * np.log(u))
    return r * np.cos(2.0 * np.pi * v), r * np.sin(2.0 * np.pi * v)


def seed_key(seed):
    """A seed (any Python int, taken mod 2^64) -> the Philox key (lo, hi)."""
    s = int(seed) & M64
    return s & 0xFFFFFFFF, s >> 32


def prior_noise(seeds, n_feats, T, dtype=np.float32):
    """z (B, n_feats, T) for a list of B seeds; dtype=np.float64 returns the values before the rounding to float32."""
    Q = (T + 3) // 4
    out = np.empty((len(seeds), n_feats, 4 * Q), dtype=np.float64)
    q = np.arange(Q, dtype=np.uint64)[None, :]
    f = np.arange(n_feats, dtype=np.uint64)[:, None]
    for i, s in enumerate(seeds):
        k0, k1 = seed_key(s)
        w0, w1, w2, w3 = philox4x32_10(q, f, 0, 0, k0, k1)
        out[i, :, 0::4], out[i, :, 1::4] = box_muller(w0, w1)
        out[i, :, 2::4], out[i, :, 3::4] = box_muller(w2, w3)
    return out[:, :, :T].astype(dtype)


def splitmix64(seed, n):
    """The first n outputs of splitmix64 (Steele, Lea and Flood 2014; Vigna's splitmix64.c) seeded with `seed` mod 2^64."""
    x, out = int(seed) & M64, []
    for _ in range(n):
        x = (x + 0x9E3779B97F4A7C15) & M64
        z = x
        z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M64
        z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M64
        out.append(z ^ (z >> 31))
    return out
