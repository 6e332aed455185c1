"""CPU restatement (numpy, test-only) of gp_object_noise, the keyed per-object prior noise (DESIGN.md section 4.6f).

Philox4x32-10 (Salmon, Moraes, Dror, Shaw: "Parallel random numbers: as easy as 1, 2, 3", SC'11; the Random123
library) keyed with (lo32, hi32) of the object's int64 key.  Element e = r*9 + c of the object's [R, 9] block belongs
to Box-Muller pair p = e // 2; pair p uses the words 2*(p % 2), 2*(p % 2) + 1 of the Philox output for counter
(p // 2, 0, 0, 0).  u = (w + 0.5) * 2^-32 in float64; n_2p = sqrt(-2 ln u_a) cos(2 pi u_b), n_2p+1 = ... sin(...),
in float64, rounded to float32; the output is n * sigma multiplied in float32.
"""
import numpy as np

M0, M1 = 0xD2511F53, 0xCD9E8D57
W0, W1 = 0x9E3779B9, 0xBB67AE85
MASK = 0xFFFFFFFF


def philox4x32_10(ctr, key):
    """ctr: uint32 [..., 4], key: uint32 [..., 2] (broadcast) -> uint32 [..., 4]."""
    ctr = np.asarray(ctr, dtype=np.uint64)
    key = np.asarray(key, dtype=np.uint64)
    c0, c1, c2, c3 = (ctr[..., i] for i in range(4))
    k0, k1 = key[..., 0], key[..., 1]
    for _ in range(10):
        p0 = np.uint64(M0) * c0          # < 2^64: exact in uint64
        p1 = np.uint64(M1) * c2
        c0, c1, c2, c3 = ((p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & np.uint64(MASK),
                          (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & np.uint64(MASK))
        k0 = (k0 + np.uint64(W0)) & np.uint64(MASK)
        k1 = (k1 + np.uint64(W1)) & np.uint64(MASK)
    return np.stack([c0, c1, c2, c3], axis=-1).astype(np.uint32)


def key_words(key):
    """int64 key -> (lo32, hi32) as uint32."""
    k = int(key) & 0xFFFFFFFFFFFFFFFF
    return np.array([k & MASK, k >> 32], dtype=np.uint32)


def object_words(key, R):
    """The Philox words of one object's block: uint32 [ceil(R*9/4), 4], row q = Philox(counter (q, 0, 0, 0), key)."""
    calls = (R * 9 + 3) // 4
    ctr = np.zeros((calls, 4), dtype=np.uint32)
    ctr[:, 0] = np.arange(calls, dtype=np.uint32)
    return philox4x32_10(ctr, key_words(key)[None, :])


def object_normals(key, R):
    """Standard normals of one object's block, float32 [R, 9] (before the sigma scaling)."""
    w = object_words(key, R).reshape(-1, 2).astype(np.float64)   # pair p = row p: (w_a, w_b)
    u = (w + 0.5) * 2.0 ** -32
    rad = np.sqrt(-2.0 * np.log(u[:, 0]))
    ang = 2.0 * np.pi * u[:, 1]
    n = np.stack([rad * np.cos(ang), rad * np.sin(ang)], axis=1).reshape(-1)[:R * 9]
    return n.astype(np.float32).reshape(R, 9)


def object_noise(keys, sigma, R):
    """gp_object_noise: keys int64 [B], sigma float32 [B] -> float32 [B*R, 9]."""
    sigma = np.asarray(sigma, dtype=np.float32)
    return np.concatenate([object_normals(k, R) * sigma[b] for b, k in enumerate(keys)])
