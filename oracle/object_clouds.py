"""CPU restatement (numpy, test-only) of gp_backproject_instances and gp_sample_points (DESIGN.md section 4.13).

Stage A: pixel (u = column, v = row) with label b + 1 in 1..B and a depth z > 0 that is finite gives the float32 point
(((float)u - cx) * z / fx, ((float)v - cy) * z / fy, z), IEEE float32 operations in that order.  Object b's points
are xyz[labels == b + 1] in row-major pixel order; offsets [B+1] delimit them.

Stage B: sample_points (datasets_omni6dpose.py:459-473) to N points with the keyed permutation pi_b of [0, K): a
4-round balanced Feistel network on k = max(2, ceil(log2 K)) bits (k rounded up to even), round r mapping (L, R) to
(R, L ^ F_r(R)), F_r(R) = Philox4x32-10(counter (R, r, 1, 0), key (lo32, hi32) of the object's key).x & mask,
cycle-walked into [0, K).  The integer permutation is exact; the centre is the float64 mean of the N rows summed in
row order, rounded to float32.
"""
import functools

import numpy as np

from oracle.object_noise import key_words, philox4x32_10


def backproject_instances(depth, labels, fx, fy, cx, cy, B):
    """depth float32 [H,W], labels int32 [H,W] -> (xyz float32 [total, 3], offsets int32 [B+1])."""
    depth = np.asarray(depth, dtype=np.float32)
    labels = np.asarray(labels, dtype=np.int32)
    H, W = depth.shape
    fx, fy, cx, cy = (np.float32(v) for v in (fx, fy, cx, cy))
    v, u = np.divmod(np.arange(H * W, dtype=np.int64), W)
    z = depth.reshape(-1)
    lab = labels.reshape(-1)
    with np.errstate(invalid="ignore"):
        keep = (lab >= 1) & (lab <= B) & (z > 0) & np.isfinite(z)
    xs, offsets = [], [0]
    with np.errstate(invalid="ignore", over="ignore"):
        x = ((u.astype(np.float32) - cx) * z) / fx
        y = ((v.astype(np.float32) - cy) * z) / fy
    pts = np.stack([x, y, z], axis=1).astype(np.float32)
    for b in range(B):
        m = keep & (lab == b + 1)
        xs.append(pts[m])
        offsets.append(offsets[-1] + int(m.sum()))
    xyz = np.concatenate(xs) if xs else np.zeros((0, 3), np.float32)
    return xyz.astype(np.float32), np.asarray(offsets, dtype=np.int32)


def feistel_bits(K):
    """k of pi for K points: max(2, ceil(log2 K)), rounded up to even."""
    k = max(2, (int(K) - 1).bit_length() if K > 1 else 0)
    return k + (k & 1)


@functools.lru_cache(maxsize=256)
def _round_tables(key, half):
    """F_r(R) for every R of `half` bits: uint64 [4, 2^half]."""
    R = np.arange(1 << half, dtype=np.uint32)
    tabs = []
    for r in range(4):
        ctr = np.zeros((R.size, 4), dtype=np.uint32)
        ctr[:, 0] = R
        ctr[:, 1] = r
        ctr[:, 2] = 1
        tabs.append(philox4x32_10(ctr, key_words(key)[None, :])[:, 0].astype(np.uint64) & np.uint64((1 << half) - 1))
    return np.stack(tabs)


def permutation(key, K, j):
    """pi_b(j) for the indices j (int array, 0 <= j < K) of an object with K points and key `key`."""
    half = feistel_bits(K) // 2
    tab = _round_tables(int(key), half)
    mask = np.uint64((1 << half) - 1)
    sh = np.uint64(half)

    def enc(x):
        L, R = x >> sh, x & mask
        for r in range(4):
            L, R = R, L ^ tab[r][R]
        return (L << sh) | R

    y = enc(np.asarray(j, dtype=np.uint64))
    while True:
        out = y >= np.uint64(K)
        if not out.any():
            return y.astype(np.int64)
        y[out] = enc(y[out])


def sample_indices(key, K, N):
    """Source point of every output row of an object with K > 0 points: int64 [N]."""
    if K == N:
        return np.arange(N, dtype=np.int64)
    if K > N:
        return permutation(key, K, np.arange(N))
    tiled = (N // K) * K
    return np.concatenate([np.arange(tiled, dtype=np.int64) % K, permutation(key, K, np.arange(N - tiled))])


def sample_points(xyz, offsets, keys, N):
    """xyz float32 [rows, 3], offsets int [B+1], keys int64 [B] -> (pts float32 [B,N,3], centre float32 [B,3],
    counts int32 [B]).  Offsets are clamped into [0, rows]; K = 0 gives zero rows and a zero centre."""
    xyz = np.asarray(xyz, dtype=np.float32)
    offsets = np.clip(np.asarray(offsets, dtype=np.int64), 0, xyz.shape[0])
    B = len(offsets) - 1
    pts = np.zeros((B, N, 3), np.float32)
    centre = np.zeros((B, 3), np.float32)
    counts = np.zeros(B, np.int32)
    for b in range(B):
        K = max(0, int(offsets[b + 1] - offsets[b]))
        counts[b] = K
        if K == 0:
            continue
        pts[b] = xyz[offsets[b] + sample_indices(int(keys[b]), K, N)]
        centre[b] = (np.cumsum(pts[b].astype(np.float64), axis=0)[-1] / N).astype(np.float32)
    return pts, centre, counts
