"""numpy restatement of the keyed noise stream of the sampler kernels (include/diffpose_b200.h, "Keyed noise").

Philox4x32-10 (Salmon, Moraes, Dror, Shaw, "Parallel random numbers: as easy as 1, 2, 3", SC'11; the round function and
constants of Random123 / cuRAND `Philox4_32_10`) with key (seed & 0xffffffff, seed >> 32) and counter (e >> 2, s, b, h) for
noise element e = joint * c + coord of pose b, hypothesis h, step s.  Output words x0..x3; with l = e & 3, m = l >> 1:

    u1 = ((x[2m] >> 8) + 1) * 2^-24        in (0, 1]
    u2 = (x[2m+1] >> 8) * 2^-24            in [0, 1)
    z  = sqrt(-2 log u1) * (cos(2 pi u2) if l is even else sin(2 pi u2))

The Philox bits here are exact (uint32); the normals are float64, which the device's fp32 values match within a few ulp.
"""
from __future__ import annotations

import numpy as np

M0, M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
W0, W1 = 0x9E3779B9, 0xBB67AE85
_MASK = np.uint64(0xFFFFFFFF)


def philox4x32_10(ctr, key):
    """ctr: uint32 array [..., 4]; key: uint32 array [..., 2] (broadcast against ctr).  Returns uint32 [..., 4]."""
    c = [np.asarray(ctr, dtype=np.uint32)[..., i].astype(np.uint64) for i in range(4)]
    k = np.asarray(key, dtype=np.uint32)
    k0 = k[..., 0].astype(np.uint64)
    k1 = k[..., 1].astype(np.uint64)
    for r in range(10):
        if r:
            k0 = (k0 + np.uint64(W0)) & _MASK
            k1 = (k1 + np.uint64(W1)) & _MASK
        p0 = M0 * c[0]
        p1 = M1 * c[2]
        hi0, lo0 = p0 >> np.uint64(32), p0 & _MASK
        hi1, lo1 = p1 >> np.uint64(32), p1 & _MASK
        c = [hi1 ^ c[1] ^ k0, lo1, hi0 ^ c[3] ^ k1, lo0]
    return np.stack(c, axis=-1).astype(np.uint32)


def seed_key(seed):
    seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    return np.array([seed & 0xFFFFFFFF, seed >> 32], dtype=np.uint32)


def normals_from_words(x, l):
    """Box-Muller of one Philox output quad x [..., 4] for lane l = e & 3 (int array broadcast against x[..., 0])."""
    l = np.asarray(l)
    m = l >> 1
    a = np.take_along_axis(x, (2 * m)[..., None], axis=-1)[..., 0].astype(np.float64)
    b = np.take_along_axis(x, (2 * m + 1)[..., None], axis=-1)[..., 0].astype(np.float64)
    u1 = (np.floor(a / 256.0) + 1.0) * 2.0 ** -24
    u2 = np.floor(b / 256.0) * 2.0 ** -24
    r = np.sqrt(-2.0 * np.log(u1))
    return np.where(l & 1, r * np.sin(2.0 * np.pi * u2), r * np.cos(2.0 * np.pi * u2))


def normal(seed, s, b, h, e):
    """z for step s, pose b, hypothesis h, element e (integer arrays, broadcast together), float64."""
    s, b, h, e = np.broadcast_arrays(*(np.asarray(v, dtype=np.int64) for v in (s, b, h, e)))
    ctr = np.stack([e >> 2, s, b, h], axis=-1).astype(np.uint32)
    return normals_from_words(philox4x32_10(ctr, seed_key(seed)), e & 3)


def noise(seed, n_steps, n_pose, n_hyp=1, n_pts=17, c=5, *, pose_offset=0, step_offset=0):
    """The keyed stream as the [n_steps, n_hyp * n_pose, n_pts, c] (hypothesis-major) float64 array the sampler's noise=
    argument takes: entry [k, h * n_pose + p, j, i] is normal(seed, step_offset + k, pose_offset + p, h, j * c + i)."""
    s = step_offset + np.arange(n_steps)[:, None, None, None, None]
    h = np.arange(n_hyp)[None, :, None, None, None]
    b = pose_offset + np.arange(n_pose)[None, None, :, None, None]
    e = np.arange(n_pts * c).reshape(n_pts, c)[None, None, None]
    z = normal(seed, s, b, h, e)
    return z.reshape(n_steps, n_hyp * n_pose, n_pts, c)
