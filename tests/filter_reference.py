"""float32 numpy statement of the pixel filter (software-raytracer_b200/csrc/rt_filter.cuh, DESIGN.md 5).

Philox4x32-10 is evaluated on uint64 arrays (exact 32 x 32 -> 64-bit products); every float operation is float32 in the order the
CUDA code uses, and sqrt is numpy's correctly rounded float32 square root (IEEE, like the device's sqrtf without fast math).
"""
import numpy as np

from temporal_reference import pose_of_camera

F = np.float32
NONE, BOX, TENT = 0, 1, 2
_MASK = np.uint64(0xFFFFFFFF)


def philox(c0, c1, c2, c3, key):
    """Philox4x32-10 of counter arrays (broadcast together) with key (k0, k1); returns four uint32 arrays."""
    c = [np.asarray(v, np.uint64) & _MASK for v in np.broadcast_arrays(c0, c1, c2, c3)]
    k0, k1 = np.uint64(key[0] & 0xFFFFFFFF), np.uint64(key[1] & 0xFFFFFFFF)
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c[0]
        p1 = np.uint64(0xCD9E8D57) * c[2]
        hi0, lo0 = p0 >> np.uint64(32), p0 & _MASK
        hi1, lo1 = p1 >> np.uint64(32), p1 & _MASK
        c = [hi1 ^ c[1] ^ k0, lo1, hi0 ^ c[3] ^ k1, lo0]
        k0 = (k0 + np.uint64(0x9E3779B9)) & _MASK
        k1 = (k1 + np.uint64(0xBB67AE85)) & _MASK
    return [v.astype(np.uint32) for v in c]


def offsets(ftype, radius, w):
    """filter_offset(): the sub-pixel offset of Philox word(s) w."""
    w = np.asarray(w, np.uint32)
    r = F(radius)
    if ftype == NONE:
        return np.zeros(w.shape, F)
    u = (w >> np.uint32(8)).astype(F) * F(2.0 ** -24)
    if ftype == BOX:
        return (u * F(2) - F(1)) * r
    v = u * F(2)
    with np.errstate(invalid="ignore"):
        lo = np.sqrt(v) - F(1)
        hi = F(1) - np.sqrt(F(2) - v)
    return np.where(v < F(1), lo, hi).astype(F) * r


def jitter(w, h, key, ftype, radius, sample):
    """(jx, jy), each (h, w): the offsets of global sample `sample` of every pixel."""
    pixel = np.arange(w * h, dtype=np.uint64).reshape(h, w)
    x, y, _, _ = philox(pixel, sample, 0, 1, key)
    return offsets(ftype, radius, x), offsets(ftype, radius, y)


def sample_dirs(cam, w, h, key, ftype, radius, sample):
    """(h, w, 3) filtered_ray_dir of global sample `sample` of every pixel (cam: an rt_camera / OrcCamera)."""
    _, u, v, f = pose_of_camera(cam, w, h)
    jx, jy = jitter(w, h, key, ftype, radius, sample)
    X = ((np.arange(w).astype(F)[None, :] + jx) / F(w)) * F(2) - F(1)
    Y = ((np.arange(h).astype(F)[:, None] + jy) / F(h)) * F(2) - F(1)
    c = [(u[k] * X + v[k] * Y) + f[k] for k in range(3)]
    ln = np.sqrt((c[0] * c[0] + c[1] * c[1]) + c[2] * c[2])
    return np.stack([c[k] / ln for k in range(3)], -1).astype(F)


def tent_cdf(x):
    """CDF of the unit tent on (-1, 1)."""
    x = np.asarray(x, np.float64)
    return np.where(x < 0, 0.5 * (1 + x) ** 2, 1 - 0.5 * (1 - x) ** 2)
