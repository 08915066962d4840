"""float32 numpy reference of the denoised resolve's filter (software-raytracer_b200/csrc/rt_denoise.cuh, DESIGN.md 5).

Every operation is float32 and evaluated in the order the CUDA code uses; the sums over the 25 taps run in the same order
(dy outer, dx inner), vectorised over the pixels.
"""
import numpy as np

F = np.float32
H = {-2: F(0.0625), -1: F(0.25), 0: F(0.375), 1: F(0.25), 2: F(0.0625)}


def luma(rgb):
    """Reinhard-mapped Rec. 709 luminance Y / (1 + Y) of (..., 3) float32 colours."""
    y = F(0.2126) * rgb[..., 0] + F(0.7152) * rgb[..., 1] + F(0.0722) * rgb[..., 2]
    return y / (F(1) + y)


def mean_of(accum, samples):
    """The pass-0 input: accum.rgb / samples (samples 0: the buffer already holds a mean)."""
    m = np.ascontiguousarray(accum[..., :3], F)
    return m / F(samples) if samples > 0 else m.copy()


def denoise(accum, samples, ids, nt, passes=5, normal_power=128, sigma_color=2.0, sigma_depth=1.0):
    """Filtered mean radiance (h, w, 3) float32 (defaults: rt_default_denoise_params).

    accum: (h, w, 4) or (h, w, 3) sum image; ids: (h, w) int32 primary-hit object ids (-1 miss);
    nt: (h, w, 4) float32 (normal xyz, t) of the primary hit (values at miss pixels are not read)."""
    assert normal_power >= 1 and normal_power & (normal_power - 1) == 0
    pow_log2 = normal_power.bit_length() - 1
    h, w = ids.shape
    ids = np.asarray(ids, np.int32)
    nt = np.asarray(nt, F)
    c = mean_of(accum, samples)
    hit = ids >= 0
    n_eff = max(int(samples), 1)
    for i in range(passes):
        s = 1 << i
        l = luma(c)
        sz = F(sigma_depth) * F(s)
        kc = (F(1 << (2 * i)) * F(n_eff)) / (F(sigma_color) * F(sigma_color))
        dz = sz * np.maximum(np.abs(nt[..., 3]), F(1e-3))
        acc = np.zeros((h, w, 3), F)
        wsum = np.zeros((h, w), F)
        for dy in range(-2, 3):
            for dx in range(-2, 3):
                oy, ox = dy * s, dx * s
                # destination window: pixels p whose tap q = p + (ox, oy) lies inside the image
                y0, y1 = max(0, -oy), min(h, h - oy)
                x0, x1 = max(0, -ox), min(w, w - ox)
                if y0 >= y1 or x0 >= x1:
                    continue
                P = (slice(y0, y1), slice(x0, x1))
                Q = (slice(y0 + oy, y1 + oy), slice(x0 + ox, x1 + ox))
                same = (ids[Q] == ids[P]) & hit[P]
                npp, nq = nt[P], nt[Q]
                d = npp[..., 0] * nq[..., 0] + npp[..., 1] * nq[..., 1] + npp[..., 2] * nq[..., 2]
                d = np.where(d > F(0), d, F(0)).astype(F)
                for _ in range(pow_log2):
                    d = d * d
                dl = l[P] - l[Q]
                e = np.abs(npp[..., 3] - nq[..., 3]) / dz[P] + dl * dl * kc
                with np.errstate(under="ignore", over="ignore", invalid="ignore"):
                    wt = (H[dx] * H[dy]) * d * np.exp(-e)
                wt = np.where(same, wt, F(0)).astype(F)
                # the CUDA code skips taps of other ids; adding exact zeros does not change a float32 sum of non-negative terms
                acc[P] = acc[P] + wt[..., None] * c[Q]
                wsum[P] = wsum[P] + wt
        out = c.copy()
        with np.errstate(divide="ignore", invalid="ignore"):
            out[hit] = acc[hit] / wsum[hit][:, None]
        c = out
    return c


def tonemap(rgb):
    """Per-channel Reinhard c / (1 + c), the resolve's tonemap, for PSNR figures."""
    rgb = np.maximum(np.asarray(rgb, np.float64), 0.0)
    return rgb / (1.0 + rgb)


def psnr(a, b):
    mse = float(np.mean((tonemap(a) - tonemap(b)) ** 2))
    return 10.0 * np.log10(1.0 / mse) if mse > 0 else float("inf")
