"""float64 statement of the denoised resolve's a-trous filter, written from the definition in the header comment of
software-raytracer_b200/csrc/rt_denoise.cuh (not from the float32 restatement tests/denoise_reference.py, whose evaluation order it
does not follow). Pass i (step s = 2^i) replaces the colour c of every pixel p with a primary hit by sum_q w_pq c_q / sum_q w_pq,

    w_pq = h[dx] h[dy] [id_q == id_p] max(0, n_p . n_q)^P exp(-(|t_p - t_q| / dz_p + (l_p - l_q)^2 kc)),
    dz_p = sigma_z s max(|t_p|, 1e-3),  kc = 4^i N / sigma_c^2,  l = Y / (1 + Y),

over the taps q = p + s (dx, dy), dx, dy in -2..2, that lie in the image; pixels without a hit are copied. N is the sample count (at
least 1); in the per-pixel count form of the temporal resolve it is the pixel's own weight N_eff (rt_temporal.cuh tp_kc).

The guides, the sums and the parameters are float32 values; they are promoted to float64 and every operation, exp included, is
float64. Returns float64 (h, w, 3) colours.
"""
import numpy as np

# kDenoiseSigmaMin (rt_denoise.cuh): the smallest sigma_color / sigma_depth the C-ABI accepts
SIGMA_MIN = 2.0 ** -16
H = {-2: 1.0 / 16, -1: 4.0 / 16, 0: 6.0 / 16, 1: 4.0 / 16, 2: 1.0 / 16}


def luma(rgb):
    """Reinhard-mapped Rec. 709 luminance Y / (1 + Y)."""
    y = 0.2126 * rgb[..., 0] + 0.7152 * rgb[..., 1] + 0.0722 * rgb[..., 2]
    return y / (1.0 + y)


def mean(accum, samples):
    """The pass-0 input: sum / samples (samples 0: the buffer already holds a mean)."""
    m = np.asarray(accum, np.float32)[..., :3].astype(np.float64)
    return m / float(samples) if samples > 0 else m


def _filter(c, n, ids, nt, passes, normal_power, sigma_color, sigma_depth):
    """The passes over colours c (h, w, 3) float64 with the colour weight n (a scalar or an (h, w) array, already at least 1)."""
    ids = np.asarray(ids, np.int64)
    nt = np.asarray(nt, np.float32).astype(np.float64)
    sc = float(np.float32(sigma_color))
    sz = float(np.float32(sigma_depth))
    h, w = ids.shape
    hit = ids >= 0
    normal, t = nt[..., :3], nt[..., 3]
    for i in range(passes):
        s = 2 ** i
        l = luma(c)
        kc = (4.0 ** i) * n / (sc * sc)
        dz = (sz * s) * np.maximum(np.abs(t), 1e-3)
        num = np.zeros((h, w, 3))
        den = np.zeros((h, w))
        for dy in range(-2, 3):
            for dx in range(-2, 3):
                # pixel p = (x, y) takes tap q = (x + dx s, y + dy s) where q is inside: p in [ylo, yhi) x [xlo, xhi)
                ylo, yhi = max(0, -dy * s), min(h, h - dy * s)
                xlo, xhi = max(0, -dx * s), min(w, w - dx * s)
                if ylo >= yhi or xlo >= xhi:
                    continue
                P = (slice(ylo, yhi), slice(xlo, xhi))
                Q = (slice(ylo + dy * s, yhi + dy * s), slice(xlo + dx * s, xhi + dx * s))
                cos = np.maximum(np.sum(normal[P] * normal[Q], axis=-1), 0.0) ** normal_power
                kcp = kc[P] if np.ndim(kc) else kc
                with np.errstate(all="ignore"):                # guides of sky pixels are not read: they may be inf
                    e = np.abs(t[P] - t[Q]) / dz[P] + (l[P] - l[Q]) ** 2 * kcp
                    wt = np.where(ids[P] == ids[Q], H[dx] * H[dy] * cos * np.exp(-e), 0.0)
                num[P] += wt[..., None] * c[Q]
                den[P] += wt
        out = c.copy()
        out[hit] = num[hit] / den[hit][:, None]
        c = out
    return c


def denoise(accum, samples, ids, nt, passes, normal_power, sigma_color, sigma_depth):
    """The filter of rt_read_denoised over an accumulation buffer holding `samples` samples (0: a mean)."""
    return _filter(mean(accum, samples), float(max(int(samples), 1)), ids, nt, passes, normal_power, sigma_color, sigma_depth)


def denoise_neff(O4, ids, nt, passes, normal_power, sigma_color, sigma_depth):
    """The per-pixel count form behind the filtered temporal resolve: O4 (h, w, 4) holds the blend and its weight N_eff."""
    O4 = np.asarray(O4, np.float32).astype(np.float64)
    return _filter(O4[..., :3], np.maximum(O4[..., 3], 1.0), ids, nt, passes, normal_power, sigma_color, sigma_depth)
