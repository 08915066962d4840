"""float32 numpy reference of the temporal resolve (software-raytracer_b200/csrc/rt_temporal.cuh, DESIGN.md 5).

Every operation is float32 and evaluated in the order the CUDA code uses, vectorised over the pixels; the inverse of the
previous pose's axes is computed in double (Python floats) in the order of tp_inverse and rounded to float32. The filter in
its per-pixel count form (filter()) restates tests/denoise_reference.py's loop with the colour tolerance of each pixel taken
from its own weight N_eff.
"""
import ctypes as C
import ctypes.util
import math

import numpy as np

from denoise_reference import H, luma

F = np.float32

_libm = C.CDLL(ctypes.util.find_library("m"))
_libm.tanf.restype = C.c_float
_libm.tanf.argtypes = [C.c_float]


def pose_of_camera(cam, w, h):
    """(o, u, v, f) float32 of an rt_camera at w x h: the host half of ray_dir (rt_host_pack.h fill_frame_view), tanf from libm."""
    clip = F(0.01)
    aspect = F(w) / F(h)
    hfov = F(cam.fov_deg * math.pi / 180.0)
    t = F(_libm.tanf(float(hfov / F(2))))
    rd, ld = (clip * t) * aspect, clip * t
    vec = lambda a: np.array([a[0], a[1], a[2]], F)
    return vec(cam.pos), vec(cam.right) * rd, vec(cam.up) * ld, vec(cam.forward) * clip


def inverse(pose):
    """tp_inverse: rows (v x f, f x u, u x v) / det in double, det = u . (v x f), rounded to float32 (row-major (9,))."""
    _, u, v, f = [[float(x) for x in a] for a in pose]
    r = []
    for a, b in ((v, f), (f, u), (u, v)):
        r.append([a[1] * b[2] - a[2] * b[1], a[2] * b[0] - a[0] * b[2], a[0] * b[1] - a[1] * b[0]])
    det = (u[0] * r[0][0] + u[1] * r[0][1]) + u[2] * r[0][2]
    with np.errstate(over="ignore"):
        out = []
        for i in range(3):
            for k in range(3):
                try:
                    q = r[i][k] / det
                except ZeroDivisionError:
                    q = math.copysign(math.inf, r[i][k]) if r[i][k] != 0 else math.nan
                out.append(q)
        return np.array(out, np.float64).astype(F)


def ray_dirs(pose, w, h):
    """(h, w, 3) ray_dir of every pixel (pixel corners, no jitter)."""
    _, u, v, f = pose
    nx = (np.arange(w).astype(F) / F(w)) * F(2) - F(1)
    ny = (np.arange(h).astype(F) / F(h)) * F(2) - F(1)
    X, Y = nx[None, :], ny[:, None]
    c = [(u[k] * X + v[k] * Y) + f[k] for k in range(3)]
    ln = np.sqrt((c[0] * c[0] + c[1] * c[1]) + c[2] * c[2])
    return np.stack([c[k] / ln for k in range(3)], -1).astype(F)


def reproject(cur, prev, ids, nt, hist_h, hist_ids, hist_nt, cap, tau_depth, tau_normal):
    """The prior (h, w, 4) (P.rgb, w_P) of every pixel rebuilt from the history (hist_h: (h, w, 4) colour and weight, hist_ids /
    hist_nt: the history's guides) for the current pose `cur` and the history's pose `prev` (pose_of_camera tuples);
    ids / nt: the current primary-hit guides. Pixels without a hit get zeros."""
    h, w = ids.shape
    m = inverse(prev)
    o, po = cur[0], prev[0]
    nt = np.asarray(nt, F)
    t = nt[..., 3]
    dp = ray_dirs(cur, w, h)
    X = [o[k] + dp[..., k] * t for k in range(3)]
    d = [X[k] - po[k] for k in range(3)]
    with np.errstate(all="ignore"):
        a = (m[0] * d[0] + m[1] * d[1]) + m[2] * d[2]
        b = (m[3] * d[0] + m[4] * d[1]) + m[5] * d[2]
        c = (m[6] * d[0] + m[7] * d[1]) + m[8] * d[2]
        ok0 = (ids >= 0) & (c > F(0))
        xq = ((a / c + F(1)) * F(0.5)) * F(w)
        yq = ((b / c + F(1)) * F(0.5)) * F(h)
        ok0 &= (xq > F(-1)) & (xq < F(w)) & (yq > F(-1)) & (yq < F(h))
    xq = np.where(ok0, xq, F(0)).astype(F)
    yq = np.where(ok0, yq, F(0)).astype(F)
    fx0, fy0 = np.floor(xq), np.floor(yq)
    x0, y0 = fx0.astype(np.int64), fy0.astype(np.int64)
    fx, fy = xq - fx0, yq - fy0
    gx, gy = F(1) - fx, F(1) - fy
    lim = F(tau_depth) * np.sqrt((d[0] * d[0] + d[1] * d[1]) + d[2] * d[2])
    pd = ray_dirs(prev, w, h)
    A = np.zeros((h, w), F)
    R, G, B = A.copy(), A.copy(), A.copy()
    for k in range(4):
        qx, qy = x0 + (k & 1), y0 + (k >> 1)
        ok = ok0 & (qx >= 0) & (qx < w) & (qy >= 0) & (qy < h)
        qx, qy = np.clip(qx, 0, w - 1), np.clip(qy, 0, h - 1)
        ok &= hist_ids[qy, qx] == ids
        nq = hist_nt[qy, qx]
        dq = pd[qy, qx]
        e = [(po[j] + dq[..., j] * nq[..., 3]) - X[j] for j in range(3)]
        with np.errstate(all="ignore"):
            ok &= np.sqrt((e[0] * e[0] + e[1] * e[1]) + e[2] * e[2]) <= lim
            ok &= ((nt[..., 0] * nq[..., 0] + nt[..., 1] * nq[..., 1]) + nt[..., 2] * nq[..., 2]) >= F(tau_normal)
        hq = hist_h[qy, qx]
        wq = ((fx if k & 1 else gx) * (fy if k >> 1 else gy)) * hq[..., 3]
        A = np.where(ok, A + wq, A)
        R = np.where(ok, R + wq * hq[..., 0], R)
        G = np.where(ok, G + wq * hq[..., 1], G)
        B = np.where(ok, B + wq * hq[..., 2], B)
    has = A > F(0)
    Ad = np.where(has, A, F(1))
    P = np.stack([R / Ad, G / Ad, B / Ad, np.where(A < F(cap), A, F(cap))], -1)
    return np.where(has[..., None], P, F(0)).astype(F)


def copy_prior(hist_h, cap):
    """The prior of an identical pose: the history, its weight capped at `cap`."""
    P = np.array(hist_h, F)
    P[..., 3] = np.where(P[..., 3] < F(cap), P[..., 3], F(cap))
    return P


def output(S, N, ids, P):
    """(h, w, 4) (O.rgb, N_eff): (S + w_P P) / (N + w_P) where w_P > 0, the pixel has a hit and N > 0; else the plain mean with N_eff = N."""
    S = np.asarray(S, F)[..., :3]
    n = F(N)
    wp = P[..., 3]
    blend = (wp > F(0)) & (ids >= 0) & (n > F(0))
    d = n + wp
    with np.errstate(all="ignore"):
        Ob = (S + wp[..., None] * P[..., :3]) / d[..., None]
        plain = S / n if N > 0 else S.copy()
    O = np.where(blend[..., None], Ob, plain)
    return np.concatenate([O, np.where(blend, d, n)[..., None]], -1).astype(F)


def filter(O4, ids, nt, passes=5, normal_power=128, sigma_color=2.0, sigma_depth=1.0):
    """The a-trous filter over O4[..., :3] in its per-pixel count form: pass i's colour tolerance at pixel p is
    (4^i max(N_eff(p), 1)) / sigma_c^2 with N_eff = O4[..., 3]. Returns (h, w, 3)."""
    pow_log2 = normal_power.bit_length() - 1
    h, w = ids.shape
    ids = np.asarray(ids, np.int32)
    nt = np.asarray(nt, F)
    c = np.ascontiguousarray(O4[..., :3], F)
    neff = O4[..., 3]
    neff1 = np.where(neff > F(0), neff, F(1)).astype(F)
    hit = ids >= 0
    for i in range(passes):
        s = 1 << i
        l = luma(c)
        sz = F(sigma_depth) * F(s)
        kc = (F(1 << (2 * i)) * neff1) / (F(sigma_color) * F(sigma_color))
        dz = sz * np.maximum(np.abs(nt[..., 3]), F(1e-3))
        acc = np.zeros((h, w, 3), F)
        wsum = np.zeros((h, w), F)
        for dy in range(-2, 3):
            for dx in range(-2, 3):
                oy, ox = dy * s, dx * s
                y0, y1 = max(0, -oy), min(h, h - oy)
                x0, x1 = max(0, -ox), min(w, w - ox)
                if y0 >= y1 or x0 >= x1:
                    continue
                P = (slice(y0, y1), slice(x0, x1))
                Q = (slice(y0 + oy, y1 + oy), slice(x0 + ox, x1 + ox))
                same = (ids[Q] == ids[P]) & hit[P]
                npp, nq = nt[P], nt[Q]
                dd = npp[..., 0] * nq[..., 0] + npp[..., 1] * nq[..., 1] + npp[..., 2] * nq[..., 2]
                dd = np.where(dd > F(0), dd, F(0)).astype(F)
                for _ in range(pow_log2):
                    dd = dd * dd
                dl = l[P] - l[Q]
                e = np.abs(npp[..., 3] - nq[..., 3]) / dz[P] + dl * dl * kc[P]
                with np.errstate(under="ignore", over="ignore", invalid="ignore"):
                    wt = (H[dx] * H[dy]) * dd * np.exp(-e)
                wt = np.where(same, wt, F(0)).astype(F)
                acc[P] = acc[P] + wt[..., None] * c[Q]
                wsum[P] = wsum[P] + wt
        out = c.copy()
        with np.errstate(divide="ignore", invalid="ignore"):
            out[hit] = acc[hit] / wsum[hit][:, None]
        c = out
    return c
