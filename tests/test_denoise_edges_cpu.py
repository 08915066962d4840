"""CPU: the denoised resolve's filter (csrc/rt_denoise.cuh through tests/host_emu/denoise_emu.cpp, the host build that
test_denoise_cpu.py pins to the float32 restatement; built here through denoise_edges_emu.cpp with the same flags) against the
float64 statement tests/denoise_f64.py at the filter's edges: images smaller than the kernels' 32 x 8 tile and than the steps of
passes 6-8, every pass count, normal powers 1 and 256, sample counts up to 2^32 - 1, and the ends of the accepted sigma ranges, on
synthetic guides with negative and tiny t, anti-parallel and orthogonal neighbour normals, all-sky, one-id and checkerboard-id
images and luminance steps of 0 and of nearly 1."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT
import denoise_f64 as f64
import denoise_reference as ref

F32_MAX = float(np.finfo(np.float32).max)
SIZES = [(1, 1), (1, 37), (37, 1), (31, 7), (33, 9), (97, 61)]      # (width, height)
KINDS = ["mixed", "sky", "one_id", "checker", "steps"]
SAMPLES = [0, 1, 1 << 20, (1 << 32) - 1]
SIGMAS = [f64.SIGMA_MIN, 1e-3, 2.0, 1e30, F32_MAX]
RTOL, ATOL = 1e-4, 1e-5                                         # atol relative to max |want|

# Colours are grey levels times one tint. Colours of different chroma whose luminances lie closer than float32 resolves them are
# weighted by an ill-conditioned exp(-(l_p - l_q)^2 kc) once kc is large (its error grows as sqrt(kc) ulp(l)), so no float32
# filter meets a float64 statement there; along one chroma line a weight error moves the output by no more than the luminance does.
TINT = np.float32([1.0, 0.8, 0.6])
# normals whose pairwise dot products are 1, -1 (anti-parallel), 0 (orthogonal) and in between
NORMALS = np.array([[0, 0, 1], [0, 0, -1], [1, 0, 0], [0, 0.6, 0.8], [0.48, 0.6, 0.64]], np.float32)


def make_guides(kind, w, h, seed):
    """(mean (h, w, 3), ids (h, w), nt (h, w, 4)) float32 / int32 synthetic inputs of one kind."""
    rng = np.random.default_rng(seed)
    y, x = np.mgrid[0:h, 0:w]
    grey = rng.uniform(0.0, 4.0, (h, w)).astype(np.float32)
    nrm = np.broadcast_to(NORMALS[0], (h, w, 3)).copy()
    t = np.full((h, w), 1.5, np.float32)
    if kind == "mixed":
        ids = ((x // 3 + y // 2) % 4 - 1).astype(np.int32)         # three objects and sky
        nrm = NORMALS[(7 * x + 3 * y) % len(NORMALS)]
        u = rng.uniform(0.0, 1.0, (h, w))
        t = np.where(u < 0.4, rng.uniform(-3.0, -0.5, (h, w)),      # negative t (a sphere around the camera) ..
                     np.where(u < 0.6, rng.uniform(-9e-4, 9e-4, (h, w)), rng.uniform(0.5, 3.0, (h, w))))   # .. and |t| < 1e-3
    elif kind == "sky":
        ids = np.full((h, w), -1, np.int32)
    elif kind == "one_id":
        ids = np.zeros((h, w), np.int32)
        t = (1.0 + 0.01 * x - 0.02 * y).astype(np.float32)
    elif kind == "checker":
        ids = ((x + y) & 1).astype(np.int32)
    else:                                                          # steps: left | right halves, equal on even rows, 0 | 60 on odd rows
        ids = np.zeros((h, w), np.int32)
        grey = np.where(y % 2 == 0, np.float32(1.5), np.where(x < w // 2, np.float32(0.0), np.float32(60.0))).astype(np.float32)
    mean = grey[..., None] * TINT
    nt = np.concatenate([nrm, t[..., None]], -1).astype(np.float32)
    return np.ascontiguousarray(mean), ids, np.ascontiguousarray(nt)


@pytest.fixture(scope="module")
def dn_emu(tmp_path_factory):
    """g++ build of tests/host_emu/denoise_edges_emu.cpp into a temporary library: run(accum, samples, ids, nt, passes, normal_power,
    sigma_color, sigma_depth) -> (h, w, 4) (r, g, b, l) of the last pass; run.sigma_min is kDenoiseSigmaMin."""
    so = str(tmp_path_factory.mktemp("denoise_edges_emu") / "libdenoise_edges_emu.so")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-o", so,
                           os.path.join(ROOT, "tests", "host_emu", "denoise_edges_emu.cpp")])
    lib = C.CDLL(so)
    lib.emu_denoise.argtypes = [C.c_void_p, C.c_uint, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, C.c_void_p]
    lib.emu_denoise_sigma_min.restype = C.c_float

    def run(accum, samples, ids, nt, passes, normal_power, sigma_color, sigma_depth):
        h, w = ids.shape
        accum = np.ascontiguousarray(accum, np.float32); nt = np.ascontiguousarray(nt, np.float32); ids = np.ascontiguousarray(ids, np.int32)
        out = np.zeros((h, w, 4), np.float32)
        p = lambda a: a.ctypes.data_as(C.c_void_p)
        lib.emu_denoise(p(accum), samples, p(nt), p(ids), w, h, passes, normal_power.bit_length() - 1, sigma_color, sigma_depth, p(out))
        return out
    run.sigma_min = lib.emu_denoise_sigma_min()
    return run


def sums(mean, samples):
    """An accumulation buffer (h, w, 4) holding `samples` samples of `mean` (samples 0: the mean itself)."""
    s = mean.astype(np.float64) * (samples if samples > 0 else 1)
    return np.concatenate([s.astype(np.float32), np.zeros(mean.shape[:2] + (1,), np.float32)], -1)


def cases():
    """(passes, normal_power, samples, sigma_color, sigma_depth): every pass count; the normal powers at every sample count; every
    pair of sigmas, the sample counts in turn (the smallest sigma_color meets 2^32 - 1 samples, the largest kc of all)."""
    out = [(passes, 2, 1, 2.0, 2.0) for passes in range(9)]
    out += [(8, power, n, 2.0, 2.0) for power in (1, 256) for n in SAMPLES]
    out += [(8, 2, SAMPLES[k % len(SAMPLES)], sc, sz) for k, (sc, sz) in enumerate((sc, sz) for sc in SIGMAS for sz in SIGMAS)]
    return out


def check_case(got, want, accum, samples, ids, label):
    """got: the host build's (h, w, 4); want: the float64 statement's (h, w, 3)."""
    rgb = got[..., :3]
    assert np.isfinite(got).all(), label
    np.testing.assert_allclose(rgb, want, rtol=RTOL, atol=ATOL * float(np.abs(want).max(initial=0.0)), err_msg=label)
    m = ref.mean_of(accum, samples)
    sky = ids < 0
    assert np.array_equal(rgb[sky].view(np.uint32), m[sky].view(np.uint32)), label
    # a convex combination of the id's pass inputs: never outside their range, per channel
    for i in np.unique(ids[~sky]):
        sel = ids == i
        lo, hi = m[sel].min(axis=0), m[sel].max(axis=0)
        slack = 1e-6 * np.maximum(np.abs(lo), np.abs(hi))
        assert (rgb[sel] >= lo - slack).all() and (rgb[sel] <= hi + slack).all(), (label, int(i))


def test_sigma_min_of_the_host_build(dn_emu):
    """kDenoiseSigmaMin as the host build sees it is the float64 statement's SIGMA_MIN."""
    assert dn_emu.sigma_min == np.float32(f64.SIGMA_MIN) == 2.0 ** -16


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("size", SIZES, ids=["%dx%d" % s for s in SIZES])
def test_host_build_matches_the_float64_statement_at_the_edges(dn_emu, kind, size):
    w, h = size
    mean, ids, nt = make_guides(kind, w, h, seed=w * 1000 + h)
    for passes, power, samples, sc, sz in cases():
        accum = sums(mean, samples)
        label = str((kind, size, passes, power, samples, sc, sz))
        got = dn_emu(accum, samples, ids, nt, passes, power, sc, sz)
        want = f64.denoise(accum, samples, ids, nt, passes, power, sc, sz)
        check_case(got, want, accum, samples, ids, label)


def test_float64_statement_of_the_count_form():
    """denoise_neff with N_eff == 1 everywhere is the sample-count form of a mean, and with per-pixel N_eff it matches the float32
    restatement of the temporal filter (tests/temporal_reference.py) on guides where every term matters."""
    import temporal_reference as tref
    w, h = 33, 9
    mean, ids, nt = make_guides("mixed", w, h, seed=5)
    rng = np.random.default_rng(6)
    for passes, power, sc, sz in ((1, 1, 2.0, 2.0), (5, 2, 0.5, 1.0), (8, 256, 30.0, 4.0)):
        O4 = np.concatenate([mean, np.ones((h, w, 1), np.float32)], -1)
        same = f64.denoise_neff(O4, ids, nt, passes, power, sc, sz)
        np.testing.assert_array_equal(same, f64.denoise(O4, 0, ids, nt, passes, power, sc, sz))
        O4[..., 3] = rng.choice(np.float32([0.0, 1.0, 7.0, 4097.0, 4294971392.0]), (h, w))
        want = f64.denoise_neff(O4, ids, nt, passes, power, sc, sz)
        got = tref.filter(O4, ids, nt, passes, power, sc, sz)
        np.testing.assert_allclose(got, want, rtol=RTOL, atol=ATOL * float(np.abs(want).max()), err_msg=str((passes, power, sc)))
