"""CPU: the pixel filter (csrc/rt_filter.cuh) compiled for the host through tests/host_emu/cuda_shim.h, bit for bit against the
float32 numpy statement (tests/filter_reference.py); its offsets' distributions; the oracle with the filter in front
(tests/oracle_filtered.c: orc_render_filtered, orc_sample_dirs) against the same directions; and the C-ABI additions that need no device."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
from scipy import stats

import rtb200
import filter_reference as ref
from conftest import ROOT, SEED
from oracle_filtered import filtered_oracle
from oracle_py import OrcCamera

EMU_DIR = os.path.join(ROOT, "tests", "host_emu")
W, H = 133, 77
SAMPLES = [0, 1, 7, 1023, 0x80000005]
KINDS = [(ref.BOX, 0.5), (ref.BOX, 1.0), (ref.BOX, 4.0), (ref.TENT, 0.5), (ref.TENT, 1.0), (ref.TENT, 4.0)]


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


@pytest.fixture(scope="session")
def fe(tmp_path_factory):
    """g++ build of tests/host_emu/filter_emu.cpp into a temporary library."""
    so = str(tmp_path_factory.mktemp("filter_emu") / "libfilter_emu.so")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-I" + os.path.join(ROOT, "include"),
                           "-o", so, os.path.join(EMU_DIR, "filter_emu.cpp")])
    lib = C.CDLL(so)
    lib.emu_filter_offsets.argtypes = [C.c_int, C.c_float, C.c_void_p, C.c_int, C.c_void_p]
    lib.emu_sample_dirs.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_float, C.c_uint32, C.c_void_p]
    return lib


def _camera():
    c = rtb200.RtCamera()
    c.right[0] = 1; c.up[1] = 1; c.forward[2] = 1; c.fov_deg = 55
    return c, (0.3, 0.8, 0.5)


def _params(w=W, h=H):
    p = rtb200.default_params(width=w, height=h, mode=rtb200.RT_MODE_PATH, seed_lo=SEED[0], seed_hi=SEED[1])
    return p


def _emu_dirs(fe, cam, par, ftype, radius, sample):
    out = np.zeros((par.height, par.width, 3), np.float32)
    fe.emu_sample_dirs(C.byref(cam), C.byref(par), ftype, radius, sample, _p(out))
    return out


def test_numpy_philox_is_the_oracles(oracle):
    key = (SEED[0], SEED[1])
    for ctr in ([0, 0, 0, 1], [1234, 7, 0, 1], [0xFFFFFFFF, 0x80000005, 3, 0]):
        got = [int(v) for v in ref.philox(*[np.array(c, np.uint64) for c in ctr], key)]
        assert got == [int(v) for v in oracle.philox(ctr, key)]


@pytest.mark.parametrize("ftype,radius", KINDS)
def test_filter_offsets_bit_exact_on_every_pixel(fe, ftype, radius):
    """filter_offset() on the words of every pixel of a 133 x 77 frame for several global sample indices."""
    pixel = np.arange(W * H, dtype=np.uint64)
    for sample in SAMPLES:
        x, y, _, _ = ref.philox(pixel, sample, 0, 1, SEED)
        for w in (x, y):
            w = np.ascontiguousarray(w, np.uint32)
            got = np.zeros(w.shape, np.float32)
            fe.emu_filter_offsets(ftype, radius, _p(w), len(w), _p(got))
            want = ref.offsets(ftype, radius, w)
            assert np.array_equal(_bits(got), _bits(want))
            assert np.all(np.abs(got) <= np.float32(radius))


def test_filter_offsets_at_the_word_edges(fe):
    """Words at the ends of the range and at the tent's fold (v = 1): exact values."""
    w = np.array([0, 0xFF, 0x100, 0x7FFFFFFF, 0x80000000, 0x800000FF, 0xFFFFFF00, 0xFFFFFFFF], np.uint32)
    for ftype, radius in KINDS:
        got = np.zeros(len(w), np.float32)
        fe.emu_filter_offsets(ftype, radius, _p(w), len(w), _p(got))
        assert np.array_equal(_bits(got), _bits(ref.offsets(ftype, radius, w)))
        assert got[0] == -np.float32(radius) and got[1] == -np.float32(radius)       # u = 0: the left edge, included
        assert got[4] == 0.0                                                           # u = 1/2: the centre
        assert got[-1] < np.float32(radius)                                            # u < 1: the right edge, excluded


@pytest.mark.parametrize("ftype,radius", KINDS)
def test_sample_dirs_bit_exact_on_every_pixel(fe, ftype, radius):
    cam, axis = _camera()
    rtb200.rotate_camera(cam, 0.07, axis)
    par = _params()
    for sample in SAMPLES[:3]:
        got = _emu_dirs(fe, cam, par, ftype, radius, sample)
        want = ref.sample_dirs(cam, W, H, SEED, ftype, radius, sample)
        assert np.array_equal(_bits(got), _bits(want))


def test_zero_offset_gives_the_corner_rays(fe, oracle):
    """RT_FILTER_NONE (offset 0) is ray_dir / orc_ray_dirs bit for bit."""
    cam, _ = _camera()
    par = _params()
    got = _emu_dirs(fe, cam, par, ref.NONE, 0.5, 3)
    ocam = OrcCamera(); ocam.right[0] = 1; ocam.up[1] = 1; ocam.forward[2] = 1; ocam.fov_deg = 55
    assert np.array_equal(_bits(got), _bits(oracle.ray_dirs(ocam, W, H)))
    assert np.array_equal(_bits(got), _bits(ref.sample_dirs(cam, W, H, SEED, ref.NONE, 0.5, 3)))


@pytest.mark.parametrize("radius", [0.5, 1.0, 4.0])
def test_box_offsets_are_uniform(radius):
    jx, jy = ref.jitter(W, H, SEED, ref.BOX, radius, 11)
    for j in (jx, jy):
        j = j.ravel().astype(np.float64)
        assert j.min() >= -radius and j.max() < radius
        assert stats.kstest(j / radius, "uniform", args=(-1.0, 2.0)).pvalue > 1e-3


@pytest.mark.parametrize("radius", [0.5, 1.0, 4.0])
def test_tent_offsets_follow_the_tent(radius):
    jx, jy = ref.jitter(W, H, SEED, ref.TENT, radius, 11)
    for j in (jx, jy):
        j = j.ravel().astype(np.float64)
        assert j.min() > -radius and j.max() < radius
        assert stats.kstest(j / radius, ref.tent_cdf).pvalue > 1e-3
    # x and y come from different words: no correlation
    assert abs(np.corrcoef(jx.ravel(), jy.ravel())[0, 1]) < 0.02


def test_oracle_restatement_uses_the_same_directions(oracle, scenes):
    """orc_sample_dirs gives the numpy directions, and orc_render_filtered feeds radiance() exactly those: with max_bounces 0 every
    sample is the emission of the hit object or the environment colour of its own ray."""
    fo = filtered_oracle()
    w, h = 61, 37
    ocam = OrcCamera(); ocam.right[0] = 1; ocam.up[1] = 1; ocam.forward[2] = 1; ocam.fov_deg = 55
    objs = scenes["Scene1"]
    p = oracle.default_params(width=w, height=h, max_bounces=0, mode=0, seed_lo=SEED[0], seed_hi=SEED[1])
    for ftype, radius in ((ref.BOX, 0.5), (ref.TENT, 1.0)):
        s0, n = 5, 3
        _, per, segs = fo.render_filtered(objs, ocam, p, s0, n, ftype, radius, per_sample=True)
        assert segs == n * w * h
        for k in range(n):
            d = fo.sample_dirs(ocam, w, h, SEED[0], SEED[1], ftype, radius, s0 + k)
            assert np.array_equal(_bits(d), _bits(ref.sample_dirs(ocam, w, h, SEED, ftype, radius, s0 + k)))
            dd = d.reshape(-1, 3)
            ids, _, _, _ = oracle.trace_rays(objs, np.zeros_like(dd), dd)
            want = oracle.env_color(p, dd)
            hit = ids >= 0
            want[hit] = np.asarray(objs["emissive"], np.float32)[ids[hit]]
            assert np.array_equal(_bits(per[k].reshape(-1, 3)), _bits(want))
    # RT_FILTER_NONE is orc_render
    a, _, sa = fo.render_filtered(objs, ocam, p, 0, 2, ref.NONE, 0.5)
    b, _, sb = oracle.render(objs, ocam, p, 0, 2)
    assert sa == sb and np.array_equal(_bits(a), _bits(b))


def test_capi_filter_declarations_and_defaults():
    """The new symbols are exported (the symbol list the C-ABI test compares with the header) and the default is NONE / 0.5."""
    lib = rtb200.load_library()
    for name in ("rt_default_pixel_filter", "rt_set_pixel_filter", "rt_get_pixel_filter", "rt_read_sample_dirs", "rt_group_set_pixel_filter"):
        assert name in rtb200.EXPORTS and hasattr(lib, name)
    assert C.sizeof(rtb200.RtPixelFilter) == 16
    f = rtb200.default_pixel_filter()
    assert (f.type, f.radius, list(f.reserved)) == (rtb200.RT_FILTER_NONE, 0.5, [0, 0])
    assert (rtb200.RT_FILTER_NONE, rtb200.RT_FILTER_BOX, rtb200.RT_FILTER_TENT) == (0, 1, 2)
