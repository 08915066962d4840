"""CPU: the temporal resolve's per-pixel math (csrc/rt_temporal.cuh: projection, tap validity, bilinear gather, blend, and the
filter's per-pixel colour tolerance; shared with the CUDA kernels of rt_temporal.cu and rt_denoise.cu) compiled for the host through
tests/host_emu/cuda_shim.h, bit for bit against the float32 numpy reference (tests/temporal_reference.py) on emulated guides of
moved cameras and on random poses; and the C-ABI additions (header declarations, struct layout, defaults)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import rtb200
from conftest import ROOT, SEED
import temporal_reference as ref

EMU_DIR = os.path.join(ROOT, "tests", "host_emu")
W, H = 97, 61


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


@pytest.fixture(scope="session")
def tp_emu(tmp_path_factory):
    """g++ build of tests/host_emu/temporal_emu.cpp into a temporary library."""
    so = str(tmp_path_factory.mktemp("temporal_emu") / "libtemporal_emu.so")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-o", so, os.path.join(EMU_DIR, "temporal_emu.cpp")])
    lib = C.CDLL(so)
    lib.emu_tp_reproject.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int] + [C.c_void_p] * 5 + [C.c_float] * 3 + [C.c_void_p]
    lib.emu_tp_copy.argtypes = [C.c_void_p, C.c_int, C.c_float, C.c_void_p]
    lib.emu_tp_output.argtypes = [C.c_void_p, C.c_float, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
    lib.emu_tp_filter.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, C.c_void_p]
    return lib


def _pose12(pose):
    return np.ascontiguousarray(np.concatenate(pose), np.float32)


def _emu_reproject(lib, cur, prev, ids, nt, hh, hid, hnt, cap, tz, tn):
    h, w = ids.shape
    out = np.zeros((h, w, 4), np.float32)
    c = lambda a, t=np.float32: np.ascontiguousarray(a, t)
    ids, nt, hh, hid, hnt = c(ids, np.int32), c(nt), c(hh), c(hid, np.int32), c(hnt)
    lib.emu_tp_reproject(_p(_pose12(cur)), _p(_pose12(prev)), w, h, _p(ids), _p(nt), _p(hh), _p(hnt), _p(hid), cap, tz, tn, _p(out))
    return out


def _cameras():
    """(name, camera) pairs around the default camera: translations, rotations about several axes, FOV changes, and combinations."""
    out = []
    base = rtb200.default_camera(55)
    out.append(("same", base))
    for name, d in (("x", (0.05, 0, 0)), ("z", (0, 0, 0.3)), ("xyz", (-0.1, 0.07, -0.2))):
        c = rtb200.default_camera(55)
        for k in range(3):
            c.pos[k] += d[k]
        out.append(("move_" + name, c))
    for name, ang, ax in (("yaw", 0.02, (0, 1, 0)), ("pitch", -0.03, (1, 0, 0)), ("roll", 0.05, (0, 0, 1)), ("oblique", 0.04, (0.3, 0.8, 0.5))):
        c = rtb200.default_camera(55)
        rtb200.rotate_camera(c, ang, ax)
        out.append(("rot_" + name, c))
    c = rtb200.default_camera(50)
    out.append(("fov", c))
    c = rtb200.default_camera(60)
    rtb200.rotate_camera(c, 0.03, (0, 1, 0))
    c.pos[0] += 0.04
    out.append(("fov_rot_move", c))
    return out


@pytest.fixture(scope="session")
def guides(scenes):
    """Emulated primary-hit guides (ids, (normal, t)) of Scene1 at 97 x 61 for every camera of _cameras()."""
    from test_device_logic_cpu import build_emu
    lib = C.CDLL(build_emu())
    lib.emu_render.restype = C.c_longlong
    objs = np.ascontiguousarray(scenes["Scene1"], rtb200.OBJECT_DTYPE)
    par = rtb200.default_params(width=W, height=H, mode=0, max_bounces=1, seed_lo=SEED[0], seed_hi=SEED[1])
    out = {}
    for name, cam in _cameras():
        rad = np.zeros((H, W, 3), np.float32)
        ids = np.zeros((H, W), np.int32); t = np.zeros((H, W), np.float32)
        nrm = np.zeros((H, W, 3), np.float32); pt = np.zeros((H, W, 3), np.float32)
        lib.emu_render(_p(objs), len(objs), C.byref(cam), C.byref(par), 0, C.c_uint32(0), 1, _p(rad), _p(ids), _p(t), _p(nrm), _p(pt))
        out[name] = (cam, ids, np.concatenate([nrm, t[..., None]], -1))
    return out


def _history(rng, shape):
    hh = np.empty(shape + (4,), np.float32)
    hh[..., :3] = rng.uniform(0.0, 8.0, shape + (3,))
    hh[..., 3] = rng.choice(np.array([0.0, 0.5, 1.0, 3.0, 17.0, 1000.0], np.float32), shape)
    return hh


TP = [(32, 0.02, 0.9), (4, 0.005, 0.99), (4096, 0.5, -1.0), (1, 1e-4, 0.0)]


@pytest.mark.parametrize("cam", [n for n, _ in _cameras()])
def test_reprojection_matches_the_reference_on_moved_cameras(tp_emu, guides, cam):
    """History at the default camera, current guides at a moved one: the prior is bit-equal to the reference."""
    _, hid, hnt = guides["same"]
    c1, ids, nt = guides[cam]
    prev, cur = ref.pose_of_camera(rtb200.default_camera(55), W, H), ref.pose_of_camera(c1, W, H)
    rng = np.random.default_rng(7)
    hh = _history(rng, (H, W))
    for cap, tz, tn in TP:
        got = _emu_reproject(tp_emu, cur, prev, ids, nt, hh, hid, hnt, cap, tz, tn)
        want = ref.reproject(cur, prev, ids, nt, hh, hid, hnt, cap, tz, tn)
        assert np.array_equal(_bits(got), _bits(want)), (cap, tz, tn)
        assert not got[ids < 0].any()
        if (cap, tz) == (32, 0.02):
            # the defaults keep the history over most of the hit pixels for these small moves
            frac = float((got[..., 3] > 0).sum()) / float((ids >= 0).sum())
            assert frac > (0.6 if cam != "move_z" else 0.3), frac
            assert float(got[..., 3].max()) <= 32.0


def test_identical_pose_reprojects_onto_itself(tp_emu, guides):
    """With the same pose and guides every hit pixel finds its own history (to rounding of the projection): the bilinear weights
    concentrate on the pixel itself, so the prior is within rounding of the copy."""
    _, ids, nt = guides["same"]
    pose = ref.pose_of_camera(rtb200.default_camera(55), W, H)
    hh = np.zeros((H, W, 4), np.float32)
    hh[..., :3] = 2.0; hh[..., 3] = 5.0
    got = _emu_reproject(tp_emu, pose, pose, ids, nt, hh, ids, nt, 32, 0.02, 0.9)
    hit = ids >= 0
    assert (got[hit][:, 3] > 0).mean() > 0.95
    np.testing.assert_allclose(got[hit][:, :3][got[hit][:, 3] > 0], 2.0, rtol=1e-6)


def test_random_poses_and_guides_match_the_reference(tp_emu):
    """Random (non-orthonormal) poses, guides and histories, including points behind the previous camera and singular bases."""
    rng = np.random.default_rng(21)
    h, w = 23, 31
    for trial in range(40):
        f = lambda *s: rng.normal(size=s).astype(np.float32)
        prev = (f(3), f(3) * np.float32(0.01), f(3) * np.float32(0.01), f(3) * np.float32(0.01))
        if trial % 10 == 9:
            prev = (prev[0], prev[1], prev[1] * np.float32(2), prev[3])          # singular
        cur = tuple(p + f(3) * np.float32(0.002 if k else 0.05) for k, p in enumerate(prev)) if trial % 2 else (f(3), f(3) * np.float32(0.01), f(3) * np.float32(0.01), f(3) * np.float32(0.01))
        ids = rng.integers(-1, 3, (h, w)).astype(np.int32)
        hid = rng.integers(-1, 3, (h, w)).astype(np.int32)
        nt = np.concatenate([f(h, w, 3), rng.uniform(-0.5, 30.0, (h, w, 1)).astype(np.float32)], -1)
        hnt = np.concatenate([f(h, w, 3), rng.uniform(-0.5, 30.0, (h, w, 1)).astype(np.float32)], -1)
        hh = _history(rng, (h, w))
        for cap, tz, tn in TP:
            got = _emu_reproject(tp_emu, cur, prev, ids, nt, hh, hid, hnt, cap, tz, tn)
            want = ref.reproject(cur, prev, ids, nt, hh, hid, hnt, cap, tz, tn)
            assert np.array_equal(_bits(got), _bits(want)), (trial, cap, tz, tn)
        m = np.zeros(9, np.float32)
        tp_emu.emu_tp_inverse(_p(_pose12(prev)), _p(m))
        want = ref.inverse(prev)
        assert np.array_equal(np.isnan(m), np.isnan(want)), trial               # a singular basis: 0 / 0, whose NaN sign differs
        assert np.array_equal(_bits(m[~np.isnan(m)]), _bits(want[~np.isnan(want)])), trial


def test_blend_and_copy_match_the_reference(tp_emu):
    rng = np.random.default_rng(5)
    n = 4096
    S = rng.uniform(0.0, 50.0, (n, 4)).astype(np.float32)
    ids = rng.integers(-1, 4, n).astype(np.int32)
    P = _history(rng, (n,))
    for N in (0, 1, 3, 1000):
        got = np.zeros((n, 4), np.float32)
        tp_emu.emu_tp_output(_p(S), float(N), _p(ids), _p(P), n, _p(got))
        want = ref.output(S[None], N, ids[None], P[None])[0]
        assert np.array_equal(_bits(got), _bits(want)), N
        plain = (ids < 0) | (P[:, 3] == 0) | (N == 0)
        mean = S[:, :3] / np.float32(N) if N else S[:, :3]
        assert np.array_equal(_bits(got[plain][:, :3]), _bits(mean[plain]))
        assert np.array_equal(got[plain][:, 3], np.full(int(plain.sum()), N, np.float32))
    for cap in (1, 32, 4096):
        got = np.zeros((n, 4), np.float32)
        tp_emu.emu_tp_copy(_p(P), n, float(cap), _p(got))
        assert np.array_equal(_bits(got), _bits(ref.copy_prior(P, cap)))


@pytest.mark.parametrize("passes", [1, 3, 5])
def test_per_pixel_count_filter_matches_the_reference(tp_emu, guides, passes):
    from denoise_reference import denoise, luma
    _, ids, nt = guides["rot_yaw"]
    rng = np.random.default_rng(9)
    O4 = np.empty((H, W, 4), np.float32)
    O4[..., :3] = rng.uniform(0.0, 4.0, (H, W, 3))
    O4[..., 3] = rng.choice(np.array([0.0, 1.0, 1.5, 9.0, 33.0], np.float32), (H, W))
    for power, sc, sz in ((128, 2.0, 1.0), (16, 0.5, 2.0)):
        got = np.zeros((H, W, 4), np.float32)
        tp_emu.emu_tp_filter(_p(O4), _p(np.ascontiguousarray(nt, np.float32)), _p(np.ascontiguousarray(ids, np.int32)), W, H, passes,
                             power.bit_length() - 1, sc, sz, _p(got))
        want = ref.filter(O4, ids, nt, passes, power, sc, sz)
        np.testing.assert_allclose(got[..., :3], want, rtol=1e-5, atol=1e-6 * float(want.max()))
        np.testing.assert_allclose(got[..., 3], luma(got[..., :3]), rtol=1e-6, atol=0)
    # with N_eff = N everywhere the form is the plain filter of a sum image at N samples, bit for bit
    S = np.concatenate([O4[..., :3] * np.float32(4), np.zeros((H, W, 1), np.float32)], -1)
    O4[..., :3] = S[..., :3] / np.float32(4)
    O4[..., 3] = 4.0
    np.testing.assert_array_equal(_bits(ref.filter(O4, ids, nt, passes)), _bits(denoise(S, 4, ids, nt, passes)))


def test_temporal_abi_declarations():
    from test_capi_cpu import header_functions
    names = header_functions()
    new = ("rt_default_temporal_params", "rt_temporal_rgba8", "rt_read_temporal", "rt_reset_temporal")
    for n in new:
        assert n in names and n in rtb200.EXPORTS
    assert C.sizeof(rtb200.RtTemporalParams) == 16
    lib = rtb200.load_library()
    for n in new:
        assert hasattr(lib, n)
    p = rtb200.default_temporal_params()
    assert p.max_history == 32 and p.tau_depth == np.float32(0.02) and p.tau_normal == np.float32(0.9) and p.reserved == 0
    q = rtb200.default_temporal_params(max_history=8, tau_normal=0.5)
    assert (q.max_history, q.tau_normal) == (8, 0.5) and q.tau_depth == np.float32(0.02)


def test_temporal_calls_refuse_without_a_context():
    """No context (NULL): RT_ERR_INVALID, never a CPU path."""
    lib = rtb200.load_library()
    out = np.zeros(16, np.uint32)
    assert lib.rt_temporal_rgba8(None, None, None, _p(out), 16, 1) == rtb200.RT_ERR_INVALID
    assert lib.rt_read_temporal(None, None, None, _p(out)) == rtb200.RT_ERR_INVALID
    assert lib.rt_reset_temporal(None) == rtb200.RT_ERR_INVALID
