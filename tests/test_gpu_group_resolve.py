"""GPU: the denoised and temporal resolves of the library-owned multi-GPU group (rt_group_denoise_rgba8 / rt_group_read_denoised /
rt_group_temporal_rgba8 / rt_group_read_temporal / rt_group_reset_temporal; the reduce kernel k_reduce_fused in csrc/rt_kernels.cu,
the exchange and the presentation on member 0 in csrc/rt_group.cu).

A group of one device goes through the same reduce as a larger one, so on one GPU it is pinned bit for bit to a plain context, and
its errors and read-only behaviour are checked. With two or more GPUs every call is pinned to a "twin": a plain context on device 0
with the same scene, camera and parameters that is handed the rank-order float32 sum of the members' buffers (rt_write_accum) - the
kernel's arithmetic, as the library is built with -fmad=false."""
import ctypes as C
import math

import numpy as np
import pytest

import rtb200
from conftest import SEED
import temporal_reference as ref

pytestmark = pytest.mark.gpu

CAP, TZ, TN = 32, 0.02, 0.9


def _n_devices():
    import torch
    return torch.cuda.device_count()


@pytest.fixture(scope="module")
def plain():
    t = rtb200.PathTracer(0)
    yield t
    t.close()


@pytest.fixture(scope="module")
def one():
    g = rtb200.TracerGroup([0])
    yield g
    g.close()


@pytest.fixture(scope="module")
def multi():
    n = _n_devices()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    g = rtb200.TracerGroup(list(range(min(n, 4))))
    yield g
    g.close()


def _setup(t, objs, w, h, mode=rtb200.RT_MODE_PATH):
    """PathTracer or TracerGroup: scene, default camera, params, a fresh accumulation. Returns the camera."""
    cam = rtb200.default_camera(55)
    t.set_scene(objs)
    t.set_camera(cam)
    t.set_params(rtb200.default_params(width=w, height=h, mode=mode, max_bounces=8, seed_lo=SEED[0], seed_hi=SEED[1]))
    t.reset_accumulation()
    return cam


def _move(cam, yaw_deg, dx=0.0):
    rtb200.rotate_camera(cam, yaw_deg * math.pi / 180.0, [cam.up[0], cam.up[1], cam.up[2]])
    cam.pos[0] += dx
    return cam


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _same(a, b):
    return np.array_equal(_bits(a), _bits(b)) if a.dtype == np.float32 else np.array_equal(a, b)


def _rank_sum(g):
    """The members' buffers added in member order in float32 (k_reduce_fused's arithmetic) and the total sample count."""
    parts = [m.read_accum() for m in g.members]
    s = parts[0][0].copy()
    for a, _ in parts[1:]:
        s = s + a
    return s, sum(n for _, n in parts)


def _feed(twin, g):
    """Hands the group's sum to the twin; returns it."""
    s, n = _rank_sum(g)
    twin.write_accum(s, n)
    return s, n


def _guides(t):
    ids, tt, nrm, _ = t.read_aov()
    return ids, np.concatenate([nrm, tt[..., None]], -1)


# ---- one GPU: a group of one device is a plain context ------------------------------------------------------------------------
def _denoise_outputs(t, dn):
    """Every form of the denoise calls on a PathTracer or a TracerGroup (same method names)."""
    w, h = t.params.width, t.params.height
    res = [t.read_denoised(dn), t.denoise_rgba8(dn, flip_y=True), t.denoise_rgba8(dn, flip_y=False)]
    wide = np.zeros((h, w + 5), np.uint32)                     # a pitch of w + 5 pixels: the columns beyond w stay untouched
    t.denoise_rgba8(dn, out=wide[:, :w])
    res.append(wide)
    surf, owner = rtb200.host_surface(w, h)
    t.denoise_rgba8(dn, out=surf)
    res.append(surf.copy())
    del owner
    return res


@pytest.mark.parametrize("scene", ["Scene1", "Scene3_indirect"])
def test_group_of_one_denoise_is_the_plain_context(one, plain, scenes, scene):
    w, h = 161, 97
    for t in (one, plain):
        _setup(t, scenes[scene], w, h)
        t.render_spp(3)
    for passes in (0, 1, 5, None):
        dn = rtb200.default_denoise_params(passes=passes) if passes is not None else None
        got, want = _denoise_outputs(one, dn), _denoise_outputs(plain, dn)
        for k, (a, b) in enumerate(zip(got, want)):
            assert _same(a, b), (passes, k)
    assert one.stats().last_resolve_ms > 0


@pytest.mark.parametrize("scene", ["Scene1", "Scene3_indirect"])
def test_group_of_one_temporal_is_the_plain_context(one, plain, scenes, scene):
    """A turning camera, 1 sample per frame, then samples added without a move (the prior is kept), with and without the filter."""
    w, h = 161, 97
    tp = rtb200.default_temporal_params()
    dn = rtb200.default_denoise_params(passes=3)
    cams = [_setup(t, scenes[scene], w, h) for t in (one, plain)]
    for f in range(5):
        for t, cam in zip((one, plain), cams):
            if f:
                _move(cam, 0.4, 0.01 * (f & 1)); t.set_camera(cam)
            t.reset_accumulation(); t.render_spp(1)
        got = [one.read_temporal(tp), one.read_temporal(tp, dn), one.temporal_rgba8(tp, None, True), one.temporal_rgba8(tp, dn, False)]
        want = [plain.read_temporal(tp), plain.read_temporal(tp, dn), plain.temporal_rgba8(tp, None, True), plain.temporal_rgba8(tp, dn, False)]
        for k, (a, b) in enumerate(zip(got, want)):
            assert _same(a, b), (f, k)
    one.render_spp(2); plain.render_spp(2)                  # more samples at the same pose: the prior is kept
    assert _same(one.read_temporal(), plain.read_temporal())  # NULL parameters: the defaults
    one.reset_temporal(); plain.reset_temporal()
    assert _same(one.read_temporal(tp, dn), plain.read_temporal(tp, dn))


def test_group_errors_leave_the_history_untouched(one, plain, scenes):
    w, h = 64, 48
    cams = [_setup(t, scenes["Scene1"], w, h) for t in (one, plain)]
    for t, cam in zip((one, plain), cams):
        t.render_spp(2); t.read_temporal()
        _move(cam, 0.5); t.set_camera(cam); t.reset_accumulation(); t.render_spp(1)
    lib, g = one.lib, one.g
    out = np.zeros((h, w, 4), np.float32)
    surf = np.zeros((h, w), np.uint32)
    P = lambda a: a.ctypes.data_as(C.c_void_p)

    def invalid(rc, fn):
        assert rc == rtb200.RT_ERR_INVALID
        msg = lib.rt_group_last_error(g).decode()
        assert msg.startswith("member 0 (device 0): " + fn + ": "), msg

    inf, nan = float("inf"), float("nan")
    bad_dn = [dict(passes=-1), dict(passes=9), dict(normal_power=0), dict(normal_power=3), dict(normal_power=512), dict(normal_power=-2),
              dict(sigma_color=0.0), dict(sigma_color=-1.0), dict(sigma_color=inf), dict(sigma_color=nan),
              dict(sigma_depth=0.0), dict(sigma_depth=-1.0), dict(sigma_depth=inf), dict(sigma_depth=nan)]
    for kw in bad_dn:
        d = rtb200.default_denoise_params(**kw)
        invalid(lib.rt_group_read_denoised(g, C.byref(d), P(out)), "rt_group_read_denoised")
        invalid(lib.rt_group_denoise_rgba8(g, C.byref(d), P(surf), w * 4, 1), "rt_group_denoise_rgba8")
        invalid(lib.rt_group_read_temporal(g, None, C.byref(d), P(out)), "rt_group_read_temporal")
        invalid(lib.rt_group_temporal_rgba8(g, None, C.byref(d), P(surf), w * 4, 1), "rt_group_temporal_rgba8")
    bad_tp = [dict(max_history=0), dict(max_history=-1), dict(max_history=4097), dict(tau_depth=0.0), dict(tau_depth=-1.0), dict(tau_depth=inf),
              dict(tau_depth=nan), dict(tau_normal=nan), dict(tau_normal=inf), dict(tau_normal=-inf), dict(tau_normal=1.01), dict(tau_normal=-1.01)]
    for kw in bad_tp:
        p = rtb200.default_temporal_params(**kw)
        invalid(lib.rt_group_read_temporal(g, C.byref(p), None, P(out)), "rt_group_read_temporal")
        invalid(lib.rt_group_temporal_rgba8(g, C.byref(p), None, P(surf), w * 4, 1), "rt_group_temporal_rgba8")
    for fn in ("rt_group_denoise_rgba8", "rt_group_temporal_rgba8"):
        args = (None,) if fn == "rt_group_denoise_rgba8" else (None, None)
        invalid(getattr(lib, fn)(g, *args, None, w * 4, 1), fn)                      # NULL output
        invalid(getattr(lib, fn)(g, *args, P(surf), w * 4 - 4, 1), fn)               # a pitch shorter than a row
    invalid(lib.rt_group_read_denoised(g, None, None), "rt_group_read_denoised")
    invalid(lib.rt_group_read_temporal(g, None, None, None), "rt_group_read_temporal")
    # the history is the one of the last good call: the next call is what it would have been
    assert _same(one.read_temporal(), plain.read_temporal())
    assert _same(one.read_temporal(dn=rtb200.default_denoise_params()), plain.read_temporal(dn=rtb200.default_denoise_params()))


def test_group_calls_are_read_only(one, scenes):
    w, h = 160, 120
    cam = _setup(one, scenes["Scene3_indirect"], w, h)
    one.render_spp(2); one.read_temporal()
    _move(cam, 0.3); one.set_camera(cam); one.reset_accumulation(); one.render_spp(3)
    acc0, n0 = one.members[0].read_accum()
    st0 = one.stats()
    surf0 = one.resolve_rgba8()
    one.read_denoised(); one.denoise_rgba8(rtb200.default_denoise_params(passes=2))
    one.read_temporal(); one.temporal_rgba8(dn=rtb200.default_denoise_params())
    acc1, n1 = one.members[0].read_accum()
    st1 = one.stats()
    assert _same(acc0, acc1) and n0 == n1 == 3
    assert (st0.samples, st0.paths, st0.segments) == (st1.samples, st1.paths, st1.segments)
    assert np.array_equal(surf0, one.resolve_rgba8())


# ---- two or more GPUs: the group against its twin ------------------------------------------------------------------------------
def test_group_without_filtering_is_the_fused_resolve(multi, scenes):
    n = multi.size()
    w, h = 161, 97
    _setup(multi, scenes["Scene1"], w, h)
    multi.render_spp(2 * n + 1)
    for flip in (True, False):
        want = multi.resolve_rgba8(flip)
        assert np.array_equal(multi.denoise_rgba8(rtb200.default_denoise_params(passes=0), flip_y=flip), want), flip
        multi.reset_temporal()
        assert np.array_equal(multi.temporal_rgba8(flip_y=flip), want), flip      # no history: the plain resolve
    p = multi.params
    p.mode = rtb200.RT_MODE_PREVIEW
    multi.set_params(p)
    multi.render_spp(1)
    for flip in (True, False):
        want = multi.resolve_rgba8(flip)
        assert np.array_equal(multi.denoise_rgba8(flip_y=flip), want), ("preview", flip)
        assert np.array_equal(multi.temporal_rgba8(dn=rtb200.default_denoise_params(), flip_y=flip), want), ("preview", flip)
    # members that differ in resolution are refused before anything runs
    m1 = multi.members[1]
    m1.set_params(rtb200.default_params(width=w + 1, height=h, mode=rtb200.RT_MODE_PATH))
    try:
        surf = np.zeros((h, w), np.uint32)
        rc = multi.lib.rt_group_denoise_rgba8(multi.g, None, surf.ctypes.data_as(C.c_void_p), w * 4, 1)
        assert rc == rtb200.RT_ERR_INVALID and "members differ in resolution" in multi.lib.rt_group_last_error(multi.g).decode()
    finally:
        multi.set_params(multi.params)


@pytest.mark.parametrize("scene", ["Scene1", "Scene3_indirect"])
def test_group_denoise_is_the_twin(multi, plain, scenes, scene):
    n = multi.size()
    w, h = 161, 97
    for t in (multi, plain):
        _setup(t, scenes[scene], w, h)
    multi.render_spp(2 * n + 1)                              # does not divide by the device count: members hold different counts
    counts = [m.read_accum()[1] for m in multi.members]
    assert len(set(counts)) > 1
    _feed(plain, multi)
    for passes in (1, 5):
        dn = rtb200.default_denoise_params(passes=passes)
        assert _same(multi.read_denoised(dn), plain.read_denoised(dn)), passes
        for flip in (True, False):
            assert np.array_equal(multi.denoise_rgba8(dn, flip_y=flip), plain.denoise_rgba8(dn, flip_y=flip)), (passes, flip)
    assert _same(multi.read_denoised(), plain.read_denoised())


@pytest.mark.parametrize("scene", ["Scene1", "Scene3_indirect"])
def test_group_temporal_along_a_turning_camera_is_the_twin(multi, plain, scenes, scene):
    n = multi.size()
    w, h = 161, 97
    tp = rtb200.default_temporal_params()
    dn = rtb200.default_denoise_params(passes=3)
    cam = _setup(multi, scenes[scene], w, h)
    _setup(plain, scenes[scene], w, h)
    hist = hid = hnt = prev_pose = None
    for f in range(5):
        if f:
            _move(cam, 0.4, 0.01 * (f & 1))
        multi.set_camera(cam); multi.reset_accumulation(); multi.render_spp(n + 1)
        plain.set_camera(cam)
        _feed(plain, multi)
        got = [multi.read_temporal(tp), multi.read_temporal(tp, dn), multi.temporal_rgba8(tp, None, True), multi.temporal_rgba8(tp, dn, False)]
        want = [plain.read_temporal(tp), plain.read_temporal(tp, dn), plain.temporal_rgba8(tp, None, True), plain.temporal_rgba8(tp, dn, False)]
        for k, (a, b) in enumerate(zip(got, want)):
            assert _same(a, b), (f, k)
        ids, nt = _guides(plain)
        pose = ref.pose_of_camera(cam, w, h)
        if f == 4:
            P = ref.reproject(pose, prev_pose, ids, nt, hist, hid, hnt, CAP, TZ, TN)
        hist, hid, hnt, prev_pose = got[0], ids, nt, pose
    assert (P[..., 3] > 0).sum() > 0.5 * (hid >= 0).sum()
    # samples added without a move: the group keeps its prior (the twin cannot follow: rt_write_accum restarts its epoch)
    multi.render_spp(n)
    S, N = _rank_sum(multi)
    got = multi.read_temporal(tp)
    want = ref.output(S, N, hid, P)
    np.testing.assert_allclose(got[..., :3], want[..., :3], rtol=1e-5, atol=0)
    np.testing.assert_allclose(got[..., 3], want[..., 3], rtol=1e-6, atol=0)
    assert (got[..., 3] > N).sum() > 0.5 * (hid >= 0).sum()


def test_group_resolve_after_a_filtered_call_is_still_the_rank_order_sum(multi, scenes, oracle):
    n = multi.size()
    w, h, spp = 320, 200, 2 * n + 1
    _setup(multi, scenes["Scene3_indirect"], w, h)
    multi.render_spp(spp)
    for call in ("denoise", "temporal"):
        if call == "denoise":
            multi.denoise_rgba8()
        else:
            multi.temporal_rgba8(dn=rtb200.default_denoise_params())
        # nothing of the filtered call may still read a member's buffer when the next render writes it
        multi.reset_accumulation(); multi.render_spp(spp)
        surf = multi.resolve_rgba8()
        S, N = _rank_sum(multi)
        assert N == spp
        assert np.array_equal(surf, oracle.resolve_argb8(S, N)), call
