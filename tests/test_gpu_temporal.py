"""GPU: the temporal resolve (rt_temporal_rgba8 / rt_read_temporal / rt_reset_temporal; kernel in csrc/rt_temporal.cu, filter in its
per-pixel count form in csrc/rt_denoise.cu) against the float32 numpy reference (tests/temporal_reference.py) after camera moves,
bit-identity with the plain and denoised resolves wherever there is no history, the copy of an identical pose, no bleeding across
object ids, read-only behaviour, image quality along a turning camera, parameter errors and the C++ host driver."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

import rtb200
from conftest import ROOT, SEED
import temporal_reference as ref
from denoise_reference import mean_of, psnr

pytestmark = pytest.mark.gpu

CAP, TZ, TN = 32, 0.02, 0.9


@pytest.fixture(scope="module")
def tt():
    """A context of its own: these tests switch options and shards and leave them at their defaults afterwards."""
    t = rtb200.PathTracer(0)
    yield t
    t.close()


def _camera(name):
    cam = rtb200.default_camera(55)
    if name == "mesh":
        cam.pos[1] = 1.5; cam.pos[2] = -1.0
    return cam


def _setup(t, scenes, name, w, h, seed=SEED, max_bounces=8, mode=rtb200.RT_MODE_PATH):
    if name == "mesh":
        from rtb200.scenes import heightfield_mesh, mesh_scene
        t.set_scene(mesh_scene())
        v, tr = heightfield_mesh(24, 16, seed=3)
        t.set_mesh(0, v, tr)
    else:
        t.set_scene(scenes[name])
    cam = _camera(name)
    t.set_camera(cam)
    t.set_params(rtb200.default_params(width=w, height=h, mode=mode, max_bounces=max_bounces, seed_lo=seed[0], seed_hi=seed[1]))
    t.reset_accumulation()
    return cam


def _move(cam, yaw_deg, dx=0.0):
    rtb200.rotate_camera(cam, yaw_deg * math.pi / 180.0, [cam.up[0], cam.up[1], cam.up[2]])
    cam.pos[0] += dx
    return cam


def _guides(t):
    ids, tt_, nrm, _ = t.read_aov()
    return ids, np.concatenate([nrm, tt_[..., None]], -1)


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _tp(**kw):
    return rtb200.default_temporal_params(**kw)


def _plain_checks(t, dn):
    """The temporal calls without a history give exactly the plain / denoised resolves: every call here first drops the history."""
    w, h = t.params.width, t.params.height
    for flip in (True, False):
        t.reset_temporal()
        assert np.array_equal(t.temporal_rgba8(flip_y=flip), t.resolve_rgba8(flip)), flip
        surf, owner = rtb200.host_surface(w, h)
        t.reset_temporal()
        t.temporal_rgba8(flip_y=flip, out=surf)
        assert np.array_equal(surf, t.resolve_rgba8(flip)), ("pinned", flip)
        del owner
        t.reset_temporal()
        assert np.array_equal(t.temporal_rgba8(dn=dn, flip_y=flip), t.denoise_rgba8(dn, flip_y=flip)), ("filtered", flip)
    t.reset_temporal()
    assert np.array_equal(_bits(t.read_temporal()[..., :3]), _bits(t.read_denoised(rtb200.default_denoise_params(passes=0))[..., :3]))
    t.reset_temporal()
    assert np.array_equal(_bits(t.read_temporal(dn=dn)[..., :3]), _bits(t.read_denoised(dn)[..., :3]))


def _blended(t):
    """True when the last history call blended some prior in (its output differs from the plain mean)."""
    acc, n = t.read_accum()
    got = t.read_temporal()
    return not np.array_equal(_bits(got[..., :3]), _bits(mean_of(acc, n)))


def test_without_history_the_output_is_the_plain_resolve(tt, scenes):
    w, h = 160, 120
    dn = rtb200.default_denoise_params(passes=4)
    cam = _setup(tt, scenes, "Scene1", w, h)
    tt.render_spp(4)
    # the first call ever on this context, then every other way of having no history
    acc, n = tt.read_accum()
    first = tt.read_temporal()
    assert np.array_equal(_bits(first[..., :3]), _bits(mean_of(acc, n))) and (first[..., 3] == 4).all()
    _plain_checks(tt, dn)

    def primed():
        """A history at the current pose, then a moved camera with one sample: the next call blends."""
        tt.read_temporal()
        _move(cam, 0.3); tt.set_camera(cam); tt.reset_accumulation(); tt.render_spp(1)

    primed()
    assert _blended(tt)
    # seed and pixel step changes keep the history
    for change in ("seed", "step"):
        tt.read_temporal()
        if change == "seed":
            tt.set_params(rtb200.default_params(width=w, height=h, mode=rtb200.RT_MODE_PATH, max_bounces=8, seed_lo=5, seed_hi=6))
        else:
            tt.set_pixel_step(2)
        _move(cam, 0.3); tt.set_camera(cam); tt.reset_accumulation(); tt.render_spp(1)
        assert _blended(tt), change
        tt.set_pixel_step(1)
    # scene, radiance parameters, resize: dropped
    for change in ("scene", "sky", "bounces", "resize"):
        primed()
        if change == "scene":
            tt.set_scene(scenes["Scene1"])
        elif change == "sky":
            p = tt.params; p.sky[0] = p.sky[0] + 0.25; tt.set_params(p)
        elif change == "bounces":
            p = tt.params; p.max_bounces = 7; tt.set_params(p)
        else:
            tt.set_params(rtb200.default_params(width=w + 1, height=h - 1, mode=rtb200.RT_MODE_PATH, max_bounces=8, seed_lo=SEED[0], seed_hi=SEED[1]))
        tt.reset_accumulation(); tt.render_spp(2)
        acc, n = tt.read_accum()
        got = tt.read_temporal()
        assert np.array_equal(_bits(got[..., :3]), _bits(mean_of(acc, n))), change
        _plain_checks(tt, dn)
        _setup(tt, scenes, "Scene1", w, h); cam = _camera("Scene1"); tt.render_spp(4)
    # preview: the plain resolve, and the history is dropped
    primed()
    p = tt.params; p.mode = rtb200.RT_MODE_PREVIEW; tt.set_params(p)
    tt.render_spp(1)
    for flip in (True, False):
        assert np.array_equal(tt.temporal_rgba8(flip_y=flip), tt.resolve_rgba8(flip))
        assert np.array_equal(tt.temporal_rgba8(dn=dn, flip_y=flip), tt.resolve_rgba8(flip))


@pytest.mark.parametrize("scene", ["Scene1", "Scene2", "Scene_indirect", "mesh"])
@pytest.mark.parametrize("accel", [rtb200.RT_ACCEL_FLAT, rtb200.RT_ACCEL_BVH])
@pytest.mark.parametrize("size", [(160, 120), (161, 97)])
def test_read_temporal_matches_the_reference_after_camera_moves(tt, scenes, scene, accel, size):
    w, h = size
    tt.set_option(rtb200.RT_OPT_ACCEL, accel)
    dn = rtb200.default_denoise_params(passes=3)
    try:
        cam = _setup(tt, scenes, scene, w, h)
        tt.render_spp(4)
        prev_pose = ref.pose_of_camera(cam, w, h)
        hid, hnt = _guides(tt)
        assert (hid >= 0).mean() > 0.2
        hist = tt.read_temporal()
        blended = 0
        for k, (yaw, dx) in enumerate(((0.4, 0.0), (-0.3, 0.02), (0.0, -0.03))):
            _move(cam, yaw, dx); tt.set_camera(cam)
            tt.reset_accumulation(); tt.render_spp(1 + k)
            acc, n = tt.read_accum()
            ids, nt = _guides(tt)
            pose = ref.pose_of_camera(cam, w, h)
            assert np.array_equal(_bits(ref.ray_dirs(pose, w, h)), _bits(tt.read_ray_dirs()))
            got = tt.read_temporal()
            P = ref.reproject(pose, prev_pose, ids, nt, hist, hid, hnt, CAP, TZ, TN)
            want = ref.output(acc, n, ids, P)
            np.testing.assert_allclose(got[..., :3], want[..., :3], rtol=1e-5, atol=0, err_msg=str(k))
            np.testing.assert_allclose(got[..., 3], want[..., 3], rtol=1e-6, atol=0, err_msg=str(k))
            blended += int((P[..., 3] > 0).sum())
            # the same prior (same epoch and pose) with the filter in front
            got_f = tt.read_temporal(dn=dn)
            want_f = ref.filter(got, ids, nt, dn.passes, dn.normal_power, dn.sigma_color, dn.sigma_depth)
            np.testing.assert_allclose(got_f[..., :3], want_f, rtol=1e-5, atol=1e-6 * float(want_f.max()), err_msg=str(k))
            np.testing.assert_array_equal(got_f[..., 3], got[..., 3])
            # the ARGB8 path is the pack of the same values
            argb = tt.temporal_rgba8(flip_y=False)
            tt.write_accum(got, 0)
            assert np.array_equal(argb, tt.resolve_rgba8(False))
            tt.write_accum(acc, n)
            hist, hid, hnt, prev_pose = tt.read_temporal(), ids, nt, pose
        assert blended > 0.5 * (hid >= 0).sum()
        assert tt.stats().last_resolve_ms > 0
    finally:
        tt.set_option(rtb200.RT_OPT_ACCEL, rtb200.RT_ACCEL_AUTO)


def test_reset_at_the_same_pose_copies_the_last_output(tt, scenes):
    w, h = 161, 97
    for cap in (32, 3):
        _setup(tt, scenes, "Scene_indirect", w, h)
        tt.render_spp(6)
        tp = _tp(max_history=cap)
        last = tt.read_temporal(tp)
        tt.reset_accumulation(); tt.render_spp(1)
        acc, n = tt.read_accum()
        ids, _ = _guides(tt)
        got = tt.read_temporal(tp)
        want = ref.output(acc, n, ids, ref.copy_prior(last, cap))
        assert np.array_equal(_bits(got), _bits(want)), cap
        hit = ids >= 0
        assert (got[hit][:, 3] == 1 + min(6, cap)).all()


@pytest.mark.parametrize("scene", ["Scene1", "mesh"])
def test_no_colour_crosses_an_object_id(tt, scenes, scene):
    w, h = 161, 97
    cam = _setup(tt, scenes, scene, w, h)
    rng = np.random.default_rng(11)
    pal = None
    for k in range(3):
        ids, _ = _guides(tt)
        if pal is None:
            pal = rng.uniform(0.0, 40.0, (int(ids.max()) + 64, 3)).astype(np.float32)
        mean = pal[ids + 1]
        buf = np.zeros((h, w, 4), np.float32)
        buf[..., :3] = mean * np.float32(2)
        tt.write_accum(buf, 2)
        for dn in (None, rtb200.default_denoise_params()):
            got = tt.read_temporal(dn=dn)
            np.testing.assert_allclose(got[..., :3], mean, rtol=1e-6, atol=0, err_msg=str((k, dn is None)))
        _move(cam, 0.5, 0.01); tt.set_camera(cam)


def test_temporal_is_read_only(tt, scenes):
    w, h = 160, 120
    cam = _setup(tt, scenes, "Scene_indirect", w, h)
    tt.render_spp(4)
    tt.read_temporal()
    _move(cam, 0.3); tt.set_camera(cam); tt.reset_accumulation(); tt.render_spp(2)
    acc0, n0 = tt.read_accum()
    st0 = tt.stats()
    a = tt.read_temporal()
    tt.temporal_rgba8(dn=rtb200.default_denoise_params(passes=3))
    acc1, n1 = tt.read_accum()
    st1 = tt.stats()
    assert np.array_equal(_bits(acc0), _bits(acc1)) and n0 == n1 == st1.samples == 2
    assert (st0.segments, st0.paths, st0.traced_segments) == (st1.segments, st1.paths, st1.traced_segments)
    # primary reuse off: the renders never build the cache; the temporal call traces it once (and counts the queries)
    tt.set_option(rtb200.RT_OPT_PRIMARY_REUSE, 0)
    try:
        cam = _setup(tt, scenes, "Scene_indirect", w, h)
        tt.render_spp(4)
        tt.read_temporal()
        _move(cam, 0.3); tt.set_camera(cam); tt.reset_accumulation(); tt.render_spp(2)
        st2 = tt.stats()
        b = tt.read_temporal()
        st3 = tt.stats()
        assert np.array_equal(_bits(a), _bits(b))
        assert st3.traced_segments - st2.traced_segments == w * h
        assert (st3.segments, st3.paths) == (st2.segments, st2.paths)
        tt.read_temporal()
        assert tt.stats().traced_segments == st3.traced_segments
    finally:
        tt.set_option(rtb200.RT_OPT_PRIMARY_REUSE, 1)


def _turning_camera_run(t, scenes, scene, w, h, frames, yaw_deg, tp, dn):
    """The host loop of a fly-through: per frame the camera turns, the accumulation restarts and one sample is traced, then the
    temporal call presents. Returns the final frame as (raw 1 spp, temporal, filter alone, temporal + filter) means and the camera."""
    cam = _setup(t, scenes, scene, w, h)
    for f in range(frames):
        if f:
            _move(cam, yaw_deg); t.set_camera(cam)
        t.reset_accumulation(); t.render_spp(1)
        tem = t.read_temporal(tp)[..., :3]
    raw = t.read_denoised(rtb200.default_denoise_params(passes=0))[..., :3]
    return raw, tem, t.read_denoised(dn)[..., :3], t.read_temporal(tp, dn)[..., :3], cam


def test_quality_along_a_turning_camera(tt, scenes):
    """160x120, depth 8, 16 frames turning 0.25 degrees each, 1 spp per frame: tonemapped PSNR of the last frame against 4096 spp of
    another seed at the final pose. Temporal at least 3 dB above raw; temporal + filter no worse than the filter alone."""
    w, h = 160, 120
    dn = rtb200.default_denoise_params()
    rows = []
    for scene in ("Scene1", "Scene2", "Scene_indirect", "Scene1_reflection"):
        raw, tem, den, both, cam = _turning_camera_run(tt, scenes, scene, w, h, 16, 0.25, _tp(), dn)
        _setup(tt, scenes, scene, w, h, seed=(0x5EED, 0xF00D))
        tt.set_camera(cam)
        tt.render_spp(4096)
        gt = tt.read_denoised(rtb200.default_denoise_params(passes=0))[..., :3]
        rows.append((scene, psnr(raw, gt), psnr(tem, gt), psnr(den, gt), psnr(both, gt)))
        print("%s: raw 1 spp %.2f dB, temporal %.2f dB, filter %.2f dB, temporal + filter %.2f dB" % rows[-1])
    for scene, p_raw, p_tem, p_den, p_both in rows:
        if scene == "Scene1_reflection":
            continue
        assert p_tem >= p_raw + 3.0, scene
        assert p_both >= p_den, scene


def test_invalid_parameters(tt, scenes):
    _setup(tt, scenes, "Scene1", 64, 48)
    tt.render_spp(1)
    lib = tt.lib
    out = np.zeros((48, 64, 4), np.float32)
    surf = np.zeros((48, 64), np.uint32)
    inf, nan = float("inf"), float("nan")
    bad = [dict(max_history=0), dict(max_history=-1), dict(max_history=4097), dict(tau_depth=0.0), dict(tau_depth=-1.0), dict(tau_depth=inf),
           dict(tau_depth=nan), dict(tau_normal=nan), dict(tau_normal=inf), dict(tau_normal=-inf), dict(tau_normal=1.01), dict(tau_normal=-1.01)]
    for kw in bad:
        p = _tp(**kw)
        assert lib.rt_read_temporal(tt.h, C.byref(p), None, out.ctypes.data_as(C.c_void_p)) == rtb200.RT_ERR_INVALID, kw
        assert lib.rt_temporal_rgba8(tt.h, C.byref(p), None, surf.ctypes.data_as(C.c_void_p), 64 * 4, 1) == rtb200.RT_ERR_INVALID, kw
    for kw in (dict(passes=9), dict(normal_power=3), dict(sigma_color=nan), dict(sigma_depth=0.0)):
        d = rtb200.default_denoise_params(**kw)
        assert lib.rt_read_temporal(tt.h, None, C.byref(d), out.ctypes.data_as(C.c_void_p)) == rtb200.RT_ERR_INVALID, kw
    for kw in (dict(max_history=1), dict(max_history=4096), dict(tau_normal=-1.0), dict(tau_normal=1.0), dict(tau_depth=1e-30)):
        tt.read_temporal(_tp(**kw))
    tt.set_shard(0, 2)
    try:
        assert lib.rt_read_temporal(tt.h, None, None, out.ctypes.data_as(C.c_void_p)) == rtb200.RT_ERR_INVALID
        assert lib.rt_temporal_rgba8(tt.h, None, None, surf.ctypes.data_as(C.c_void_p), 64 * 4, 1) == rtb200.RT_ERR_INVALID
    finally:
        tt.set_shard(0, 1)
    tt.read_temporal()


def _read_ppm(path):
    with open(path, "rb") as f:
        assert f.readline().strip() == b"P6"
        w, h = [int(x) for x in f.readline().split()]
        assert f.readline().strip() == b"255"
        return np.frombuffer(f.read(), np.uint8).reshape(h, w, 3)


def test_headless_temporal_matches_the_python_sequence(tt, scenes, tmp_path):
    exe = os.path.join(ROOT, "software-raytracer_b200", "bin", "rt_headless")
    if not os.path.exists(exe):
        pytest.skip("bin/rt_headless not built")
    scene_file = str(tmp_path / "Scene1.json")
    assert rtb200.scene_file_write(scene_file, scenes["Scene1"], None, "Scene1") == 0
    w, h, frames, orbit = 160, 120, 12, 0.5
    for passes in (0, 3):
        ppm = str(tmp_path / ("t%d.ppm" % passes))
        args = [exe, "--scene", scene_file, "--width", str(w), "--height", str(h), "--interactive", str(frames), "--orbit", str(orbit),
                "--temporal", "32", "--scale", "1", "--out", ppm] + (["--denoise", str(passes)] if passes else [])
        r = subprocess.run(args, capture_output=True, text=True, timeout=300)
        assert r.returncode == 0 and '"p50_ms"' in r.stdout, r.stdout + r.stderr
        img = _read_ppm(ppm)
        # the same calls through Python: Raytracer::RenderFrame of every frame (10 warm-up frames included)
        tt.set_scene(scenes["Scene1"])
        tt.reset_temporal()
        par = rtb200.default_params(width=w, height=h, mode=rtb200.RT_MODE_PATH, max_bounces=8, selected_id=-1)
        cam = rtb200.default_camera(55)
        tp = _tp(max_history=32)
        dn = rtb200.default_denoise_params(passes=passes) if passes else None
        angle = C.c_float(orbit * math.pi / 180.0).value
        for f in range(frames + 10):
            rtb200.rotate_camera(cam, angle, [cam.up[0], cam.up[1], cam.up[2]])
            tt.set_params(par); tt.set_camera(cam); tt.reset_accumulation()
            tt.set_pixel_step(rtb200.reference_pixel_step(1.0, 1.0), rtb200.reference_strip_columns(w))
            tt.render_spp(1)
            argb = tt.temporal_rgba8(tp, dn, True)
        tt.set_pixel_step(1)
        want = np.stack([(argb >> 16) & 255, (argb >> 8) & 255, argb & 255], -1).astype(np.uint8)
        assert np.array_equal(img, want), passes
        assert not np.array_equal(argb, tt.resolve_rgba8(True))
    # the multi-GPU group has no temporal resolve: refused with a message, whatever the device count
    r = subprocess.run([exe, "--scene", scene_file, "--gpus", "2", "--temporal", "8"], capture_output=True, text=True, timeout=300)
    assert r.returncode != 0 and "--temporal" in r.stderr
