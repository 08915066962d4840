"""GPU: the denoised resolve (rt_denoise_rgba8 / rt_read_denoised; kernels in csrc/rt_denoise.cu) against the float32 numpy
reference (tests/denoise_reference.py), its ARGB8 path against the plain pack, bit-identity where nothing is filtered, no bleeding
across object ids, read-only behaviour, image quality against a 4096-spp render, parameter errors and the C++ host driver."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import rtb200
from conftest import ROOT, SEED
import denoise_reference as ref

pytestmark = pytest.mark.gpu

DN_SCENES = ["Scene1", "Scene2", "Scene_indirect", "Scene1_reflection", "mesh"]


@pytest.fixture(scope="module")
def dn():
    """A context of its own: these tests switch options (back end, primary reuse) and leave them at their defaults afterwards."""
    t = rtb200.PathTracer(0)
    yield t
    t.close()


def _setup(t, scenes, name, w, h, seed=SEED, max_bounces=8, mode=rtb200.RT_MODE_PATH):
    cam = rtb200.default_camera(55)
    if name == "mesh":
        from rtb200.scenes import heightfield_mesh, mesh_scene
        cam.pos[1] = 1.5; cam.pos[2] = -1.0
        t.set_scene(mesh_scene())
        v, tr = heightfield_mesh(24, 16, seed=3)
        t.set_mesh(0, v, tr)
    else:
        t.set_scene(scenes[name])
    t.set_camera(cam)
    t.set_params(rtb200.default_params(width=w, height=h, mode=mode, max_bounces=max_bounces, seed_lo=seed[0], seed_hi=seed[1]))
    t.reset_accumulation()


def _guides(t):
    ids, tt, nrm, _ = t.read_aov()
    return ids, np.concatenate([nrm, tt[..., None]], -1)


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


@pytest.mark.parametrize("scene", DN_SCENES)
@pytest.mark.parametrize("accel", [rtb200.RT_ACCEL_FLAT, rtb200.RT_ACCEL_BVH])
@pytest.mark.parametrize("size", [(160, 120), (161, 97)])
def test_read_denoised_matches_the_reference(dn, scenes, scene, accel, size):
    w, h = size
    dn.set_option(rtb200.RT_OPT_ACCEL, accel)
    try:
        _setup(dn, scenes, scene, w, h)
        ids, nt = _guides(dn)
        assert (ids >= 0).mean() > 0.2
        done = 0
        for spp in (1, 4, 64):
            dn.render_spp(spp - done); done = spp
            acc, n = dn.read_accum()
            assert n == spp
            for passes in (1, 3, 5):
                for prm in (rtb200.default_denoise_params(passes=passes), rtb200.default_denoise_params(passes=passes, normal_power=16, sigma_color=0.5, sigma_depth=2.0)):
                    got = dn.read_denoised(prm)
                    want = ref.denoise(acc, n, ids, nt, passes, prm.normal_power, prm.sigma_color, prm.sigma_depth)
                    np.testing.assert_allclose(got[..., :3], want, rtol=1e-4, atol=1e-5 * float(want.max()), err_msg=str((spp, passes)))
                    assert not got[..., 3].any()
            assert dn.stats().last_resolve_ms > 0
    finally:
        dn.set_option(rtb200.RT_OPT_ACCEL, rtb200.RT_ACCEL_AUTO)


def test_block_filled_frames_are_filtered_with_per_pixel_guides(dn, scenes):
    _setup(dn, scenes, "Scene1", 161, 97)
    dn.set_pixel_step(2)
    try:
        dn.render_spp(4)
        acc, n = dn.read_accum()
        ids, nt = _guides(dn)
        prm = rtb200.default_denoise_params(passes=3)
        got = dn.read_denoised(prm)
        want = ref.denoise(acc, n, ids, nt, prm.passes, prm.normal_power, prm.sigma_color, prm.sigma_depth)
        np.testing.assert_allclose(got[..., :3], want, rtol=1e-4, atol=1e-5 * float(want.max()))
        argb = dn.denoise_rgba8(rtb200.default_denoise_params(passes=3))
        assert not np.array_equal(argb, dn.resolve_rgba8())
    finally:
        dn.set_pixel_step(1)


def test_argb_path_is_the_float_path_plus_the_plain_pack(dn, scenes):
    w, h = 161, 97
    _setup(dn, scenes, "Scene_indirect", w, h)
    dn.render_spp(4)
    prm = rtb200.default_denoise_params(passes=4)
    mean = dn.read_denoised(prm)
    outs = {}
    for flip in (True, False):
        outs[(flip, "pageable")] = dn.denoise_rgba8(prm, flip_y=flip).copy()
        surf, owner = rtb200.host_surface(w, h)
        dn.denoise_rgba8(prm, flip_y=flip, out=surf)
        outs[(flip, "pinned")] = surf.copy()
        del owner
    dn.write_accum(mean, 0)
    for flip in (True, False):
        plain = dn.resolve_rgba8(flip)
        for kind in ("pageable", "pinned"):
            assert np.array_equal(outs[(flip, kind)], plain), (flip, kind)


def test_bit_identity_where_nothing_is_filtered(dn, scenes):
    w, h = 160, 120
    _setup(dn, scenes, "Scene1", w, h)
    dn.render_spp(4)
    ids, _ = _guides(dn)
    plain = dn.resolve_rgba8(True)
    den = dn.denoise_rgba8(rtb200.default_denoise_params(passes=5), flip_y=True)
    sky = (ids < 0)[::-1]                                      # the surface is y-down
    assert sky.any() and np.array_equal(den[sky], plain[sky])
    assert not np.array_equal(den[~sky], plain[~sky])
    acc, n = dn.read_accum()
    mean = dn.read_denoised()
    assert np.array_equal(_bits(mean[ids < 0][:, :3]), _bits(ref.mean_of(acc, n)[ids < 0]))
    for flip in (True, False):
        assert np.array_equal(dn.denoise_rgba8(rtb200.default_denoise_params(passes=0), flip_y=flip), dn.resolve_rgba8(flip))
    assert np.array_equal(_bits(dn.read_denoised(rtb200.default_denoise_params(passes=0))[..., :3]), _bits(ref.mean_of(acc, n)))
    # preview: nothing random to filter
    _setup(dn, scenes, "Scene1", w, h, mode=rtb200.RT_MODE_PREVIEW)
    dn.render_spp(1)
    for flip in (True, False):
        assert np.array_equal(dn.denoise_rgba8(None, flip_y=flip), dn.resolve_rgba8(flip))


@pytest.mark.parametrize("scene", ["Scene1", "mesh"])
def test_no_colour_crosses_an_object_id(dn, scenes, scene):
    w, h = 161, 97
    _setup(dn, scenes, scene, w, h)
    ids, _ = _guides(dn)
    rng = np.random.default_rng(11)
    pal = rng.uniform(0.0, 40.0, (int(ids.max()) + 2, 3)).astype(np.float32)
    mean = pal[ids + 1]
    for samples in (0, 4):
        buf = np.zeros((h, w, 4), np.float32)
        buf[..., :3] = mean * np.float32(samples) if samples else mean
        dn.write_accum(buf, samples)
        got = dn.read_denoised(rtb200.default_denoise_params(passes=5))
        np.testing.assert_allclose(got[..., :3], mean, rtol=1e-6, atol=0)


def test_denoise_is_read_only(dn, scenes):
    w, h = 160, 120
    _setup(dn, scenes, "Scene_indirect", w, h)
    dn.render_spp(4)
    acc0, n0 = dn.read_accum()
    st0 = dn.stats()
    a = dn.read_denoised()
    dn.denoise_rgba8(rtb200.default_denoise_params(passes=3))
    acc1, n1 = dn.read_accum()
    st1 = dn.stats()
    assert np.array_equal(_bits(acc0), _bits(acc1)) and n0 == n1 == st1.samples == 4
    assert (st0.segments, st0.paths) == (st1.segments, st1.paths)
    dn.render_spp(4)
    with_dn, _ = dn.read_accum()
    _setup(dn, scenes, "Scene_indirect", w, h)
    dn.render_spp(4); dn.render_spp(4)
    without, _ = dn.read_accum()
    assert np.array_equal(_bits(with_dn), _bits(without))
    # primary reuse off: the renders never build the cache; the denoiser traces it (and counts the queries)
    dn.set_option(rtb200.RT_OPT_PRIMARY_REUSE, 0)
    try:
        _setup(dn, scenes, "Scene_indirect", w, h)
        dn.render_spp(4)
        st2 = dn.stats()
        b = dn.read_denoised()
        st3 = dn.stats()
        assert np.array_equal(_bits(a), _bits(b))
        assert st3.traced_segments - st2.traced_segments == w * h
        assert (st3.segments, st3.paths) == (st2.segments, st2.paths)
    finally:
        dn.set_option(rtb200.RT_OPT_PRIMARY_REUSE, 1)


def test_quality_against_4096_spp(dn, scenes):
    """160x120, depth 8: 4 spp denoised at least 3 dB above raw (tonemapped PSNR against 4096 spp of another seed), and a
    4096-spp image is moved no further from that ground truth than 1.05x the raw one's RMSE."""
    w, h = 160, 120
    rows = []
    for scene in ("Scene1", "Scene2", "Scene_indirect"):
        _setup(dn, scenes, scene, w, h, seed=(0x5EED, 0xF00D))
        dn.render_spp(4096)
        gt = dn.read_denoised(rtb200.default_denoise_params(passes=0))[..., :3]
        _setup(dn, scenes, scene, w, h)
        dn.render_spp(4)
        raw4 = dn.read_denoised(rtb200.default_denoise_params(passes=0))[..., :3]
        den4 = dn.read_denoised()[..., :3]
        dn.render_spp(4092)
        raw_hi = dn.read_denoised(rtb200.default_denoise_params(passes=0))[..., :3]
        den_hi = dn.read_denoised()[..., :3]
        p_raw, p_den = ref.psnr(raw4, gt), ref.psnr(den4, gt)
        rmse = lambda x: float(np.sqrt(np.mean((ref.tonemap(x) - ref.tonemap(gt)) ** 2)))
        rows.append((scene, p_raw, p_den, rmse(raw_hi), rmse(den_hi)))
        print("%s: 4 spp raw %.2f dB, denoised %.2f dB; 4096 spp RMSE raw %.5f, denoised %.5f" % rows[-1])
    for scene, p_raw, p_den, r_raw, r_den in rows:
        assert p_den >= p_raw + 3.0, scene
        assert r_den <= 1.05 * r_raw, scene


def test_invalid_parameters(dn, scenes):
    _setup(dn, scenes, "Scene1", 64, 48)
    dn.render_spp(1)
    lib = dn.lib
    out = np.zeros((48, 64, 4), np.float32)
    surf = np.zeros((48, 64), np.uint32)
    bad = [dict(passes=-1), dict(passes=9), dict(normal_power=0), dict(normal_power=3), dict(normal_power=512), dict(normal_power=-2),
           dict(sigma_color=0.0), dict(sigma_color=-1.0), dict(sigma_color=float("inf")), dict(sigma_color=float("nan")),
           dict(sigma_depth=0.0), dict(sigma_depth=-1.0), dict(sigma_depth=float("inf")), dict(sigma_depth=float("nan"))]
    for kw in bad:
        p = rtb200.default_denoise_params(**kw)
        assert lib.rt_read_denoised(dn.h, C.byref(p), out.ctypes.data_as(C.c_void_p)) == rtb200.RT_ERR_INVALID, kw
        assert lib.rt_denoise_rgba8(dn.h, C.byref(p), surf.ctypes.data_as(C.c_void_p), 64 * 4, 1) == rtb200.RT_ERR_INVALID, kw
    for kw in (dict(passes=0), dict(passes=8), dict(normal_power=1), dict(normal_power=256)):
        dn.read_denoised(rtb200.default_denoise_params(**kw))


def _read_ppm(path):
    with open(path, "rb") as f:
        assert f.readline().strip() == b"P6"
        w, h = [int(x) for x in f.readline().split()]
        assert f.readline().strip() == b"255"
        return np.frombuffer(f.read(), np.uint8).reshape(h, w, 3)


def test_headless_denoise_matches_the_python_sequence(dn, scenes, tmp_path):
    exe = os.path.join(ROOT, "software-raytracer_b200", "bin", "rt_headless")
    if not os.path.exists(exe):
        pytest.skip("bin/rt_headless not built")
    scene_file = str(tmp_path / "Scene1.json")
    assert rtb200.scene_file_write(scene_file, scenes["Scene1"], None, "Scene1") == 0
    w, h, spp = 320, 180, 6
    ppm = str(tmp_path / "d.ppm")
    r = subprocess.run([exe, "--scene", scene_file, "--width", str(w), "--height", str(h), "--spp", str(spp), "--bounces", "8", "--scale", "1",
                        "--denoise", "3", "--out", ppm], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    img = _read_ppm(ppm)
    dn.set_scene(scenes["Scene1"]); dn.set_camera(rtb200.default_camera())
    dn.set_params(rtb200.default_params(width=w, height=h, mode=rtb200.RT_MODE_PATH, max_bounces=8))
    dn.reset_accumulation()
    dn.render_spp(1); dn.render_spp(spp - 1)
    argb = dn.denoise_rgba8(rtb200.default_denoise_params(passes=3), True)
    want = np.stack([(argb >> 16) & 255, (argb >> 8) & 255, argb & 255], -1).astype(np.uint8)
    assert np.array_equal(img, want)
    assert not np.array_equal(argb, dn.resolve_rgba8(True))
    r = subprocess.run([exe, "--scene", scene_file, "--width", "640", "--height", "360", "--interactive", "20", "--scale", "1", "--denoise", "3"],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and '"p50_ms"' in r.stdout, r.stdout + r.stderr
    # the multi-GPU group has no denoised resolve: refused with a message, whatever the device count
    r = subprocess.run([exe, "--scene", scene_file, "--gpus", "2", "--denoise", "3"], capture_output=True, text=True, timeout=300)
    assert r.returncode != 0 and "--denoise" in r.stderr
