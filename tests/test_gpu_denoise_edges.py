"""GPU: every form of the a-trous filter's kernel (csrc/rt_denoise.cu k_denoise_pass: first / later pass, staged / unstaged, each
output, the per-pixel count form) at its edges, against the float32 restatements (tests/denoise_reference.py,
tests/temporal_reference.py) and the float64 statement (tests/denoise_f64.py): images smaller than the 32 x 8 tile and than the steps
of passes 6-8, every pass count, normal powers 1 and 256, up to 2^32 - 1 samples and the ends of the sigma ranges. The guides are a
real scene's primary-hit cache (Scene1, the heightfield mesh); the sums are written with rt_write_accum, so the sample count can be
anything without rendering. Staging thresholds other than the default (RTB200_DENOISE_STAGE, read once per process) run the same
cases in child processes. Sigmas below kDenoiseSigmaMin, which would make every hit pixel NaN, are refused by every present call
and change nothing."""
import ctypes as C
import math
import os
import subprocess
import sys

import numpy as np
import pytest

import rtb200
from conftest import ROOT, SEED
import denoise_f64 as f64
import denoise_reference as ref
import temporal_reference as tref
from test_denoise_edges_cpu import ATOL, F32_MAX, RTOL, SIZES as CPU_SIZES, TINT, sums

pytestmark = pytest.mark.gpu

SIZES = CPU_SIZES + [(160, 120)]                               # (width, height); 160 x 120 is a whole number of tiles
SCENES = ["Scene1", "mesh"]
N31, N32 = 1 << 31, (1 << 32) - 1
SMIN = f64.SIGMA_MIN
# (passes, normal_power, samples, sigma_color, sigma_depth): every pass count, then the edges with all eight steps
PLAIN = [(p, 128, 4, 2.0, 1.0) for p in range(9)] + [
    (8, 1, 0, 2.0, 1.0), (8, 256, 1, 1e-3, 2.0), (8, 2, N31, SMIN, SMIN), (8, 256, N32, SMIN, 1e30),
    (3, 1, N32, F32_MAX, F32_MAX), (5, 2, 1 << 20, 1e30, 1e-3), (8, 128, N32, 2.0, F32_MAX), (6, 16, 64, 0.5, SMIN)]
# per-pixel count form: (passes, normal_power, sigma_color, sigma_depth, max_history, tau_normal, samples before, samples after)
NEFF = [(1, 128, 2.0, 1.0, 1, -1.0, 4, 1), (5, 256, SMIN, 2.0, 4096, 1.0, N32, N31),
        (8, 1, SMIN, SMIN, 4096, -1.0, 1 << 20, N32), (3, 2, 1e-3, 1e30, 4096, -1.0, 64, 1)]
# ARGB8 outputs in turn: (flip_y, surface) with surface "tight", "pitched" (a row pitch wider than the image) or "pinned"
ARGB = [(1, "tight"), (0, "pitched"), (1, "pinned"), (0, "tight"), (1, "pitched"), (0, "pinned")]
STAGE_CHILDREN = ["0", "1", "2"]


def _camera(name, yaw_deg=0.0):
    cam = rtb200.default_camera(55)
    if name == "mesh":
        cam.pos[1] = 1.5; cam.pos[2] = -1.0
    if yaw_deg:
        rtb200.rotate_camera(cam, yaw_deg * math.pi / 180.0, [cam.up[0], cam.up[1], cam.up[2]])
    return cam


def _setup(t, scenes, name, w, h):
    if name == "mesh":
        from rtb200.scenes import heightfield_mesh, mesh_scene
        t.set_scene(mesh_scene())
        v, tr = heightfield_mesh(24, 16, seed=3)
        t.set_mesh(0, v, tr)
    else:
        t.set_scene(scenes[name])
    t.set_camera(_camera(name))
    t.set_params(rtb200.default_params(width=w, height=h, mode=rtb200.RT_MODE_PATH, max_bounces=8, seed_lo=SEED[0], seed_hi=SEED[1]))
    t.reset_accumulation()


def _guides(t):
    ids, tt, nrm, _ = t.read_aov()
    return ids, np.concatenate([nrm, tt[..., None]], -1)


def _means(key, w, h):
    """Two deterministic synthetic mean images (grey levels in [0, 4) times one tint, as in the CPU file)."""
    rng = np.random.default_rng(sum(map(ord, key)))
    return [(rng.uniform(0.0, 4.0, (h, w)).astype(np.float32)[..., None] * TINT) for _ in range(2)]


def _argb(t, call, w, h, k):
    """The ARGB8 output of call(flip_y, out) on the k-th surface kind of ARGB, as a (h, w) array."""
    flip, kind = ARGB[k % len(ARGB)]
    if kind == "pinned":
        surf, owner = rtb200.host_surface(w, h)
        call(flip, surf)
        out = surf.copy()
        del owner
        return out
    buf = np.zeros((h, w + (5 if kind == "pitched" else 0)), np.uint32)
    call(flip, buf[:, :w])
    return buf[:, :w].copy()


def run_cases(scenes):
    """Every case on a fresh context: {name: array}. The in-process run and the staging children call this alike."""
    t = rtb200.PathTracer(0)
    out = {}
    try:
        for name in SCENES:
            for w, h in SIZES:
                key = "%s/%dx%d" % (name, w, h)
                _setup(t, scenes, name, w, h)
                out[key + "/ids"], out[key + "/nt"] = _guides(t)
                mean, mean2 = _means(key, w, h)
                for k, (passes, power, n, sc, sz) in enumerate(PLAIN):
                    t.write_accum(sums(mean, n), n)
                    dn = rtb200.default_denoise_params(passes=passes, normal_power=power, sigma_color=sc, sigma_depth=sz)
                    out["%s/plain%d" % (key, k)] = t.read_denoised(dn)
                    out["%s/plain%d/argb" % (key, k)] = _argb(t, lambda flip, o: t.denoise_rgba8(dn, flip_y=flip, out=o), w, h, k)
                for k, (passes, power, sc, sz, cap, tau_n, n0, n1) in enumerate(NEFF):
                    tp = rtb200.default_temporal_params(max_history=cap, tau_normal=tau_n)
                    dn = rtb200.default_denoise_params(passes=passes, normal_power=power, sigma_color=sc, sigma_depth=sz)
                    # a history at the scene's pose, then a turned camera with other samples: the prior is reprojected
                    t.set_camera(_camera(name)); t.reset_temporal()
                    t.write_accum(sums(mean, n0), n0)
                    t.read_temporal(tp)
                    t.set_camera(_camera(name, 0.4 + 0.1 * k))
                    t.write_accum(sums(mean2, n1), n1)
                    kk = "%s/neff%d" % (key, k)
                    out[kk + "/ids"], out[kk + "/nt"] = _guides(t)
                    out[kk + "/blend"] = t.read_temporal(tp)           # the same prior below: same pose, same accumulation
                    out[kk] = t.read_temporal(tp, dn)
                    out[kk + "/argb"] = _argb(t, lambda flip, o: t.temporal_rgba8(tp, dn, flip_y=flip, out=o), w, h, k)
                t.set_camera(_camera(name))
    finally:
        t.close()
    return out


CHILD = r"""
import sys
import numpy as np
sys.path[:0] = [sys.argv[1], sys.argv[2], sys.argv[3]]
from test_gpu_denoise_edges import run_cases
np.savez(sys.argv[5], **run_cases(dict(np.load(sys.argv[4]))))
"""


def _check(label, got, f32, want, argb, oracle, flip):
    assert np.isfinite(got).all(), label
    np.testing.assert_allclose(got[..., :3], f32, rtol=RTOL, atol=ATOL * float(np.abs(f32).max()), err_msg=label + " float32")
    np.testing.assert_allclose(got[..., :3], want, rtol=RTOL, atol=ATOL * float(np.abs(want).max()), err_msg=label + " float64")
    mean = np.concatenate([got[..., :3], np.zeros(got.shape[:2] + (1,), np.float32)], -1)
    assert np.array_equal(argb, oracle.resolve_argb8(mean, 0, flip_y=bool(flip))), label + " argb"


def test_every_kernel_form_matches_the_references_at_the_edges(scenes, oracle, tmp_path):
    src = tmp_path / "scenes.npz"
    np.savez(src, Scene1=scenes["Scene1"])
    tests = os.path.join(ROOT, "tests")
    children = {}
    for stage in STAGE_CHILDREN:
        dst = tmp_path / ("stage%s.npz" % stage)
        env = dict(os.environ, RTB200_DENOISE_STAGE=stage)
        children[stage] = (dst, subprocess.Popen([sys.executable, "-c", CHILD, tests, os.path.join(ROOT, "software-raytracer_b200", "python"),
                                                  os.path.join(ROOT, "oracle"), str(src), str(dst)],
                                                 env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True))
    runs = {}
    try:
        runs["default"] = run_cases(scenes)
        for stage, (dst, proc) in children.items():
            log, _ = proc.communicate(timeout=600)
            assert proc.returncode == 0, log[-3000:]
            runs["stage" + stage] = dict(np.load(dst))
    finally:
        for _, proc in children.values():
            if proc.poll() is None:
                proc.kill()
                proc.wait()
    base = runs["default"]
    for name in SCENES:
        for w, h in SIZES:
            key = "%s/%dx%d" % (name, w, h)
            ids, nt = base[key + "/ids"], base[key + "/nt"]
            mean, _ = _means(key, w, h)
            for k, (passes, power, n, sc, sz) in enumerate(PLAIN):
                acc = sums(mean, n)
                with np.errstate(over="ignore"):                # sigma FLT_MAX: sigma^2 and sigma_z s overflow to inf, as on the device
                    f32 = ref.denoise(acc, n, ids, nt, passes, power, sc, sz)
                want = f64.denoise(acc, n, ids, nt, passes, power, sc, sz)
                for run, o in runs.items():
                    label = str((run, key, "plain", passes, power, n, sc, sz))
                    assert np.array_equal(o[key + "/ids"], ids) and np.array_equal(o[key + "/nt"].view(np.uint32), nt.view(np.uint32)), label
                    got = o["%s/plain%d" % (key, k)]
                    assert not got[..., 3].any(), label
                    _check(label, got, f32, want, o["%s/plain%d/argb" % (key, k)], oracle, ARGB[k % len(ARGB)][0])
            for k, (passes, power, sc, sz, cap, tau_n, n0, n1) in enumerate(NEFF):
                kk = "%s/neff%d" % (key, k)
                nids, nnt, blend = base[kk + "/ids"], base[kk + "/nt"], base[kk + "/blend"]
                f32 = tref.filter(blend, nids, nnt, passes, power, sc, sz)
                want = f64.denoise_neff(blend, nids, nnt, passes, power, sc, sz)
                for run, o in runs.items():
                    label = str((run, kk, passes, power, sc, sz, cap, tau_n, n0, n1))
                    assert np.array_equal(o[kk + "/blend"].view(np.uint32), blend.view(np.uint32)), label
                    got = o[kk]
                    np.testing.assert_array_equal(got[..., 3], blend[..., 3], err_msg=label)
                    _check(label, got, f32, want, o[kk + "/argb"], oracle, ARGB[k % len(ARGB)][0])
    # the history really was blended in: N_eff above the sample count somewhere
    assert any((base["%s/%dx%d/neff%d/blend" % (name, w, h, k)][..., 3] > NEFF[k][7]).any()
               for name in SCENES for w, h in SIZES[-2:] for k in range(len(NEFF)))


BAD_SIGMAS = [1e-20, 1e-40, float(np.nextafter(np.float32(SMIN), np.float32(0)))]     # 1e-40: subnormal


def _calls(lib, h, dn, surf, rgba):
    """The four single-context present calls with the filter parameters dn: their return codes."""
    return [lib.rt_denoise_rgba8(h, C.byref(dn), surf.ctypes.data_as(C.c_void_p), surf.strides[0], 1),
            lib.rt_read_denoised(h, C.byref(dn), rgba.ctypes.data_as(C.c_void_p)),
            lib.rt_temporal_rgba8(h, None, C.byref(dn), surf.ctypes.data_as(C.c_void_p), surf.strides[0], 1),
            lib.rt_read_temporal(h, None, C.byref(dn), rgba.ctypes.data_as(C.c_void_p))]


def _stats(s):
    return (s.paths, s.segments, s.samples, s.total_paths, s.total_segments, s.traced_segments, s.total_traced_segments)


def test_sigmas_below_the_minimum_are_refused_and_change_nothing(scenes):
    w, h = 97, 61
    t = rtb200.PathTracer(0)
    try:
        _setup(t, scenes, "Scene1", w, h)
        t.render_spp(2)
        ids, _ = _guides(t)
        a, b = _means("refusal", w, h)
        tp = rtb200.default_temporal_params()
        t.write_accum(sums(a, 4), 4)
        t.read_temporal(tp)
        t.write_accum(sums(b, 2), 2)
        last = t.read_temporal(tp)                             # blended with the history of the call before
        assert not np.array_equal(last[..., :3].view(np.uint32), ref.mean_of(sums(b, 2), 2).view(np.uint32))
        acc0, n0 = t.read_accum()
        st0 = _stats(t.stats())
        surf = np.zeros((h, w), np.uint32)
        rgba = np.zeros((h, w, 4), np.float32)
        for which in ("sigma_color", "sigma_depth"):
            for v in BAD_SIGMAS:
                assert 0.0 < np.float32(v) < np.float32(SMIN)
                dn = rtb200.default_denoise_params(passes=3, **{which: v})
                assert _calls(t.lib, t.h, dn, surf, rgba) == [rtb200.RT_ERR_INVALID] * 4, (which, v)
                assert b"2^-16" in t.lib.rt_last_error(t.h), (which, v)
        acc1, n1 = t.read_accum()
        assert n1 == n0 and np.array_equal(acc1.view(np.uint32), acc0.view(np.uint32))
        assert _stats(t.stats()) == st0
        # the history is the one `last` left: a new accumulation at the same pose blends exactly that in
        t.write_accum(sums(a, 1), 1)
        got = t.read_temporal(tp)
        want = tref.output(sums(a, 1), 1, ids, tref.copy_prior(last, tp.max_history))
        assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
        # the smallest accepted sigmas, at the largest sample count: accepted by every call, finite
        t.write_accum(sums(b, N32), N32)
        dn = rtb200.default_denoise_params(passes=8, sigma_color=SMIN, sigma_depth=SMIN)
        assert _calls(t.lib, t.h, dn, surf, rgba) == [rtb200.RT_OK] * 4
        assert np.isfinite(t.read_denoised(dn)).all() and np.isfinite(t.read_temporal(tp, dn)).all()
    finally:
        t.close()


def test_group_calls_refuse_the_same_sigmas(scenes):
    w, h = 33, 9
    g = rtb200.TracerGroup([0])
    try:
        g.set_scene(scenes["Scene1"])
        g.set_camera(_camera("Scene1"))
        g.set_params(rtb200.default_params(width=w, height=h, mode=rtb200.RT_MODE_PATH, max_bounces=8, seed_lo=SEED[0], seed_hi=SEED[1]))
        g.reset_accumulation()
        g.render_spp(2)
        m = g.members[0]
        acc0, n0 = m.read_accum()
        st0 = _stats(g.stats())
        surf = np.zeros((h, w), np.uint32)
        for which in ("sigma_color", "sigma_depth"):
            for v in BAD_SIGMAS:
                dn = rtb200.default_denoise_params(passes=3, **{which: v})
                p = surf.ctypes.data_as(C.c_void_p)
                assert g.lib.rt_group_denoise_rgba8(g.g, C.byref(dn), p, w * 4, 1) == rtb200.RT_ERR_INVALID, (which, v)
                assert g.lib.rt_group_temporal_rgba8(g.g, None, C.byref(dn), p, w * 4, 1) == rtb200.RT_ERR_INVALID, (which, v)
                assert b"2^-16" in g.lib.rt_group_last_error(g.g), (which, v)
        acc1, n1 = m.read_accum()
        assert n1 == n0 and np.array_equal(acc1.view(np.uint32), acc0.view(np.uint32))
        assert _stats(g.stats()) == st0
        dn = rtb200.default_denoise_params(passes=8, sigma_color=SMIN, sigma_depth=SMIN)
        assert np.isfinite(g.read_denoised(dn)).all() and np.isfinite(g.read_temporal(None, dn)).all()
        g.denoise_rgba8(dn); g.temporal_rgba8(None, dn)
    finally:
        g.close()
