"""GPU (B200): every render kernel form, through the C-ABI, against the oracle at the render parameters of
tests/test_render_params_cpu.py (environment, dissipation, eps, depth, camera, inert fields).

The forms are selected by options, never by size thresholds: the per-lane megakernel with and without the primary-hit cache,
the pixel pool, the pooled and per-lane flat traversals, brute force, the binary BVH with float and with quantised nodes, the
8-wide BVH, the traversal-statistics instantiation, the bounce-round wavefront and streaming pipelines (spheres and a mesh),
rt_render_frame, block-filled frames and the large-grid stash form. Images are small and not tile multiples; samples come in
two calls so that the sample offset matters. Radiance sums within RAD_RTOL of the oracle, segment counts exact."""
import os
import subprocess
import sys

import numpy as np
import pytest

import rtb200
from conftest import ROOT
from oracle_py import OrcCamera
from rtb200.scenes import heightfield_mesh, mesh_scene, synthetic_spheres
from test_render_params_cpu import (ENV_SETS, PARAM_SETS, RAD_ATOL, RAD_RTOL, env_directions, env_reference, make_cam,
                                    make_params)

pytestmark = pytest.mark.gpu

W, H = 133, 77
SPLIT, LONG, SHORT = (5, 11), (16, 17), (1, 3)       # LONG: every call long enough for the pooled flat traversal (16+ spp)
CORE = ENV_SETS + ["dissipation_0.5", "dissipation_1", "eps_1e-3", "eps_1e-7", "bounces_61"]

O = rtb200
DEFAULT_OPTIONS = {O.RT_OPT_PIPELINE: O.RT_PIPELINE_AUTO, O.RT_OPT_ACCEL: O.RT_ACCEL_AUTO, O.RT_OPT_POOL_TILES: 0, O.RT_OPT_FLAT_COOP: 2,
                   O.RT_OPT_BVH_WIDE: 0, O.RT_OPT_BVH_QUANT: 1, O.RT_OPT_PRIMARY_REUSE: 1, O.RT_OPT_TRAVERSAL_STATS: 0}

# form -> (options, scene: None = the set's own, calls, sets). "big": 1000 spheres, a BVH too large to stage in shared memory,
# so it is walked from global memory (with the quantised nodes unless RT_OPT_BVH_QUANT 0).
FORMS = {
    "lane": ({O.RT_OPT_POOL_TILES: 1}, None, SPLIT, list(PARAM_SETS)),
    "lane_no_reuse": ({O.RT_OPT_POOL_TILES: 1, O.RT_OPT_PRIMARY_REUSE: 0}, None, SPLIT, CORE + ["bounces_-3", "fov_120"]),
    "pixel_pool": ({O.RT_OPT_POOL_TILES: 2}, None, SHORT, CORE + ["bounces_-3"]),
    "flat_pooled": ({O.RT_OPT_ACCEL: O.RT_ACCEL_FLAT, O.RT_OPT_FLAT_COOP: 1}, None, LONG, CORE),
    "flat_lane": ({O.RT_OPT_ACCEL: O.RT_ACCEL_FLAT, O.RT_OPT_FLAT_COOP: 0}, None, SPLIT, CORE),
    "brute": ({O.RT_OPT_ACCEL: O.RT_ACCEL_BRUTE}, None, SPLIT, CORE),
    "bvh_float_nodes": ({O.RT_OPT_ACCEL: O.RT_ACCEL_BVH, O.RT_OPT_BVH_QUANT: 0}, "big", SPLIT, CORE),
    "bvh_quant_nodes": ({O.RT_OPT_ACCEL: O.RT_ACCEL_BVH, O.RT_OPT_BVH_QUANT: 1}, "big", SPLIT, CORE),
    "bvh_wide": ({O.RT_OPT_ACCEL: O.RT_ACCEL_BVH, O.RT_OPT_BVH_WIDE: 2}, None, SPLIT, CORE),
    "traversal_stats": ({O.RT_OPT_ACCEL: O.RT_ACCEL_BVH, O.RT_OPT_TRAVERSAL_STATS: 1}, None, SPLIT, CORE),
    "wavefront": ({O.RT_OPT_PIPELINE: O.RT_PIPELINE_WAVEFRONT}, None, SPLIT, CORE + ["bounces_60", "bounces_3"]),
    "stream": ({O.RT_OPT_PIPELINE: O.RT_PIPELINE_STREAM, O.RT_OPT_ACCEL: O.RT_ACCEL_BVH}, "big", SPLIT, CORE + ["bounces_60"]),
    "stream_mesh": ({O.RT_OPT_PIPELINE: O.RT_PIPELINE_STREAM, O.RT_OPT_ACCEL: O.RT_ACCEL_BVH}, "mesh", SPLIT, CORE),
}


def scene_of(scenes, key):
    """(objects, mesh (vertices, triangles) of object 0 or None, camera position, fov)"""
    if key == "big":
        return synthetic_spheres(1000, seed=7), None, (0.0, 8.0, -20.0), 60
    if key == "mesh":
        return mesh_scene(), heightfield_mesh(8, 6, seed=3), (0.0, 1.5, -1.0), 55
    return scenes[key], None, (0.0, 0.0, 0.0), 55


def camera(cls, scenes, key, name):
    c = make_cam(cls, name)
    _, _, pos, fov = scene_of(scenes, key)
    c.pos[0], c.pos[1], c.pos[2] = pos
    if "fov_deg" not in PARAM_SETS[name][2]:
        c.fov_deg = fov
    return c


_ORACLE = {}


def expected(oracle, scenes, key, name, calls):
    """The oracle's sums of the same consecutive sample ranges, added in float32 like the accumulation buffer; segments."""
    total, segs, s0 = np.zeros((H, W, 3), np.float32), 0, 0
    for n in calls:
        k = (key, name, s0, n)
        if k not in _ORACLE:
            objs, mesh, _, _ = scene_of(scenes, key)
            if mesh is not None:
                oracle.set_triangles(objs, {0: mesh})
            try:
                _ORACLE[k] = oracle.render(objs, camera(OrcCamera, scenes, key, name), make_params(oracle.default_params, name, W, H), s0, n)[::2]
            finally:
                if mesh is not None:
                    oracle.set_triangles(objs, {})
        total = total + _ORACLE[k][0]
        segs += _ORACLE[k][1]
        s0 += n
    return total, segs


def load(tracer, scenes, key, name):
    objs, mesh, _, _ = scene_of(scenes, key)
    tracer.set_scene(objs)
    if mesh is not None:
        tracer.set_mesh(0, *mesh)
    tracer.set_camera(camera(rtb200.RtCamera, scenes, key, name))
    tracer.set_params(make_params(rtb200.default_params, name, W, H))
    tracer.reset_accumulation()


def close(a, b):
    return np.allclose(a, b, rtol=RAD_RTOL, atol=RAD_ATOL)


def set_options(tracer, opts):
    for k, v in opts.items():
        tracer.set_option(k, v)


def bounces(name):
    return max(PARAM_SETS[name][1].get("max_bounces", 8), 0)


CASES = [(f, s) for f, spec in FORMS.items() for s in spec[3]]


@pytest.mark.parametrize("form,name", CASES)
def test_form_matches_oracle_at_render_parameters(tracer, oracle, scenes, form, name):
    opts, key, calls, _ = FORMS[form]
    key = key or PARAM_SETS[name][0]
    try:
        set_options(tracer, opts)
        load(tracer, scenes, key, name)
        for n in calls:
            tracer.render_spp(n)
        acc, n = tracer.read_accum()
        st = tracer.stats()
        trav = tracer.traversal_stats()
    finally:
        set_options(tracer, DEFAULT_OPTIONS)
    want, segs = expected(oracle, scenes, key, name, calls)
    assert n == sum(calls) and st.paths == W * H * sum(calls)
    assert st.segments == segs
    assert close(acc[..., :3], want)
    if O.RT_OPT_ACCEL in opts:
        assert st.accel == opts[O.RT_OPT_ACCEL]
    pipe = opts.get(O.RT_OPT_PIPELINE, O.RT_PIPELINE_REGEN)
    if pipe == O.RT_PIPELINE_WAVEFRONT and bounces(name) > 60:
        pipe = O.RT_PIPELINE_REGEN                                 # one queue counter per bounce round: deeper paths take the megakernel
    assert st.pipeline == pipe
    if opts.get(O.RT_OPT_PRIMARY_REUSE) == 0:
        assert st.traced_segments == st.segments
    elif pipe == O.RT_PIPELINE_REGEN:
        assert st.traced_segments < st.segments                  # the primary hits came from the cache
    if opts.get(O.RT_OPT_TRAVERSAL_STATS):
        assert trav.queries > 0 and trav.node_visits > 0        # the counting instantiation ran


@pytest.mark.parametrize("name", CORE)
def test_render_frame_matches_oracle_at_render_parameters(tracer, oracle, scenes, name):
    """rt_render_frame into a page-locked surface: 1 spp (the pixel pool resolves the frame inside the render), then 2 spp
    (render, then resolve). The accumulation against the oracle, the surface against the oracle's resolve of it."""
    key = PARAM_SETS[name][0]
    surf, owner = rtb200.host_surface(W, H)
    load(tracer, scenes, key, name)
    for calls in ((1,), (1, 2)):
        surf[:] = 0
        tracer.render_frame(calls[-1], out=surf)
        acc, n = tracer.read_accum()
        want, segs = expected(oracle, scenes, key, name, calls)
        assert n == sum(calls) and tracer.stats().segments == segs
        assert close(acc[..., :3], want)
        assert np.array_equal(surf, oracle.resolve_argb8(acc, n)), calls
    del owner


@pytest.mark.parametrize("steps", [2, 4])
@pytest.mark.parametrize("name", CORE)
def test_block_filled_frames_match_oracle_at_render_parameters(tracer, oracle, scenes, name, steps):
    """rt_set_pixel_step with the reference's strips: every block holds the oracle's full-resolution sum at its first pixel."""
    key = PARAM_SETS[name][0]
    strip = rtb200.reference_strip_columns(W)
    try:
        load(tracer, scenes, key, name)
        tracer.set_pixel_step(steps, strip)
        tracer.reset_accumulation()
        for n in SPLIT:
            tracer.render_spp(n)
        acc, n = tracer.read_accum()
        st = tracer.stats()
    finally:
        tracer.set_pixel_step(1, 0)
    full, _ = expected(oracle, scenes, key, name, SPLIT)
    want = np.zeros_like(full)
    blocks = 0
    for x0 in range(0, W, strip):
        x1 = min(x0 + strip, W)
        for i in range(x0, x1, steps):
            for j in range(0, H, steps):
                want[j:j + steps, i:min(i + steps, x1)] = full[j, i]
                blocks += 1
    assert n == sum(SPLIT) and st.paths == blocks * sum(SPLIT)
    assert close(acc[..., :3], want)


@pytest.mark.parametrize("name", ENV_SETS)
def test_env_color_on_device_matches_float64_statement(tracer, scenes, name):
    load(tracer, scenes, "Scene1", name)
    p = make_params(rtb200.default_params, name, W, H)
    dirs = env_directions(p)
    out = tracer.env_color(dirs)
    want, disc, sdot = env_reference(p, dirs)
    clear = np.abs(sdot - 0.99) > 1e-6
    assert np.allclose(out[clear], want[clear], rtol=2e-6, atol=1e-6)
    assert np.array_equal(np.all(out >= np.array(p.sun[:], np.float32) * np.float32(0.999), axis=1)[clear], disc[clear])


# one context through every set by rt_set_params / rt_set_camera alone, then back to the defaults: the primary-hit cache
# (miss colours), the accelerator margins (eps grows, shrinks, grows again) and the tuned choices must follow each change
SEQUENCE = ["defaults"] + [n for n in PARAM_SETS if n != "defaults"] + ["eps_1e-3", "defaults"]


@pytest.mark.parametrize("accel", [O.RT_ACCEL_FLAT, O.RT_ACCEL_BVH, O.RT_ACCEL_AUTO])
def test_one_context_follows_every_parameter_change(oracle, scenes, accel):
    t = rtb200.PathTracer(0)
    try:
        t.set_option(O.RT_OPT_ACCEL, accel)
        t.set_scene(scenes["Scene1"])
        for name in SEQUENCE:
            t.set_camera(camera(rtb200.RtCamera, scenes, "Scene1", name))
            t.set_params(make_params(rtb200.default_params, name, W, H))
            t.reset_accumulation()
            for n in SPLIT:
                t.render_spp(n)
            acc, n = t.read_accum()
            st = t.stats()
            want, segs = expected(oracle, scenes, "Scene1", name, SPLIT)
            assert st.segments == segs, name
            assert close(acc[..., :3], want), name
            if accel != O.RT_ACCEL_AUTO:
                assert st.accel == accel
    finally:
        t.close()


STASH_CHILD = r"""
import sys
import numpy as np
tests = sys.argv[1]
sys.path[:0] = [tests, sys.argv[2], sys.argv[3]]
import rtb200
from test_render_params_cpu import make_params
from test_gpu_render_params import CORE, LONG, W, H, camera
objs = dict(np.load(sys.argv[4]))
t = rtb200.PathTracer(0)
out = {}
t.set_option(rtb200.RT_OPT_ACCEL, rtb200.RT_ACCEL_FLAT)
t.set_option(rtb200.RT_OPT_FLAT_COOP, 1)
t.set_option(rtb200.RT_OPT_PRIMARY_REUSE, 1)
for name in CORE:
    key = "Scene_indirect" if name.startswith("bounces") else "Scene1"
    t.set_scene(objs[key])
    t.set_camera(camera(rtb200.RtCamera, objs, key, name))
    t.set_params(make_params(rtb200.default_params, name, W, H))
    t.reset_accumulation()
    for n in LONG:
        t.render_spp(n)
    acc, n = t.read_accum()
    st = t.stats()
    out[name] = acc
    out[name + "/stats"] = np.array([n, st.paths, st.segments, st.accel, st.pipeline], np.int64)
t.close()
np.savez(sys.argv[5], **out)
"""


def test_large_grid_stash_form_matches_oracle(oracle, scenes, tmp_path):
    """The 7-CTA form of the pooled flat traversal with the primary-hit cache (k_render_regen STASH) is taken for large grids
    only; RTB200_STASH_MIN_TILES, read once per process, lowers the threshold in a child process so that a small image takes it."""
    src = tmp_path / "scenes.npz"
    np.savez(src, Scene1=scenes["Scene1"], Scene_indirect=scenes["Scene_indirect"])
    dst = tmp_path / "stash.npz"
    env = dict(os.environ, RTB200_STASH_MIN_TILES="1")
    tests = os.path.join(ROOT, "tests")
    r = subprocess.run([sys.executable, "-c", STASH_CHILD, tests, os.path.join(ROOT, "software-raytracer_b200", "python"),
                        os.path.join(ROOT, "oracle"), str(src), str(dst)], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    got = np.load(dst)
    for name in CORE:
        key = PARAM_SETS[name][0]
        want, segs = expected(oracle, scenes, key, name, LONG)
        n, paths, seg, accel, pipe = got[name + "/stats"].tolist()
        assert n == sum(LONG) and paths == W * H * sum(LONG), name
        assert accel == O.RT_ACCEL_FLAT and pipe == O.RT_PIPELINE_REGEN, name
        assert seg == segs, name
        assert close(got[name][..., :3], want), name
